"""Train losses with the reference's names and semantics (dfd/timm/loss/cross_entropy.py:6-36).

On `[N, K]` logits these are a handful of tiny torch ops; when the runner is given one of these objects together with
a NativeModel it uses the fused classifier + softmax cross-entropy kernels instead (`native_smoothing` / `native_soft`
tell it which target encoding to use), for any 2 <= K <= DFD_HEAD_KMAX. At K = 2 the kernel computes sigmoid-BCE on
z1 - z0, which is the same function as 2-class softmax-CE."""
import torch
import torch.nn as nn
import torch.nn.functional as F


class LabelSmoothingCrossEntropy(nn.Module):
    def __init__(self, smoothing=0.1):
        super().__init__()
        assert smoothing < 1.0
        self.smoothing = smoothing
        self.confidence = 1.0 - smoothing
        self.native_smoothing = float(smoothing)
        self.native_soft = False

    def forward(self, x, target):
        logp = F.log_softmax(x, dim=-1)
        nll = -logp.gather(dim=-1, index=target.unsqueeze(1)).squeeze(1)
        return (self.confidence * nll + self.smoothing * (-logp.mean(dim=-1))).mean()


class SoftTargetCrossEntropy(nn.Module):
    native_smoothing = 0.0
    native_soft = True

    def forward(self, x, target):
        return torch.sum(-target * F.log_softmax(x, dim=-1), dim=-1).mean()


class CrossEntropyLoss(nn.CrossEntropyLoss):
    """nn.CrossEntropyLoss (train.py:509-520) tagged for the fused path"""
    native_smoothing = 0.0
    native_soft = False
