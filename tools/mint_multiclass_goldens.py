"""Mint the multi-class golden fixtures under tests/golden/ FROM THE UNMODIFIED REFERENCE.

TEST INFRASTRUCTURE, the K-class companion of oracle/mint_goldens.py (same shims, weights, batches and record format;
every record also stores `num_classes`).  Run where the reference tree is available:

    python tools/mint_multiclass_goldens.py

It writes only the files below and never touches the 2-class fixtures:
    step_resnet18_k5_ls.json.gz                  ResNet-18, 4 x 64^2, SGD, label smoothing 0.1, 5 classes
    step_efficientnet_b0_k5_soft_rmsprop.json.gz EfficientNet-B0, soft 5-class targets, RMSpropTF
    step_efficientnet_b0_k1000.json.gz           EfficientNet-B0, hard labels, the reference's default 1000 classes
    state_keys_multiclass.json.gz                state_dict / parameter key and shape lists for 5 and 1000 classes
The files are gzip-compressed JSON; fp32 values (logits, sampled elements) are written as the shortest decimal that reads
back as the same fp32 number.
"""
import gzip
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from deepfake_detection_b200.arch import get_spec  # noqa: E402
from oracle import ref_shims  # noqa: E402
from oracle.mint_goldens import GOLDEN, _args, _summ  # noqa: E402
from oracle.weights import synth_batch, synth_state  # noqa: E402


def _write(name, rec):
    def f32(v):
        if isinstance(v, dict):
            return {k: (f32(x) if k in ("logits", "samples") or isinstance(x, (dict, list)) else x) for k, x in v.items()}
        if isinstance(v, list):
            return [f32(x) for x in v]
        return float(str(np.float32(v))) if isinstance(v, float) else v

    with gzip.open(os.path.join(GOLDEN, name + ".gz"), "wt", compresslevel=9) as f:
        json.dump(f32(rec), f)


def mint_step(arch, batch, H, W, num_classes, n_steps=2, smoothing=0.0, opt_name="sgd", soft=False, tag=""):
    """oracle/mint_goldens.py::mint_step with the class count as a parameter"""
    from dfd.timm.loss import LabelSmoothingCrossEntropy, SoftTargetCrossEntropy
    from dfd.timm.models import create_model
    from dfd.timm.optim import create_optimizer
    from dfd.timm.utils import accuracy
    torch.manual_seed(0)
    spec = get_spec(arch, num_classes=num_classes)
    model = create_model(arch, num_classes=num_classes)
    model.load_state_dict(synth_state(spec, seed=7), strict=True)
    model.train()
    lr = 0.01 if opt_name == "sgd" else 1e-3
    wd = 1e-4
    optimizer = create_optimizer(_args(opt=opt_name, lr=lr, weight_decay=wd), model)
    if soft:
        loss_fn = SoftTargetCrossEntropy()
    elif smoothing > 0:
        loss_fn = LabelSmoothingCrossEntropy(smoothing)
    else:
        loss_fn = torch.nn.CrossEntropyLoss()
    rec = dict(arch=arch, num_classes=num_classes, batch=batch, H=H, W=W, weight_seed=7, opt=opt_name, lr=lr,
               momentum=0.9, weight_decay=wd, smoothing=smoothing, soft=soft, torch=torch.__version__, steps=[])
    for step in range(n_steps):
        x, y = synth_batch(batch, 3, H, W, seed=1234 + step, soft=soft, num_classes=num_classes)
        out = model(x)
        loss = loss_fn(out, y)
        prec1 = accuracy(out, y, topk=(1,))
        optimizer.zero_grad()
        loss.backward()
        grads = {k: _summ(p.grad) for k, p in model.named_parameters()}
        optimizer.step()
        rec["steps"].append(dict(
            logits=out.detach().tolist(), loss=float(loss), prec1=float(prec1), grads=grads,
            params={k: _summ(p) for k, p in model.named_parameters()},
            buffers={k: _summ(b.float()) for k, b in model.named_buffers()}))
    model.eval()
    with torch.no_grad():
        x, y = synth_batch(batch, 3, H, W, seed=999, num_classes=num_classes)
        out = model(x)
        rec["eval"] = dict(logits=out.tolist(), loss=float(torch.nn.CrossEntropyLoss()(out, y)))
    name = "step_%s%s.json" % (arch, tag)
    _write(name, rec)
    print(name, "loss", [s["loss"] for s in rec["steps"]], "eval", rec["eval"]["loss"])


def mint_state_keys():
    from dfd.timm.models import create_model
    out = {}
    for k in (5, 1000):
        for arch in ("efficientnet_b0", "resnet18"):
            m = create_model(arch, num_classes=k)
            out["%s_k%d" % (arch, k)] = dict(
                arch=arch, num_classes=k, state=[[n, list(v.shape)] for n, v in m.state_dict().items()],
                params=[[n, list(v.shape)] for n, v in m.named_parameters()],
                n_params=sum(p.numel() for p in m.parameters()))
    _write("state_keys_multiclass.json", out)
    print("state_keys_multiclass.json:", {k: v["n_params"] for k, v in out.items()})


def main():
    ref_shims.install()
    torch.set_num_threads(8)
    mint_state_keys()
    mint_step("resnet18", 4, 64, 64, 5, smoothing=0.1, tag="_k5_ls")
    mint_step("efficientnet_b0", 4, 64, 64, 5, soft=True, opt_name="rmsproptf", tag="_k5_soft_rmsprop")
    mint_step("efficientnet_b0", 4, 64, 64, 1000, tag="_k1000")


if __name__ == "__main__":
    main()
