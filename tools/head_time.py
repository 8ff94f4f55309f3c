"""Classifier head kernels at batch 256: dfd_head_fwd (logits + softmax-CE + top-1 + dL/dlogits) and dfd_head_bwd
(dpooled, dW, db) for F in {256, 1280, 2048} (ResNet-18, EfficientNet-B0, ResNet-50 feature widths) and K in {2, 5, 1000}.
CUDA events over 200 back-to-back launches after a warm-up; the operands (at most 16 MB) stay in L2, as they do inside a
train step. Prints the GPU name and power limit with the numbers."""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deepfake_detection_b200 import _lib  # noqa: E402

N = 256
st = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
P = lambda t: t.data_ptr()  # noqa: E731


def timeit(fn, reps=200):
    for _ in range(10):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


def main():
    if not torch.cuda.is_available():
        raise SystemExit("head_time.py needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    print("gpu:", q or torch.cuda.get_device_name())
    for F in (256, 1280, 2048):
        for K in (2, 5, 1000):
            g = torch.Generator(device="cuda").manual_seed(0)
            pooled = torch.randn(N, F, device="cuda", generator=g)
            W = torch.randn(K, F, device="cuda", generator=g) / F ** 0.5
            b = torch.zeros(K, device="cuda")
            y = torch.randint(0, K, (N,), device="cuda", generator=g)
            logits, dlog = torch.zeros(N, K, device="cuda"), torch.zeros(N, K, device="cuda")
            acc = torch.zeros(2, device="cuda")
            dW, db, dpooled = torch.zeros_like(W), torch.zeros_like(b), torch.zeros(N, F, device="cuda")
            fwd = lambda: _lib.call("dfd_head_fwd", P(pooled), P(W), P(b), P(logits), N, F, K, P(y), None, 0.1, 1.0, None,  # noqa: E731
                                    P(acc), P(acc) + 4, P(dlog), st())
            bwd = lambda: _lib.call("dfd_head_bwd", P(dlog), P(pooled), P(W), P(dW), P(db), P(dpooled), N, F, K, st())  # noqa: E731
            tf, tb = timeit(fwd), timeit(bwd)
            flop = 3 * 2.0 * N * F * K
            print("N=%d F=%4d K=%4d  fwd %7.1f us  bwd %7.1f us  total %7.1f us  (%.2f GFLOP, %.2f TFLOP/s fp32)"
                  % (N, F, K, tf, tb, tf + tb, flop / 1e9, flop / ((tf + tb) * 1e-6) / 1e12), flush=True)


if __name__ == "__main__":
    main()
