"""Device-side train step (Trainer.step_resident, CUDA-graph replayed, as bench.py times it) of EfficientNet-B0, batch 256,
224^2, bf16, SGD, for 2 and 1000 classes. The two class counts alternate in ROUNDS rounds of STEPS steps (CUDA events
around each round) so that drift of the shared machine hits both alike. Prints the GPU name and power limit."""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deepfake_detection_b200.arch import get_spec  # noqa: E402
from deepfake_detection_b200.models import init_state_dict  # noqa: E402
from deepfake_detection_b200.trainer import Trainer  # noqa: E402

B, RES, STEPS, ROUNDS = 256, 224, 20, 5


def make(K):
    tr = Trainer("efficientnet_b0", B, RES, RES, dtype="bf16", num_classes=K)
    tr.load_state_dict(init_state_dict(get_spec("efficientnet_b0", num_classes=K), seed=42))
    g = torch.Generator(device="cuda").manual_seed(1234)
    tr.engine.set_input(torch.randn(B, 3, RES, RES, device="cuda", generator=g))
    tr.engine.set_target(torch.randint(0, K, (B,), device="cuda", generator=g))
    for _ in range(5):
        tr.step_resident()
    torch.cuda.synchronize()
    return tr


def main():
    if not torch.cuda.is_available():
        raise SystemExit("multiclass_step_time.py needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    print("gpu:", q or torch.cuda.get_device_name())
    trs = {K: make(K) for K in (2, 1000)}
    ms = {K: [] for K in trs}
    for _ in range(ROUNDS):
        for K, tr in trs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(STEPS):
                tr.step_resident()
            e1.record()
            torch.cuda.synchronize()
            ms[K].append(e0.elapsed_time(e1) / STEPS)
    for K, v in ms.items():
        v = sorted(v)
        print("efficientnet_b0 b%d %d^2 bf16 K=%4d  step %.3f ms (median of %d rounds x %d steps; min %.3f max %.3f)  loss %.4f"
              % (B, RES, K, v[len(v) // 2], ROUNDS, STEPS, v[0], v[-1], float(trs[K].engine.loss)))
    m2, m1000 = sorted(ms[2])[ROUNDS // 2], sorted(ms[1000])[ROUNDS // 2]
    print("K=1000 vs K=2: %+.2f %% (%+.3f ms)" % (100.0 * (m1000 / m2 - 1.0), m1000 - m2))


if __name__ == "__main__":
    main()
