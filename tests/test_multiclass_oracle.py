"""Pins oracle/ to the reference for class counts other than 2: the fixtures were produced by the UNMODIFIED reference
(tools/mint_multiclass_goldens.py, gzip-compressed JSON) with 5 classes (label smoothing, soft targets) and the reference's default 1000
classes. Same checks and tolerances as test_oracle_vs_reference_goldens.py::test_train_steps_match_reference; plus the
host-side interface for any class count (no GPU needed)."""
import gzip
import json
import os

import pytest
import torch

from deepfake_detection_b200.arch import get_spec, param_entries, state_entries
from oracle import train as OT
from oracle.weights import synth_batch, synth_state
from test_oracle_vs_reference_goldens import RTOL, _check_summ

def load(golden_dir, name):
    with gzip.open(os.path.join(golden_dir, name + ".json.gz"), "rt") as f:
        return json.load(f)


CASES = ["step_resnet18_k5_ls", "step_efficientnet_b0_k5_soft_rmsprop", "step_efficientnet_b0_k1000"]


@pytest.mark.parametrize("case", CASES)
def test_multiclass_train_steps_match_reference(case, golden_dir):
    rec = load(golden_dir, case)
    K = rec["num_classes"]
    torch.set_num_threads(8)
    spec = get_spec(rec["arch"], num_classes=K)
    sd = synth_state(spec, seed=rec["weight_seed"])
    assert tuple(sd[("classifier" if spec.family == "efficientnet" else "fc") + ".weight"].shape) == (K, spec.num_features)
    wd = rec["weight_decay"]
    if rec["opt"] == "adamw":
        wd = wd / rec["lr"]
    opt = OT.OptState(kind=rec["opt"], lr=rec["lr"], momentum=rec["momentum"], weight_decay=wd, eps=1e-8)
    for i, st in enumerate(rec["steps"]):
        x, y = synth_batch(rec["batch"], 3, rec["H"], rec["W"], seed=1234 + i, soft=rec["soft"], num_classes=K)
        out = OT.train_step(spec, sd, x, y, opt, smoothing=rec["smoothing"])
        ref_logits = torch.tensor(st["logits"])
        assert tuple(ref_logits.shape) == (rec["batch"], K)
        assert torch.allclose(out["logits"], ref_logits, rtol=1e-3, atol=1e-4 * float(ref_logits.abs().max() + 1)), "logits step %d" % i
        assert float(out["loss"]) == pytest.approx(st["loss"], rel=1e-4)
        assert float(out["prec1"]) == pytest.approx(st["prec1"], abs=1e-3)
        rt = RTOL * (1 if i == 0 else 25)
        gfloor = 1e-5 * max(v["norm"] / max(out["grads"][k].numel(), 1) ** 0.5 for k, v in st["grads"].items())
        for k, s in st["grads"].items():
            _check_summ(out["grads"][k], s, "grad %s step %d" % (k, i), rt, floor=gfloor)
        noise = {k for k, v in st["grads"].items()
                 if v["norm"] / max(out["grads"][k].numel(), 1) ** 0.5 < 10 * gfloor} if rec["opt"] != "sgd" else set()
        if i == 0:
            skipped = set(noise)
        for k, s in st["params"].items():
            if k in skipped or k in noise:
                continue
            _check_summ(sd[k], s, "param %s step %d" % (k, i), rt)
        for k, s in st["buffers"].items():
            _check_summ(sd[k].float(), s, "buffer %s step %d" % (k, i), rt)
    x, y = synth_batch(rec["batch"], 3, rec["H"], rec["W"], seed=999, num_classes=K)
    ev = OT.validate_step(spec, sd, x, y)
    ref = torch.tensor(rec["eval"]["logits"])
    assert torch.allclose(ev["logits"], ref, rtol=5e-3, atol=5e-3 * float(ref.abs().max()))


@pytest.mark.parametrize("key", ["efficientnet_b0_k5", "resnet18_k5", "efficientnet_b0_k1000", "resnet18_k1000"])
def test_multiclass_state_entries_match_reference(key, golden_dir):
    ref = load(golden_dir, "state_keys_multiclass")[key]
    spec = get_spec(ref["arch"], num_classes=ref["num_classes"])
    assert [[n, list(s)] for n, s, _ in state_entries(spec)] == ref["state"]
    assert [[n, list(s)] for n, s, _ in param_entries(spec)] == ref["params"]


def test_num_classes_bounds():
    """1 .. DFD_HEAD_KMAX classes are accepted at construction (CPU plan); 0 (timm's identity classifier) and counts above
    the kernel limit are refused with a message before anything is built."""
    from deepfake_detection_b200 import _lib
    from deepfake_detection_b200.engine import Engine
    from deepfake_detection_b200.models import NativeModel, create_deepfake_model_v4, create_model
    kmax = _lib.lib().head_kmax
    assert kmax >= 4096
    for bad in (0, -1, kmax + 1):
        with pytest.raises(ValueError, match="num_classes"):
            create_model("efficientnet_b0", num_classes=bad)
        with pytest.raises(ValueError, match="num_classes"):
            Engine("resnet18", 2, 64, 64, num_classes=bad, device="plan-only")
    with pytest.raises(ValueError, match="num_classes"):
        create_deepfake_model_v4("efficientnet_deepfake_v4", num_classes=0, in_chans=12)
    m = create_model("efficientnet_b0")
    assert isinstance(m, NativeModel) and m.num_classes == 1000 and m.spec.num_classes == 1000
    for arch in ("efficientnet_b0", "resnet18"):
        for K in (1, 5, 1000, kmax):
            eng = Engine(arch, 2, 64, 64, num_classes=K, device="plan-only")
            assert tuple(eng.logits.shape) == (2, K) and tuple(eng.target_f.shape) == (2, K)
            head = [a for _, n, a in eng.bwd_ops if n == "dfd_head_bwd"]
            assert len(head) == 1 and head[0][-1] == K


def test_head_entry_points_refuse_unsupported_sizes():
    """Size checks of dfd_head_fwd / dfd_head_bwd return before anything is launched (NULL pointers never dereferenced)"""
    from deepfake_detection_b200 import _lib
    L = _lib.lib()
    kmax = L.head_kmax
    nul = [None] * 4
    assert L.dfd_head_fwd(*nul, 2, 16, kmax + 1, None, None, 0.0, 1.0, None, None, None, None, None) == -3
    assert "KMAX" in L.last_error()
    assert L.dfd_head_fwd(*nul, 2, 16, 1, None, None, 0.0, 1.0, None, 1, 1, None, None) == -3
    assert "num_classes >= 2" in L.last_error()
    assert L.dfd_head_fwd(*nul, 0, 16, 5, None, None, 0.0, 1.0, None, None, None, None, None) == -1
    assert L.dfd_head_bwd(None, None, None, None, None, None, 2, 16, kmax + 1, None) == -3
    assert L.dfd_head_bwd(None, None, None, None, None, None, 2, 0, 5, None) == -1
