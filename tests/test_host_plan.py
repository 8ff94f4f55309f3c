"""Host logic without a GPU: the C-ABI library loads and exports every symbol include/dfd_b200.h declares, the
ctypes signature table agrees with the header, and the engine's call plan (arenas, pointer arithmetic, argument
lists) builds for the BASELINE configurations."""
import os
import re

import pytest

from deepfake_detection_b200 import _lib
from deepfake_detection_b200.arch import get_spec, param_entries

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _protos():
    hdr = open(os.path.join(ROOT, "include", "dfd_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return re.findall(r"\b(?:int|const char\*)\s+(dfd_\w+)\s*\(([^)]*)\)\s*;", hdr)


def test_library_exports_every_declared_symbol():
    L = _lib.lib()
    names = [n for n, _ in _protos()]
    assert len(names) >= 30
    for n in names:
        assert hasattr(L.cdll, n), n
    assert L.cdll.dfd_abi_version() == 1
    assert L.stat_slots == 8


def test_ctypes_signatures_match_header():
    for name, params in _protos():
        if name == "dfd_last_error":
            continue
        codes = ""
        if params.strip() != "void":
            for p in params.split(","):
                p = p.strip()
                codes += "p" if "*" in p else "l" if "long long" in p else "f" if p.startswith("float") else \
                    "d" if p.startswith("double") else "i"
        assert _lib.SIGNATURES[name] == codes, name


@pytest.mark.parametrize("arch,batch,res", [("efficientnet_b0", 2, 64), ("efficientnet_b4", 1, 76),
                                             ("efficientnet_b0", 4, 224)])
def test_engine_plan_builds(arch, batch, res):
    from deepfake_detection_b200.engine import Engine
    eng = Engine(arch, batch, res, res, device="plan-only")
    spec = get_spec(arch)
    n = sum(int(__import__("math").prod(s)) for _, s, _ in param_entries(spec))
    assert eng.n_params >= n
    assert set(eng.p_off) == {e[0] for e in param_entries(spec)}
    assert eng.n_launch["fwd"] > 100 and eng.n_launch["bwd"] > 150
    # arena offsets never overlap
    spans = sorted((o, o + k) for o, _, k in eng.p_off.values())
    assert all(a[1] <= b[0] for a, b in zip(spans, spans[1:]))


def test_no_oracle_on_product_path():
    """The product package must never import oracle/ (or fall back to torch compute)."""
    pkg = os.path.join(ROOT, "deepfake_detection_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f


def test_bench_native_arm_does_not_touch_the_oracle():
    """bench.py may execute oracle/ only on its cpu_baseline / --impl reference leg (run_reference)."""
    src = open(os.path.join(ROOT, "bench.py")).read()
    end = min(src.index("def cpu_baseline"), src.index("def run_reference"))
    native = src[src.index("def run_native"):end]
    assert src.index("def run_native") < end
    # the only mention allowed is the call into cpu_baseline(), which lives outside this function
    assert not re.search(r"(from|import)\s+oracle", native)


def test_bench_dump_outputs_stays_in_budget_and_samples_the_same_positions(tmp_path):
    """bench.py --dump-outputs: small arrays are written whole, a large one as a fixed-seed sample, all of them within the
    byte budget; a second dump of the same arrays is identical."""
    import numpy as np
    import torch
    import bench
    g = torch.Generator().manual_seed(0)
    arrays = dict(loss=torch.tensor([0.5]), logits=torch.randn(8, 2, generator=g), state=torch.randn(5000, generator=g),
                  grads=torch.randn(3000, generator=g, dtype=torch.float64))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, budget=16384)
    got = {f[:-4]: np.load(str(tmp_path / "a" / f)) for f in os.listdir(str(tmp_path / "a"))}
    assert set(got) == set(arrays)
    assert sum(os.path.getsize(str(tmp_path / "a" / (n + ".npy"))) - 128 for n in got) <= 16384
    assert got["logits"].dtype == np.float32 and np.array_equal(got["logits"], arrays["logits"].numpy())
    assert got["grads"].dtype == np.float64 and got["state"].dtype == np.float32
    assert 0 < got["state"].size < 5000 and np.isin(got["state"], arrays["state"].numpy()).all()
    for n in got:
        assert np.array_equal(got[n], np.load(str(tmp_path / "b" / (n + ".npy")))), n


def test_row_pack_rule():
    """small-K pointwise convs are read `pack` rows at a time; pack must divide M and only applies below 64 channels"""
    from deepfake_detection_b200.engine import Engine
    assert Engine._row_pack(3211264, 16) == 4 and Engine._row_pack(802816, 24) == 8 and Engine._row_pack(3211264, 32) == 4
    assert Engine._row_pack(200704, 40) == 2 and Engine._row_pack(50176, 80) == 1 and Engine._row_pack(12544, 1152) == 1
    assert Engine._row_pack(802816 + 4, 24) == 4 and Engine._row_pack(7, 16) == 1        # halves until it divides M
    for M in (49, 50, 52, 56):
        for K in (8, 16, 24, 32, 40, 48, 56):
            assert M % Engine._row_pack(M, K) == 0


def test_plan_uses_the_fused_and_packed_kernels():
    """EfficientNet-B0 plan: every expansion block's depthwise backward is ONE fused launch, small-K pointwise convs go
    through the row-packed GEMM with block-diagonal weights registered for refresh, weight gradients use tcgen05."""
    from deepfake_detection_b200.engine import Engine
    eng = Engine("efficientnet_b0", 4, 224, 224, device="plan-only")
    names_f = [op[1] for op in eng.fwd_ops]
    names_b = [op[1] for op in eng.bwd_ops]
    assert names_b.count("dfd_dwconv_bwd") == 16 and "dfd_dwconv_wgrad" not in names_b and "dfd_dwconv_dgrad" not in names_b
    assert names_f.count("dfd_gemm_tn_rowpack") >= 5 and names_b.count("dfd_gemm_tn_rowpack") >= 4
    assert names_b.count("dfd_gemm_wgrad") == 33 and "dfd_gemm_wgrad_mma" not in names_b
    reg = eng._bd_reg
    assert len(reg) == names_f.count("dfd_gemm_tn_rowpack") + names_b.count("dfd_gemm_tn_rowpack")
    for (B, Nn, K, pack), t in reg.items():
        assert t.numel() == pack * Nn * pack * K and (4 * 224 * 224 // 4) % 1 == 0
    # a second plan over the same weights (other batch size) shares the registry of the owner
    eng2 = Engine("efficientnet_b0", 2, 224, 224, device="plan-only", share_from=eng)
    assert eng2.params32 is eng.params32 and not hasattr(eng2, "_bd_reg") and len(eng._bd_reg) >= len(reg)
    # an arena-only engine (what NativeModel.engine / the optimizer hold) owns weights but no plan and no activations
    ar = Engine("efficientnet_b0", 1, device="plan-only", params_only=True)
    assert ar.params_only and ar.fwd_ops == [] and not hasattr(ar, "acts") and ar.n_params == eng.n_params
    eng3 = Engine("efficientnet_b0", 2, 64, 64, device="plan-only", share_from=ar)
    assert eng3.arena is ar and eng3.grads32 is ar.grads32 and len(ar._bd_reg) > 0 and len(ar._stem_reg) == 1
