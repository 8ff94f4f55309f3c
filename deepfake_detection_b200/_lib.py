"""ctypes binding of libdfd_b200.so (the C-ABI of the sm_100a kernels, see include/dfd_b200.h).

There is NO fallback: if the shared library is missing or a symbol is absent, importing / calling raises.
The library is built in-tree by `__graft_entry__.build()` (csrc/Makefile) so that it travels to the GPU box.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdfd_b200.so")

_C = {"p": ctypes.c_void_p, "i": ctypes.c_int, "l": ctypes.c_longlong, "f": ctypes.c_float, "d": ctypes.c_double}

# name -> argument codes (p pointer, i int, l long long, f float, d double); all return int unless noted
SIGNATURES = {
    "dfd_abi_version": "",
    "dfd_stat_slots": "",
    "dfd_memset_async": "pilp",
    "dfd_gemm_tn": "ppplii" "i" "ppp" "p",
    "dfd_gemm_tn_rowpack": "ppplii" "ii" "ppp" "p",
    "dfd_conv_tc": "ppp" "iiiiiiii" "ppp" "p",
    "dfd_conv_wgrad_tc": "ppp" "iiiiiiii" "pl" "p",
    "dfd_conv_wgrad_splits": "iiiiiii",
    "dfd_conv_dgrad_s2_tc": "ppp" "iiiiii" "p",
    "dfd_conv1x1_dgrad_add": "ppp" "iiiiiii" "p",
    "dfd_blockdiag_weights": "piip",
    "dfd_gemm_tn_mma": "pppp" "lii" "i" "ppp",
    "dfd_gemm_wgrad_mma": "ppp" "lii" "i" "p",
    "dfd_gemm_wgrad": "ppp" "lii" "i" "pl" "p",
    "dfd_gemm_wgrad_splits": "lii",
    "dfd_ordered_reduce": "pi" "pi" "p",
    "dfd_dwconv_fwd": "ppppp" "iiiiii" "ii" "ppp" "p",
    "dfd_dwconv_dgrad": "ppppp" "pppppp" "pp" "iiiiii" "ii" "ppp",
    "dfd_dwconv_wgrad": "ppppp" "pppp" "iiiiii" "i" "p",
    "dfd_dwconv_bwd": "ppppp" "pppppp" "ppp" "iiiiii" "i" "pp" "pl" "p" "p",
    "dfd_dwconv_bwd_parts": "iiiiii",
    "dfd_dwconv_block_channels": "i",
    "dfd_stem_fwd": "ppp" "iiiiiiii" "i" "ppp",
    "dfd_stem_wgrad": "ppppppp" "iiiiiiii" "i" "p",
    "dfd_colstats": "p" "ili" "i" "ppp",
    "dfd_bn_finalize": "ppd" "ppppp" "ffii" "ppppp",
    "dfd_bn_act": "pppppp" "ili" "iii" "p",
    "dfd_pool": "pppp" "ili" "ii" "pi" "p",
    "dfd_bn_bwd_reduce": "ppppp" "ili" "i" "ppp" "p",
    "dfd_relu_bn_bwd_reduce": "ppppppp" "ili" "i" "pp" "p",
    "dfd_bn_bwd_finalize": "ppd" "pppppppp" "i" "p",
    "dfd_bn_bwd_apply": "ppppppp" "ili" "i" "p",
    "dfd_se_bwd_reduce": "ppppp" "ili" "i" "p",
    "dfd_act_bwd": "ppppppppp" "ili" "ii" "ppp" "p",
    "dfd_add_inplace": "pp" "li" "p",
    "dfd_se_fc_fwd": "pppppp" "iii" "p",
    "dfd_se_fc_bwd": "pppppp" "pppppppp" "iii" "p",
    "dfd_se_fc_wgrad": "pppp" "pppp" "iii" "p",
    "dfd_pool_se": "pppp" "ppppp" "ili" "iii" "i" "p",
    "dfd_se_bwd_chain": "ppppp" "ppppp" "pppp" "ili" "ii" "p",
    "dfd_head_max_classes": "",
    "dfd_head_fwd": "pppp" "iii" "pp" "ff" "pppp" "p",
    "dfd_head_bwd": "pppppp" "iii" "p",
    "dfd_sgd_step": "ppp" "l" "fffi" "f" "ppp" "i" "p" "p",
    "dfd_adam_step": "pppp" "l" "fffff" "ii" "f" "ppp" "i" "pp" "p",
    "dfd_rmsprop_tf_step": "pppp" "l" "fffff" "f" "ppp" "i" "p" "p",
    "dfd_opt_tick": "pp" "p",
    "dfd_set_floats": "pi" "ffffffff" "p",
    "dfd_ema_update": "ppl" "ppi" "f" "p",
    "dfd_input_normalize": "pppp" "iiii" "i" "p",
    "dfd_rng_masks": "pip" "p",
    "dfd_rng_tick": "p" "p",
    "dfd_mul_f32": "ppl" "p",
    "dfd_cast_arena": "pp" "li" "p",
    "dfd_check_finite": "p" "l" "pp",
    "dfd_update_loss_scale": "ppp" "i" "pp",
    "dfd_transpose_weights": "p" "ii" "p",
    "dfd_im2col": "pp" "iiiiiii" "i" "p",
    "dfd_col2im": "ppp" "iiiiiii" "i" "p",
    "dfd_repack_weights": "p" "ii" "p",
    "dfd_unpack_grad": "pp" "iii" "p",
    "dfd_maxpool_fwd": "ppp" "iiii" "i" "p",
    "dfd_maxpool_bwd": "ppp" "iiii" "i" "p",
    "dfd_relu_bwd": "ppp" "li" "p",
    "dfd_pool_bwd": "pp" "ili" "i" "p",
    "dfd_stem_im2col": "pp" "iiiiiiii" "i" "p",
    "dfd_pad_weight": "pp" "iii" "i" "p",
    "dfd_unpad_grad": "pp" "iii" "p",
}

DT_BF16, DT_FP16 = 0, 1
ACT_NONE, ACT_SWISH, ACT_RELU = 0, 1, 2


class NativeError(RuntimeError):
    pass


class _Lib:
    def __init__(self):
        if not os.path.exists(LIB_PATH):
            raise NativeError(
                "libdfd_b200.so not found at %s: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU / PyTorch fallback for the hot path)" % LIB_PATH)
        self.cdll = ctypes.CDLL(LIB_PATH)
        self.cdll.dfd_last_error.restype = ctypes.c_char_p
        self.cdll.dfd_last_error.argtypes = []
        for name, codes in SIGNATURES.items():
            fn = getattr(self.cdll, name)  # AttributeError if the symbol is missing: fail loudly
            fn.restype = ctypes.c_int
            fn.argtypes = [_C[c] for c in codes]
            setattr(self, name, fn)
        if self.cdll.dfd_abi_version() != 1:
            raise NativeError("libdfd_b200.so ABI version mismatch")
        self.stat_slots = self.cdll.dfd_stat_slots()
        self.head_kmax = self.cdll.dfd_head_max_classes()      # largest num_classes the classifier kernels take

    def last_error(self):
        return self.cdll.dfd_last_error().decode("utf-8", "replace")

    def check(self, rc, what=""):
        if rc != 0:
            raise NativeError("%s failed (%d): %s" % (what or "native call", rc, self.last_error()))


_lib = None
N_CALLS = [0]       # C-ABI calls issued by this process (bench.py reports the count of one step as `gpu_launches`)


def lib():
    global _lib
    if _lib is None:
        _lib = _Lib()
    return _lib


def call(name, *args):
    """Call an entry point, raising NativeError on a non-zero status."""
    L = lib()
    N_CALLS[0] += 1
    rc = getattr(L, name)(*args)
    if rc != 0:
        raise NativeError("%s failed (%d): %s" % (name, rc, L.last_error()))
