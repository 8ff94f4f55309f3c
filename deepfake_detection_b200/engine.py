"""Native train / validate engine: lays the network out in HBM and drives the sm_100a kernels.

This is the host side of the hot path (dfd/runners/train.py:610-649): given an architecture spec it
  * owns the flat fp32 parameter / gradient arenas (reference tensor names, OIHW shapes) plus their 16-bit
    copies in the layouts the kernels read ([Cout,Cin] and transposed [Cin,Cout] for the 1x1 convs),
  * keeps every conv output NHWC in 16-bit (the only activation tensors that touch HBM),
  * builds, once, the ordered list of C-ABI calls ("plan") for forward, backward and the optimizer, and
  * replays the plan on the caller's current CUDA stream (optionally captured into a CUDA graph).

PyTorch is used for device memory and streams only; there is no PyTorch compute on the hot path and no CPU
fallback: constructing an Engine without a CUDA device or without libdfd_b200.so raises.
"""
import ctypes
import numbers
import os
from collections import OrderedDict

import torch

from . import _lib
from .arch import get_spec, is_no_decay, param_entries, state_entries

ACT_NONE, ACT_SWISH, ACT_RELU = _lib.ACT_NONE, _lib.ACT_SWISH, _lib.ACT_RELU
POOL_CHUNKS = 8          # row chunks per image of the pooling kernels when the batch alone cannot fill the GPU


def _ptr(t, off_elems=0):
    return t.data_ptr() + off_elems * t.element_size()


def check_num_classes(num_classes):
    """The classifier kernels take 1 <= num_classes <= DFD_HEAD_KMAX; refused here, before any plan or graph exists.
    0 (timm's identity classifier, pooled features out) has no native path."""
    kmax = _lib.lib().head_kmax
    if not isinstance(num_classes, numbers.Integral) or not 1 <= num_classes <= kmax:
        raise ValueError("num_classes=%r: the native classifier takes 1 <= num_classes <= %d (num_classes=0, the "
                         "identity classifier, is not supported)" % (num_classes, kmax))


class _BN:
    """Pointers of one BatchNorm layer (parameters, running stats, per-step statistics, bwd coefficients)."""
    __slots__ = ("name", "C", "gamma", "beta", "dgamma", "dbeta", "rm", "rv", "nbt", "scale", "shift", "mean",
                 "rstd", "cA", "cB", "cC", "fsum", "fsq", "bs1", "bs2", "fin", "bfin", "count", "idx", "fused", "stat_off")


class Engine:
    def __init__(self, arch, batch, height=None, width=None, num_classes=2, in_chans=3, dtype="bf16",
                 bn_momentum=0.1, bn_eps=1e-5, device=None, gemm_impl="tc", share_from=None, stem_impl="gemm",
                 params_only=False, drop_rate=0.0, drop_path_rate=0.0, sync_bn=False):
        # _plan_only: build the arenas and the call plan on the CPU for host-logic tests; nothing can be executed
        self._plan_only = device == "plan-only"
        if self._plan_only:
            device = "cpu"
        elif not torch.cuda.is_available():
            raise _lib.NativeError("deepfake_detection_b200.Engine needs a CUDA device (B200, sm_100a); "
                                   "there is no CPU path")
        self.L = _lib.lib()
        check_num_classes(num_classes)
        self.spec = spec = get_spec(arch, num_classes=num_classes, in_chans=in_chans)
        self.cls_name = "classifier" if spec.family == "efficientnet" else "fc"
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.N = int(batch)
        self.H = int(height or spec.input_size[1])
        self.W = int(width or spec.input_size[2])
        if dtype in ("bf16", "bfloat16", torch.bfloat16):
            self.dt, self.tdtype = _lib.DT_BF16, torch.bfloat16
        elif dtype in ("fp16", "float16", "half", torch.float16):
            self.dt, self.tdtype = _lib.DT_FP16, torch.float16
        else:
            raise ValueError("dtype %r: the native path computes in 'bf16' or 'fp16' (fp32 master weights)" % (dtype,))
        self.drop_rate = float(drop_rate)
        self.drop_path_rate = float(drop_path_rate)
        # synchronised BatchNorm (train.py:388-400 `convert_syncbn_model`): batch statistics and the BN-backward sums are
        # all-reduced over the process group between the kernel that produces them and the finalisation
        self.sync_bn = bool(sync_bn)
        self.sync_world = 1
        if self.sync_bn:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                self.sync_world = dist.get_world_size()
            self.sync_bn = self.sync_world > 1
        self.bn_momentum = float(bn_momentum)
        self.bn_eps = float(bn_eps)
        self.gemm_impl = gemm_impl
        # 1x1 weight gradient: tcgen05 with MN-major operands, or the mma.sync cross-check path
        self._wgrad_name = "dfd_gemm_wgrad" if gemm_impl == "tc" and not os.environ.get("DFD_WGRAD_MMA") else "dfd_gemm_wgrad_mma"
        self.stem_impl = stem_impl
        self.training = True
        self.n_launch = {"fwd": 0, "bwd": 0, "opt": 0}
        self._shared_from = share_from
        if share_from is not None:
            # a second plan (other batch size / resolution, e.g. the validation loader) over the SAME weights,
            # gradients and running statistics
            if share_from.spec.arch != spec.arch or share_from.dt != self.dt:
                raise ValueError("share_from: architecture / dtype mismatch")
            share_from = self._shared_from = share_from.arena
            for a in ("p_off", "n_decay", "n_params", "param_names", "params32", "grads32", "params16", "b_off", "bn_names",
                      "buffers32", "nbt", "t_off", "paramsT16", "_ttable", "_ttable_count", "loss_scale_state", "flags",
                      "rng_state"):
                setattr(self, a, getattr(share_from, a))
        else:
            self._layout_params()
            self.loss_scale_state = torch.ones(2, dtype=torch.float32, device=self.device)   # scale, 1/scale
            self.flags = torch.zeros(2, dtype=torch.int32, device=self.device)              # found_inf, good_steps
            # counter-based generator state of the dropout / drop-path masks: [seed, step]; the step advances on the device
            self.rng_state = torch.zeros(2, dtype=torch.int64, device=self.device)
            self.rng_state[0] = torch.initial_seed() & 0x7FFFFFFFFFFFFFFF          # follows torch.manual_seed (train.py:299)
            self._derived_dirty = False
            # bumped whenever weights or BN running statistics change (load, a training forward, EMA / distribute_bn): an
            # eval-mode plan recomputes its per-channel scale / shift vectors only when this moved (see forward)
            self.state_version = 0
        self._eval_version = -1
        self.params_only = bool(params_only)
        self._red_pending, self._ws_bytes = [], 0
        if self.params_only:
            # the owner of the parameter / gradient / running-statistic arenas without any activation plan: what
            # `NativeModel.engine`, the optimizer and the EMA need (a plan is built per (batch, H, W) that reaches forward)
            self.fwd_ops, self.bwd_ops = [], []
            return
        self._build()
        if not self._plan_only and self.arena._derived_dirty:
            # this plan registered new derived weight layouts with the owner: fill them now (never inside a graph capture)
            self.refresh_weight_layouts(torch.cuda.current_stream().cuda_stream)

    # ------------------------------------------------------------------------------------------
    # parameter / buffer arenas
    # ------------------------------------------------------------------------------------------
    def _layout_params(self):
        spec, dev = self.spec, self.device
        entries = param_entries(spec)
        decay = [(n, s) for n, s, _ in entries if not is_no_decay(n, s)]
        nodecay = [(n, s) for n, s, _ in entries if is_no_decay(n, s)]
        self.p_off = OrderedDict()
        off = 0
        for n, s in decay + nodecay:
            numel = 1
            for d in s:
                numel *= d
            self.p_off[n] = (off, tuple(s), numel)
            off += (numel + 3) // 4 * 4          # keep every tensor 16-byte aligned in fp32 and 8-byte in 16-bit
            if n == decay[-1][0]:
                off = (off + 7) // 8 * 8
                self.n_decay = off
        self.n_params = off
        self.param_names = [n for n, _, _ in entries]
        self.params32 = torch.zeros(off, dtype=torch.float32, device=dev)
        self.grads32 = torch.zeros(off, dtype=torch.float32, device=dev)
        self.params16 = torch.zeros(off, dtype=self.tdtype, device=dev)
        # buffers (running stats): flat fp32 + int64 counters
        self.b_off = OrderedDict()
        boff = 0
        self.bn_names = []
        for n, s, role in state_entries(spec):
            if role in ("bn_rm", "bn_rv"):
                self.b_off[n] = (boff, s[0])
                boff += (s[0] + 3) // 4 * 4
            elif role == "bn_nbt":
                self.bn_names.append(n[: -len(".num_batches_tracked")])
        self.buffers32 = torch.zeros(boff, dtype=torch.float32, device=dev)
        for n, (o, c) in self.b_off.items():
            if n.endswith("running_var"):
                self.buffers32[o:o + c] = 1.0
        self.nbt = torch.zeros(len(self.bn_names), dtype=torch.int64, device=dev)
        # transposed 16-bit copies of the 1x1 conv weights (dgrad B operand)
        self.t_off = OrderedDict()
        toff = 0
        for n, s, role in entries:
            if role == "conv_w" and s[2] == 1 and s[3] == 1:
                self.t_off[n] = (toff, s[0], s[1])
                toff += (s[0] * s[1] + 7) // 8 * 8
        self.paramsT16 = torch.zeros(max(toff, 8), dtype=self.tdtype, device=dev)
        import struct
        raw = b"".join(struct.pack("<QQii", _ptr(self.params16, self.p_off[n][0]), _ptr(self.paramsT16, o), O, I)
                       for n, (o, O, I) in self.t_off.items())
        self._ttable = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(dev)
        self._ttable_count = len(self.t_off)

    @property
    def arena(self):
        """the engine that owns the weights, gradients, running statistics and derived weight layouts"""
        return self._shared_from if self._shared_from is not None else self

    def param_view(self, name):
        o, s, n = self.p_off[name]
        return self.params32[o:o + n].view(s)

    def grad_view(self, name):
        o, s, n = self.p_off[name]
        return self.grads32[o:o + n].view(s)

    def buffer_view(self, name):
        if name.endswith("num_batches_tracked"):
            return self.nbt[self.bn_names.index(name[: -len(".num_batches_tracked")])]
        o, c = self.b_off[name]
        return self.buffers32[o:o + c]

    def state_dict(self):
        """Reference-layout state dict (fp32 master weights, OIHW), a copy."""
        sd = OrderedDict()
        for n, s, role in state_entries(self.spec):
            if role in ("bn_rm", "bn_rv", "bn_nbt"):
                sd[n] = self.buffer_view(n).clone()
            else:
                sd[n] = self.param_view(n).clone()
        return sd

    def load_state_dict(self, sd, strict=True):
        missing = []
        with torch.no_grad():
            for n, s, role in state_entries(self.spec):
                if n not in sd:
                    missing.append(n)
                    continue
                src = sd[n].to(self.device)
                if role in ("bn_rm", "bn_rv"):
                    self.buffer_view(n).copy_(src.float())
                elif role == "bn_nbt":
                    self.nbt[self.bn_names.index(n[: -len(".num_batches_tracked")])] = int(src)
                else:
                    self.param_view(n).copy_(src.float().reshape(self.p_off[n][1]))
        if strict and missing:
            raise KeyError("missing keys in state_dict: %s" % missing[:5])
        self.sync_weights()
        return missing

    def sync_weights(self):
        """fp32 master -> 16-bit kernel copies (call after any out-of-band weight change)."""
        self.arena.state_version += 1
        st = torch.cuda.current_stream().cuda_stream
        _lib.call("dfd_cast_arena", _ptr(self.params32), _ptr(self.params16), self.n_params, self.dt, st)
        self.refresh_weight_layouts(st)

    # ------------------------------------------------------------------------------------------
    # plan construction
    # ------------------------------------------------------------------------------------------
    # ---- order-deterministic weight gradients ------------------------------------------------------------------
    # The tcgen05 weight gradient and the fused depthwise backward run in WORKSPACE mode: every CTA stores its split partial
    # sum in a fixed slot of one workspace (plain stores, no atomics) and `dfd_ordered_reduce` - one table-driven launch per
    # block of the network, right behind that block's backward ops - adds the partials into the gradient arena in slot
    # order. Gradients (and with them every later step) therefore do not depend on the arrival order of CTAs; the reduce
    # launches are also the points at which a block's gradients become final for the DDP bucketing.
    # DFD_NONDET=1 switches back to the atomic flushes (diagnostics / timing comparison).
    def _wgrad(self, G, X, dW, M, Nw, Kw):
        if self._wgrad_name != "dfd_gemm_wgrad":
            return (self._wgrad_name, (G, X, dW, M, Nw, Kw, self.dt))
        if os.environ.get("DFD_NONDET"):
            return ("dfd_gemm_wgrad", (G, X, dW, M, Nw, Kw, self.dt, None, 0))
        splits = self.L.cdll.dfd_gemm_wgrad_splits(M, Nw, Kw)
        off, nbytes = self._ws_take(splits * Nw * Kw * 4)
        self._red_pending.append((off, dW, Nw * Kw, Nw * Kw, splits))
        return ("dfd_gemm_wgrad", [G, X, dW, M, Nw, Kw, self.dt, ("WS", off), nbytes])

    def _wgrad_conv(self, dY, X, dW, N, H, W, Cin, Cout, k, stride=1):
        """implicit-GEMM weight gradient of a dense k x k convolution (H, W = input extents) into the packed
        [Cout][kh][kw][Cin] fp32 buffer"""
        Kw = k * k * Cin
        if os.environ.get("DFD_NONDET"):
            return ("dfd_conv_wgrad_tc", (dY, X, dW, N, H, W, Cin, Cout, k, stride, self.dt, None, 0))
        splits = self.L.cdll.dfd_conv_wgrad_splits(N, H, W, Cin, Cout, k, stride)
        off, nbytes = self._ws_take(splits * Cout * Kw * 4)
        self._red_pending.append((off, dW, Cout * Kw, Cout * Kw, splits))
        return ("dfd_conv_wgrad_tc", [dY, X, dW, N, H, W, Cin, Cout, k, stride, self.dt, ("WS", off), nbytes])

    def _dw_bwd(self, args, N, H, W, C, k, stride, fin=None):
        if os.environ.get("DFD_NONDET"):
            return ("dfd_dwconv_bwd", list(args) + [None, 0, fin])
        parts = self.L.cdll.dfd_dwconv_bwd_parts(N, H, W, C, k, stride)
        cw = self.L.cdll.dfd_dwconv_block_channels(C)          # channels per CTA: 64, or 32 / 16 for C = 32, 96 / 144
        cbs = (C + cw - 1) // cw
        off, nbytes = self._ws_take(cbs * parts * cw * k * k * 4)
        dW = args[13]
        for cb in range(cbs):
            n = min(cw, C - cw * cb) * k * k
            self._red_pending.append((off + cb * parts * cw * k * k * 4, dW + cb * cw * k * k * 4, n, cw * k * k, parts))
        return ("dfd_dwconv_bwd", list(args) + [("WS", off), nbytes, fin])

    def _ws_take(self, nbytes):
        off = getattr(self, "_ws_bytes", 0)
        self._ws_bytes = off + (nbytes + 255) // 256 * 256
        return off, nbytes

    def _flush_reduce(self, ops):
        """emit the ordered-reduce launch for the partial sums produced since the last flush (call at block boundaries)"""
        pend = self.__dict__.setdefault("_red_pending", [])
        if pend:
            ops.append(("dfd_ordered_reduce", ["REDUCE", list(pend)]))
            del pend[:]

    def _patch_workspace(self, ops):
        import struct
        self._flush_reduce(ops)
        total = getattr(self, "_ws_bytes", 0)
        if not total:
            return ops
        self.det_ws = torch.empty(total // 4, dtype=torch.float32, device=self.device)
        base = _ptr(self.det_ws)
        entries = [e for n, a in ops if n == "dfd_ordered_reduce" for e in a[1]]
        raw = b"".join(struct.pack("<QQqqii", base + off, dst, n, stride, parts, 0) for off, dst, n, stride, parts in entries)
        self._red_table = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(self.device)
        out, pos = [], 0
        for n, a in ops:
            if n == "dfd_ordered_reduce":
                ents = a[1]
                bx = max((e[2] // 4 + 7) // 8 if e[4] > 64 else (e[2] // 4 + 255) // 256 for e in ents)
                a = (_ptr(self._red_table, pos * 40), len(ents), min(e[1] for e in ents), max(1, min(bx, 1024)))
                pos += len(ents)
            elif isinstance(a, list):
                a = [base + v[1] if isinstance(v, tuple) and v[0] == "WS" else v for v in a]
            out.append((n, a))
        return out

    def _alloc16(self, *shape):
        # the plan holds RAW pointers: every buffer must stay referenced for the engine's lifetime
        t = torch.empty(shape, dtype=self.tdtype, device=self.device)
        self._keep.append(t)
        return t

    # rows of A fused per TMA row for small-K pointwise convs, measured on B200 at batch 256 (tools/gemm_time2.py): the best
    # factor makes pack*K a multiple of the 64-element k-block where that keeps pack*N modest
    _ROW_PACK = {8: 8, 16: 4, 24: 8, 32: 4, 40: 2, 48: 4, 56: 2}

    @classmethod
    def _row_pack(cls, M, K):
        """rows of A read as one (dfd_gemm_tn_rowpack): keeps the TMA rows of small-K pointwise convs at >= 128 bytes"""
        if os.environ.get("DFD_NO_ROWPACK"):
            return 1
        pack = cls._ROW_PACK.get(K, 1)
        while pack > 1 and M % pack:
            pack //= 2
        return pack

    # Derived 16-bit weight layouts (block-diagonal small-K copies, the padded stem weight, the packed k x k weights of
    # the ResNet path) are registered with, owned by and refreshed through the ARENA engine, whichever plan asked for them:
    # the optimizer refreshes them once per step for every plan that shares the weights.
    def _upload_fin_descs(self):
        """fill the BatchNorm finalisation descriptors once the plan knows every layer's element count"""
        import struct
        n = len(self.bns)
        raw = bytearray(2 * n * 128)
        for bn in self.bns.values():
            if bn.count is None:
                continue
            cnt = float(bn.count)
            unb = cnt / (cnt - 1.0) if cnt > 1 else 1.0
            struct.pack_into("<12Qddffii", raw, bn.idx * 128, bn.fsum, bn.fsq, bn.gamma, bn.beta, bn.rm, bn.rv, bn.nbt, bn.scale,
                             bn.shift, bn.mean, bn.rstd, _ptr(self._fin_tickets, bn.idx), 1.0 / cnt, unb, self.bn_momentum,
                             self.bn_eps, bn.C, 0)
            struct.pack_into("<11Qdii", raw, (n + bn.idx) * 128, bn.bs1, bn.bs2, bn.gamma, bn.mean, bn.rstd, bn.dgamma, bn.dbeta,
                             bn.cA, bn.cB, bn.cC, _ptr(self._fin_tickets, n + bn.idx), 1.0 / cnt, bn.C, 0)
        self._fin_buf.copy_(torch.frombuffer(raw, dtype=torch.int32).to(self._fin_buf.device))

    def _blockdiag(self, B, Nn, K, pack):
        """block-diagonal [pack*Nn, pack*K] copy of the weight at B"""
        o = self.arena
        reg = o.__dict__.setdefault("_bd_reg", OrderedDict())
        key = (B, Nn, K, pack)
        if key not in reg:
            reg[key] = torch.zeros(pack * Nn * pack * K, dtype=self.tdtype, device=self.device)
            o._bd_table = None
            o._derived_dirty = True
        return _ptr(reg[key])

    def refresh_weight_layouts(self, stream):
        """derived 16-bit weight layouts (transposed 1x1, packed k x k, block-diagonal small-K) from the 16-bit arena"""
        o = self.arena
        _lib.call("dfd_transpose_weights", _ptr(o._ttable), o._ttable_count, o.dt, stream)
        reg = getattr(o, "_bd_reg", None)
        if reg and getattr(o, "_bd_table", None) is None:
            import struct
            raw = b"".join(struct.pack("<QQiiii", B, _ptr(t), Nn, K, pack, 0) for (B, Nn, K, pack), t in reg.items())
            o._bd_table = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(o.device)
        if getattr(o, "_rtable_count", 0):
            _lib.call("dfd_repack_weights", _ptr(o._rtable), o._rtable_count, o.dt, stream)
        for (name, O, taps, Kp), wpad in getattr(o, "_stem_reg", {}).items():
            _lib.call("dfd_pad_weight", _ptr(o.params16, o.p_off[name][0]), _ptr(wpad), O, taps, Kp, o.dt, stream)
        if reg:
            _lib.call("dfd_blockdiag_weights", _ptr(o._bd_table), len(reg), o.dt, stream)
        o._derived_dirty = False

    def _stem_gemm_setup(self, wname, Cout, k, M):
        """stem convolution as im2col + tcgen05 GEMM (K = Cin*k*k padded to a multiple of 8)"""
        taps = self.spec.in_chans * k * k
        Kp = (taps + 7) // 8 * 8
        o = self.arena
        reg = o.__dict__.setdefault("_stem_reg", OrderedDict())
        key = (wname, Cout, taps, Kp)
        if key not in reg:
            reg[key] = torch.zeros(Cout * Kp, dtype=self.tdtype, device=self.device)
            o._derived_dirty = True
        self.stem_wpad = reg[key]
        self.stem_gpad = torch.zeros(Cout * Kp, dtype=torch.float32, device=self.device)
        self.stem_cols = self._alloc16(M, Kp)
        return taps, Kp

    def _alloc_bn(self, bn_specs):
        """per-BN pointers into the parameter / running-stat arenas + the per-step statistic and coefficient arenas"""
        dev, S = self.device, self.L.stat_slots
        tot_c = sum((c + 3) // 4 * 4 for _, c in bn_specs)
        self.bnstate = torch.zeros(7 * tot_c, dtype=torch.float32, device=dev)      # scale shift mean rstd cA cB cC
        self.stats = torch.zeros(4 * S * tot_c + 8, dtype=torch.float64, device=dev)  # fsum fsq bs1 bs2 (+ loss/correct)
        self.bns = {}
        co = 0
        # finalisation descriptors (csrc/bn_finalize.cuh: BnFinDesc / BnBwdFinDesc, 128-byte stride) + one ticket each: the
        # last CTA of the kernel that produced a layer's statistics finalises that BatchNorm (no one-block launches)
        self._fin_buf = torch.zeros(2 * len(bn_specs) * 32, dtype=torch.int32, device=dev)
        self._fin_tickets = torch.zeros(2 * len(bn_specs), dtype=torch.int32, device=dev)
        for bi, (name, c) in enumerate(bn_specs):
            bn = _BN()
            bn.name, bn.C = name, c
            bn.idx, bn.count, bn.fused = bi, None, False
            bn.fin = _ptr(self._fin_buf, bi * 32)
            bn.bfin = _ptr(self._fin_buf, (len(bn_specs) + bi) * 32)
            bn.gamma = _ptr(self.params32, self.p_off[name + ".weight"][0])
            bn.beta = _ptr(self.params32, self.p_off[name + ".bias"][0])
            bn.dgamma = _ptr(self.grads32, self.p_off[name + ".weight"][0])
            bn.dbeta = _ptr(self.grads32, self.p_off[name + ".bias"][0])
            bn.rm = _ptr(self.buffers32, self.b_off[name + ".running_mean"][0])
            bn.rv = _ptr(self.buffers32, self.b_off[name + ".running_var"][0])
            bn.nbt = _ptr(self.nbt, self.bn_names.index(name))
            for i, f in enumerate(("scale", "shift", "mean", "rstd", "cA", "cB", "cC")):
                setattr(bn, f, _ptr(self.bnstate, i * tot_c + co))
            # per layer [fsum | fsq | bs1 | bs2], S slots x C doubles each: the forward pair and the backward pair are contiguous
            # (one collective each under synchronised BatchNorm)
            for i, f in enumerate(("fsum", "fsq", "bs1", "bs2")):
                setattr(bn, f, _ptr(self.stats, (4 * co + i * c) * S))
            bn.stat_off = 4 * co * S
            co += (c + 3) // 4 * 4
            self.bns[name] = bn
        self.scalars = torch.zeros(4, dtype=torch.float32, device=dev)     # loss_acc, correct_acc, (spare)


    def _build(self):
        if self.spec.family == "resnet":
            from .engine_resnet import build_resnet
            return build_resnet(self)
        spec, N, dev, L = self.spec, self.N, self.device, self.L
        S = L.stat_slots
        self._keep = []
        self.acts = {}
        fwd, bwd = [], []
        bn_list = []

        # ---- pass 1: shapes --------------------------------------------------------------------
        Hs = (self.H + 2 - 3) // 2 + 1
        Ws = (self.W + 2 - 3) // 2 + 1
        blocks = []
        h, w = Hs, Ws
        for b in spec.blocks:
            ho = (h + 2 * b.pad - b.k) // b.stride + 1
            wo = (w + 2 * b.pad - b.k) // b.stride + 1
            blocks.append((b, h, w, ho, wo))
            h, w = ho, wo
        Hf, Wf = h, w

        # ---- BN bookkeeping arenas ---------------------------------------------------------------
        bn_specs = [("bn1", spec.stem)]
        for b in spec.blocks:
            if b.kind == "ir":
                bn_specs += [(b.name + ".bn1", b.cmid), (b.name + ".bn2", b.cmid), (b.name + ".bn3", b.cout)]
            else:
                bn_specs += [(b.name + ".bn1", b.cmid), (b.name + ".bn2", b.cout)]
        bn_specs.append(("bn2", spec.num_features))
        self._alloc_bn(bn_specs)

        P32 = lambda n: _ptr(self.params32, self.p_off[n][0])
        G32 = lambda n: _ptr(self.grads32, self.p_off[n][0])
        P16 = lambda n: _ptr(self.params16, self.p_off[n][0])
        T16 = lambda n: _ptr(self.paramsT16, self.t_off[n][0])
        dt = self.dt
        mom, eps = self.bn_momentum, self.bn_eps

        # BatchNorm finalisation by the last CTA of the statistics-producing kernel (descriptors, csrc/bn_finalize.cuh) instead of
        # 98 one-block launches: implemented and tested, but MEASURED SLOWER inside the captured graph (17.29 vs 16.69 ms per
        # B0 step): every CTA pays a __threadfence + a same-address ticket atomic before it may retire (the depthwise kernels
        # run ~14k short CTAs), and the one finalising CTA walks C channels with a fraction of the threads of the standalone
        # launch. Off unless DFD_FUSED_FINALIZE=1.
        # DFD_FUSED_FINALIZE=gemm: only the BatchNorms whose statistics come from the persistent tcgen05 GEMM (148 CTAs: the
        # ticket is free there) are finalised by their producer - MEASURED slower too (15.38 vs 15.30 ms: one CTA finalising C
        # channels is a longer dependent chain than the standalone launch); =1: every producer, forward and backward.
        ff_mode = os.environ.get("DFD_FUSED_FINALIZE", "")
        fused_fin = ff_mode not in ("", "0", "gemm") and not self.sync_bn
        fused_gemm = (fused_fin or ff_mode == "gemm") and not self.sync_bn

        def gemm(A, B, C, M, Nn, K, bn=None):
            fs, fq = (bn.fsum, bn.fsq) if bn is not None else (None, None)
            if self.gemm_impl == "tc":
                fin = bn.fin if (bn is not None and fused_gemm) else None
                if bn is not None:
                    bn.fused = fin is not None
                pack = self._row_pack(M, K)
                if pack > 1:
                    return ("dfd_gemm_tn_rowpack", (A, self._blockdiag(B, Nn, K, pack), C, M, Nn, K, pack, dt, fs, fq, fin))
                return ("dfd_gemm_tn", (A, B, C, M, Nn, K, dt, fs, fq, fin))
            return ("dfd_gemm_tn_mma", (A, B, C, None, M, Nn, K, dt, fs, fq))

        def finalize(bn, count):
            # Training: the producing kernel's last CTA finalises (descriptor bn.fin), this op is skipped (see _run); it runs
            # in eval mode (running statistics -> scale / shift, once per weight state) and when the producer cannot finalise.
            bn.count = count
            if self.sync_bn:
                # SUM of every rank's statistics, finalised against the GLOBAL element count (torch SyncBatchNorm semantics)
                fwd.append(("ALLREDUCE_train", (self.stats[bn.stat_off:bn.stat_off + 2 * S * bn.C], "sum")))
                return ("dfd_bn_finalize_sync", [bn.fsum, bn.fsq, float(count), bn.gamma, bn.beta, bn.rm, bn.rv, bn.nbt, mom, eps,
                                                 "TRAINING", bn.C, bn.scale, bn.shift, bn.mean, bn.rstd])
            return ("dfd_bn_finalize" + ("_evalonly" if bn.fused else ""),
                    [bn.fsum, bn.fsq, float(count), bn.gamma, bn.beta, bn.rm, bn.rv, bn.nbt, mom, eps,
                     "TRAINING", bn.C, bn.scale, bn.shift, bn.mean, bn.rstd])

        def bwd_finalize(bn, count):
            bn.count = count
            if self.sync_bn:
                # MEAN over the ranks of (sum g, sum g*xhat) with the LOCAL count: the coefficients of dy then use the global
                # means, and dgamma / dbeta receive global_sum / world - what the DDP gradient mean of the per-rank sums gives
                bwd.append(("ALLREDUCE", (self.stats[bn.stat_off + 2 * S * bn.C:bn.stat_off + 4 * S * bn.C], "avg")))
                return ("dfd_bn_bwd_finalize", (bn.bs1, bn.bs2, float(count), bn.gamma, bn.mean, bn.rstd, bn.dgamma, bn.dbeta,
                                                bn.cA, bn.cB, bn.cC, bn.C))
            if fused_fin:
                return None         # done by the last CTA of the kernel that produced bs1 / bs2 (descriptor bn.bfin)
            return ("dfd_bn_bwd_finalize", (bn.bs1, bn.bs2, float(count), bn.gamma, bn.mean, bn.rstd, bn.dgamma, bn.dbeta,
                                            bn.cA, bn.cB, bn.cC, bn.C))

        BF = (lambda bn: bn.bfin) if fused_fin else (lambda bn: None)
        def FF(bn):         # forward producer other than the GEMM (depthwise conv): fused finalisation of its BatchNorm
            bn.fused = fused_fin
            return bn.fin if fused_fin else None

        # ---- scratch for backward ----------------------------------------------------------------
        mid_max = max([N * h * w * b.cmid for b, h, w, ho, wo in blocks if b.kind == "ir"] +
                      [N * ho * wo * b.cmid for b, h, w, ho, wo in blocks] + [N * Hf * Wf * spec.num_features] +
                      [N * Hs * Ws * spec.stem])
        small_max = max([N * h * w * b.cin for b, h, w, ho, wo in blocks] +
                        [N * ho * wo * b.cout for b, h, w, ho, wo in blocks])
        self.mid = [self._alloc16(mid_max) for _ in range(2)]
        self.small = [self._alloc16(small_max) for _ in range(3)]
        mid_a, mid_b = _ptr(self.mid[0]), _ptr(self.mid[1])
        sm = [_ptr(t) for t in self.small]
        se_max_c = max([b.cmid for b in spec.blocks if b.cse] + [8])
        se_max_r = max([b.cse for b in spec.blocks if b.cse] + [8])
        self.se_tmp = torch.zeros(3 * N * se_max_c + 2 * N * se_max_r, dtype=torch.float32, device=dev)
        se_draw = _ptr(self.se_tmp)
        self.pool_partial = torch.zeros(POOL_CHUNKS * N * max(se_max_c, spec.num_features), dtype=torch.float32, device=dev)
        se_de = _ptr(self.se_tmp, N * se_max_c)
        se_dpool = _ptr(self.se_tmp, 2 * N * se_max_c)
        se_r = _ptr(self.se_tmp, 3 * N * se_max_c)
        se_drp = _ptr(self.se_tmp, 3 * N * se_max_c + N * se_max_r)

        # ---- forward -----------------------------------------------------------------------------
        self.x_in = torch.zeros(N, spec.in_chans, self.H, self.W, dtype=self.tdtype, device=dev)
        y0 = self._alloc16(N, Hs, Ws, spec.stem)
        stem_out = self._alloc16(N, Hs, Ws, spec.stem)
        self.acts["conv_stem"] = y0
        self.acts["stem.out"] = stem_out
        bn = self.bns["bn1"]
        if self.stem_impl == "gemm":
            taps, Kp = self._stem_gemm_setup("conv_stem.weight", spec.stem, 3, N * Hs * Ws)
            fwd.append(("dfd_stem_im2col", (_ptr(self.x_in), _ptr(self.stem_cols), N, spec.in_chans, self.H, self.W, 3, 2, 1, Kp, dt)))
            fwd.append(gemm(_ptr(self.stem_cols), _ptr(self.stem_wpad), _ptr(y0), N * Hs * Ws, spec.stem, Kp, bn))
        else:
            fwd.append(("dfd_stem_fwd", (_ptr(self.x_in), P32("conv_stem.weight"), _ptr(y0), N, spec.in_chans, self.H, self.W,
                                         spec.stem, 3, 2, 1, dt, bn.fsum, bn.fsq)))
        fwd.append(finalize(bn, N * Hs * Ws))
        fwd.append(("dfd_bn_act", (_ptr(y0), bn.scale, bn.shift, None, None, _ptr(stem_out), N, Hs * Ws, spec.stem,
                                   ACT_SWISH, 0, dt)))
        x = stem_out
        recs = []
        # stochastic regularisation (train mode only): per-sample drop-path scale of every residual block
        # (rate = drop_path_rate * block_idx / n_blocks, efficientnet_builder.py:228-230,343) and the classifier dropout mask;
        # the gates are [N, C] fp32 tensors (one draw per sample replicated over the channels) filled by ONE dfd_rng_masks
        # launch at the head of the forward plan, consumed through the GATE operand of dfd_bn_act
        masks = []               # (tensor, rows, width, keep_prob)
        n_blocks = len(blocks)
        ones_c = zeros_c = None
        for bi, (b, h, w, ho, wo) in enumerate(blocks):
            p = b.name
            M1, M2 = N * h * w, N * ho * wo
            rec = dict(b=b, h=h, w=w, ho=ho, wo=wo, x=x)
            if b.kind == "ir":
                bn1, bn2, bn3 = self.bns[p + ".bn1"], self.bns[p + ".bn2"], self.bns[p + ".bn3"]
                y1 = self._alloc16(N, h, w, b.cmid)
                self.acts[p + ".conv_pw"] = y1
                fwd.append(gemm(_ptr(x), P16(p + ".conv_pw.weight"), _ptr(y1), M1, b.cmid, b.cin, bn1))
                fwd.append(finalize(bn1, M1))
                dw_in, dw_bn, bn_mid, bn_out, pw_name = y1, bn1, bn2, bn3, ".conv_pwl"
                rec.update(y1=y1)
            else:
                dw_in, dw_bn, bn_mid, bn_out, pw_name = x, None, self.bns[p + ".bn1"], self.bns[p + ".bn2"], ".conv_pw"
            y2 = self._alloc16(N, ho, wo, b.cmid)
            self.acts[p + ".conv_dw"] = y2
            fwd.append(("dfd_dwconv_fwd", (_ptr(dw_in), dw_bn.scale if dw_bn else None, dw_bn.shift if dw_bn else None,
                                           P32(p + ".conv_dw.weight"), _ptr(y2), N, h, w, b.cmid, b.k, b.stride,
                                           ACT_SWISH if dw_bn else ACT_NONE, dt, bn_mid.fsum, bn_mid.fsq, FF(bn_mid))))
            fwd.append(finalize(bn_mid, M2))
            gate_ptr = None
            if b.cse:
                pooled = torch.zeros(N, b.cmid, dtype=torch.float32, device=dev)
                gate = torch.zeros(N, b.cmid, dtype=torch.float32, device=dev)
                self._keep += [pooled, gate]
                rec.update(pooled=pooled, gate=gate)
                if os.environ.get("DFD_SE_FUSED"):
                    # squeeze + excite in ONE launch (the CTA that completes an image's pooled vector runs its FC chain):
                    # measured SLOWER than the two launches (+0.2 ms per step: a 256-thread CTA walks the latency-bound chain
                    # four times longer than the 1024-thread FC kernel and the tail is not hidden); kept selectable
                    fwd.append(("dfd_pool_se", (_ptr(y2), bn_mid.scale, bn_mid.shift, _ptr(pooled), P32(p + ".se.conv_reduce.weight"),
                                                P32(p + ".se.conv_reduce.bias"), P32(p + ".se.conv_expand.weight"),
                                                P32(p + ".se.conv_expand.bias"), _ptr(gate), N, ho * wo, b.cmid, b.cse, ACT_SWISH, dt,
                                                POOL_CHUNKS)))
                else:
                    fwd.append(("dfd_pool", (_ptr(y2), bn_mid.scale, bn_mid.shift, _ptr(pooled), N, ho * wo, b.cmid, ACT_SWISH, dt,
                                             None, POOL_CHUNKS)))
                    fwd.append(("dfd_se_fc_fwd", (_ptr(pooled), P32(p + ".se.conv_reduce.weight"), P32(p + ".se.conv_reduce.bias"),
                                                  P32(p + ".se.conv_expand.weight"), P32(p + ".se.conv_expand.bias"),
                                                  _ptr(gate), N, b.cmid, b.cse)))
                gate_ptr = _ptr(gate)
            a2 = self._alloc16(N, ho, wo, b.cmid)
            fwd.append(("dfd_bn_act", (_ptr(y2), bn_mid.scale, bn_mid.shift, gate_ptr, None, _ptr(a2), N, ho * wo, b.cmid,
                                       ACT_SWISH, 0, dt)))
            y3 = self._alloc16(N, ho, wo, b.cout)
            self.acts[p + pw_name] = y3
            fwd.append(gemm(_ptr(a2), P16(p + pw_name + ".weight"), _ptr(y3), M2, b.cout, b.cmid, bn_out))
            fwd.append(finalize(bn_out, M2))
            out = self._alloc16(N, ho, wo, b.cout)
            self.acts[p + ".out"] = out
            dp_rate = self.drop_path_rate * bi / n_blocks if b.has_residual else 0.0
            dp_gate = None
            if dp_rate > 0.0:
                dp_gate = torch.ones(N, b.cout, dtype=torch.float32, device=dev)
                self._keep.append(dp_gate)
                masks.append((dp_gate, N, b.cout, 1.0 - dp_rate))
            fwd.append(("dfd_bn_act", [_ptr(y3), bn_out.scale, bn_out.shift, ("TRAIN_ONLY", _ptr(dp_gate)) if dp_gate is not None else None,
                                       _ptr(x) if b.has_residual else None,
                                       _ptr(out), N, ho * wo, b.cout, ACT_NONE, 1 if b.has_residual else 0, dt]))
            rec.update(y2=y2, a2=a2, y3=y3, out=out, dw_bn=dw_bn, bn_mid=bn_mid, bn_out=bn_out, pw_name=pw_name, dp_gate=dp_gate)
            recs.append(rec)
            x = out
        # head
        F = spec.num_features
        Mf = N * Hf * Wf
        bnh = self.bns["bn2"]
        yh = self._alloc16(N, Hf, Wf, F)
        self.acts["conv_head"] = yh
        fwd.append(gemm(_ptr(x), P16("conv_head.weight"), _ptr(yh), Mf, F, spec.head_in, bnh))
        fwd.append(finalize(bnh, Mf))
        self.pooled = torch.zeros(N, F, dtype=torch.float32, device=dev)
        fwd.append(("dfd_pool", (_ptr(yh), bnh.scale, bnh.shift, _ptr(self.pooled), N, Hf * Wf, F, ACT_SWISH, dt,
                             None, POOL_CHUNKS)))
        self.drop_masks = OrderedDict()
        if self.drop_rate > 0.0:
            self.dropout_mask = torch.ones(N, F, dtype=torch.float32, device=dev)
            masks.append((self.dropout_mask, N * F, 1, 1.0 - self.drop_rate))
            fwd.append(("dfd_mul_f32_train", (_ptr(self.pooled), _ptr(self.dropout_mask), N * F)))
        for r_ in recs:
            if r_["dp_gate"] is not None:
                self.drop_masks[r_["b"].name] = r_["dp_gate"]
        if masks:
            import struct
            raw = b"".join(struct.pack("<Qqifii", _ptr(t), rows, width, keep, si, 0) for si, (t, rows, width, keep) in enumerate(masks))
            self._mask_table = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(dev)
            fwd.insert(0, ("dfd_rng_masks_train", (_ptr(self._mask_table), len(masks), _ptr(self.rng_state))))
            fwd.insert(1, ("dfd_rng_tick_train", (_ptr(self.rng_state),)))
            cmax = max(t.shape[-1] for t, _, _, _ in masks)
            self._unit_affine = torch.cat([torch.ones(cmax, device=dev), torch.zeros(cmax, device=dev)]).float()
            self._keep.append(self._unit_affine)
        K = spec.num_classes
        self.logits = torch.zeros(N, K, dtype=torch.float32, device=dev)
        self.dlogits = torch.zeros(N, K, dtype=torch.float32, device=dev)
        self.dpooled = torch.zeros(N, F, dtype=torch.float32, device=dev)
        self.target_i = torch.zeros(N, dtype=torch.int64, device=dev)
        self.target_f = torch.zeros(N, K, dtype=torch.float32, device=dev)
        self._head_in = x

        # ---- backward ----------------------------------------------------------------------------
        bwd.append(("dfd_head_bwd", (_ptr(self.dlogits), _ptr(self.pooled), P32("classifier.weight"),
                                     G32("classifier.weight"), G32("classifier.bias"), _ptr(self.dpooled), N, F, K)))
        if self.drop_rate > 0.0:
            bwd.append(("dfd_mul_f32", (_ptr(self.dpooled), _ptr(self.dropout_mask), N * F)))
        bwd.append(("dfd_act_bwd", (None, _ptr(yh), bnh.scale, bnh.shift, bnh.mean, bnh.rstd, None, _ptr(self.dpooled),
                                    mid_a, N, Hf * Wf, F, ACT_SWISH, dt, bnh.bs1, bnh.bs2, BF(bnh))))
        bwd.append(bwd_finalize(bnh, Mf))
        bwd.append(("dfd_bn_bwd_apply", (mid_a, _ptr(yh), None, bnh.cA, bnh.cB, bnh.cC, mid_b, N, Hf * Wf, F, dt)))
        cur = 0
        bwd.append(gemm(mid_b, T16("conv_head.weight"), sm[cur], Mf, spec.head_in, F))
        bwd.append(self._wgrad(mid_b, _ptr(self._head_in), G32("conv_head.weight"), Mf, F, spec.head_in))
        self._flush_reduce(bwd)
        for rec in reversed(recs):
            b, h, w, ho, wo, xin = rec["b"], rec["h"], rec["w"], rec["ho"], rec["wo"], rec["x"]
            p = b.name
            M1, M2 = N * h * w, N * ho * wo
            bn_out, bn_mid, dw_bn, pw_name = rec["bn_out"], rec["bn_mid"], rec["dw_bn"], rec["pw_name"]
            y2, a2, y3 = rec["y2"], rec["a2"], rec["y3"]
            dout = sm[cur]
            t1, t2 = sm[(cur + 1) % 3], sm[(cur + 2) % 3]
            gbn = dout
            if rec["dp_gate"] is not None:
                # drop path: the gradient reaching bn3 is dout * mask / keep (the identity branch keeps dout itself); one extra
                # pass through the gated streaming kernel with a unit affine, only in this regularised configuration
                cm = self._unit_affine.numel() // 2
                bwd.append(("dfd_bn_act", (dout, _ptr(self._unit_affine), _ptr(self._unit_affine, cm), _ptr(rec["dp_gate"]), None, t2,
                                           N, ho * wo, b.cout, ACT_NONE, 0, dt)))
                gbn = t2
            bwd.append(("dfd_bn_bwd_reduce", (gbn, _ptr(y3), None, bn_out.mean, bn_out.rstd, N, ho * wo, b.cout, dt,
                                              bn_out.bs1, bn_out.bs2, BF(bn_out))))
            bwd.append(bwd_finalize(bn_out, M2))
            bwd.append(("dfd_bn_bwd_apply", (gbn, _ptr(y3), None, bn_out.cA, bn_out.cB, bn_out.cC, t1, N, ho * wo, b.cout, dt)))
            bwd.append(gemm(t1, T16(p + pw_name + ".weight"), mid_a, M2, b.cmid, b.cout))
            bwd.append(self._wgrad(t1, _ptr(a2), G32(p + pw_name + ".weight"), M2, b.cout, b.cmid))
            gate_ptr = dpool_ptr = None
            if b.cse:
                gate_ptr, dpool_ptr = _ptr(rec["gate"]), se_dpool
                if os.environ.get("DFD_SE_FUSED"):
                    bwd.append(("dfd_se_bwd_chain", (mid_a, _ptr(y2), bn_mid.scale, bn_mid.shift, se_draw, _ptr(rec["pooled"]),
                                                     P32(p + ".se.conv_reduce.weight"), P32(p + ".se.conv_reduce.bias"),
                                                     P32(p + ".se.conv_expand.weight"), P32(p + ".se.conv_expand.bias"),
                                                     se_de, se_r, se_drp, se_dpool, N, ho * wo, b.cmid, b.cse, dt)))
                    bwd.append(("dfd_se_fc_wgrad", (se_de, se_r, se_drp, _ptr(rec["pooled"]),
                                                    G32(p + ".se.conv_reduce.weight"), G32(p + ".se.conv_reduce.bias"),
                                                    G32(p + ".se.conv_expand.weight"), G32(p + ".se.conv_expand.bias"),
                                                    N, b.cmid, b.cse)))
                else:
                    bwd.append(("dfd_se_bwd_reduce", (mid_a, _ptr(y2), bn_mid.scale, bn_mid.shift, se_draw, N, ho * wo, b.cmid, dt)))
                    bwd.append(("dfd_se_fc_bwd", (se_draw, _ptr(rec["pooled"]), P32(p + ".se.conv_reduce.weight"),
                                                  P32(p + ".se.conv_reduce.bias"), P32(p + ".se.conv_expand.weight"),
                                                  P32(p + ".se.conv_expand.bias"), se_de, se_r, se_drp, se_dpool,
                                                  G32(p + ".se.conv_reduce.weight"), G32(p + ".se.conv_reduce.bias"),
                                                  G32(p + ".se.conv_expand.weight"), G32(p + ".se.conv_expand.bias"),
                                                  N, b.cmid, b.cse)))
            bwd.append(("dfd_act_bwd", (mid_a, _ptr(y2), bn_mid.scale, bn_mid.shift, bn_mid.mean, bn_mid.rstd, gate_ptr,
                                        dpool_ptr, mid_b, N, ho * wo, b.cmid, ACT_SWISH, dt, bn_mid.bs1, bn_mid.bs2, BF(bn_mid))))
            bwd.append(bwd_finalize(bn_mid, M2))
            if b.kind == "ir":
                y1 = rec["y1"]
                if os.environ.get("DFD_DW_SPLIT_BWD"):      # diagnostics: the two-pass form (same results)
                    bwd.append(("dfd_dwconv_dgrad", (mid_b, _ptr(y2), bn_mid.cA, bn_mid.cB, bn_mid.cC, P32(p + ".conv_dw.weight"),
                                                     _ptr(y1), dw_bn.scale, dw_bn.shift, dw_bn.mean, dw_bn.rstd, None, mid_a,
                                                     N, h, w, b.cmid, b.k, b.stride, 1, dt, dw_bn.bs1, dw_bn.bs2)))
                    bwd.append(("dfd_dwconv_wgrad", (_ptr(y1), dw_bn.scale, dw_bn.shift, mid_b, _ptr(y2), bn_mid.cA, bn_mid.cB,
                                                     bn_mid.cC, G32(p + ".conv_dw.weight"), N, h, w, b.cmid, b.k, b.stride, dt)))
                else:
                    # input gradient (through bn1 + Swish) and weight gradient in one pass over the dy tile
                    bwd.append(self._dw_bwd((mid_b, _ptr(y2), bn_mid.cA, bn_mid.cB, bn_mid.cC, P32(p + ".conv_dw.weight"),
                                             _ptr(y1), dw_bn.scale, dw_bn.shift, dw_bn.mean, dw_bn.rstd, None, mid_a,
                                             G32(p + ".conv_dw.weight"), N, h, w, b.cmid, b.k, b.stride, dt,
                                             dw_bn.bs1, dw_bn.bs2), N, h, w, b.cmid, b.k, b.stride, BF(dw_bn)))
                bwd.append(bwd_finalize(dw_bn, M1))
                bwd.append(("dfd_bn_bwd_apply", (mid_a, _ptr(y1), None, dw_bn.cA, dw_bn.cB, dw_bn.cC, mid_b, N, h * w, b.cmid, dt)))
                bwd.append(gemm(mid_b, T16(p + ".conv_pw.weight"), t2, M1, b.cin, b.cmid))
                if b.has_residual:
                    bwd.append(("dfd_add_inplace", (t2, dout, M1 * b.cin, dt)))
                bwd.append(self._wgrad(mid_b, _ptr(xin), G32(p + ".conv_pw.weight"), M1, b.cmid, b.cin))
            elif os.environ.get("DFD_DW_SPLIT_BWD"):
                bwd.append(("dfd_dwconv_dgrad", (mid_b, _ptr(y2), bn_mid.cA, bn_mid.cB, bn_mid.cC, P32(p + ".conv_dw.weight"),
                                                 None, None, None, None, None, dout if b.has_residual else None, t2,
                                                 N, h, w, b.cmid, b.k, b.stride, 0, dt, None, None)))
                bwd.append(("dfd_dwconv_wgrad", (_ptr(xin), None, None, mid_b, _ptr(y2), bn_mid.cA, bn_mid.cB, bn_mid.cC,
                                                 G32(p + ".conv_dw.weight"), N, h, w, b.cmid, b.k, b.stride, dt)))
            else:
                # DS block: the depthwise conv reads the block input as is (mode 0 of the fused pass)
                bwd.append(self._dw_bwd((mid_b, _ptr(y2), bn_mid.cA, bn_mid.cB, bn_mid.cC, P32(p + ".conv_dw.weight"),
                                         _ptr(xin), None, None, None, None, dout if b.has_residual else None, t2,
                                         G32(p + ".conv_dw.weight"), N, h, w, b.cmid, b.k, b.stride, dt, None, None),
                                        N, h, w, b.cmid, b.k, b.stride))
            self._flush_reduce(bwd)
            cur = (cur + 2) % 3
        # stem
        bn = self.bns["bn1"]
        bwd.append(("dfd_act_bwd", (sm[cur], _ptr(y0), bn.scale, bn.shift, bn.mean, bn.rstd, None, None, mid_a, N, Hs * Ws,
                                    spec.stem, ACT_SWISH, dt, bn.bs1, bn.bs2, BF(bn))))
        bwd.append(bwd_finalize(bn, N * Hs * Ws))
        if self.stem_impl == "gemm":
            bwd.append(("dfd_bn_bwd_apply", (mid_a, _ptr(y0), None, bn.cA, bn.cB, bn.cC, mid_b, N, Hs * Ws, spec.stem, dt)))
            bwd.append(("dfd_memset_async", (_ptr(self.stem_gpad), 0, spec.stem * Kp * 4)))
            bwd.append(self._wgrad(mid_b, _ptr(self.stem_cols), _ptr(self.stem_gpad), N * Hs * Ws, spec.stem, Kp))
            self._flush_reduce(bwd)          # the padded gradient must be complete before it is un-padded into the arena
            bwd.append(("dfd_unpad_grad", (_ptr(self.stem_gpad), G32("conv_stem.weight"), spec.stem, taps, Kp)))
        else:
            bwd.append(("dfd_stem_wgrad", (_ptr(self.x_in), mid_a, _ptr(y0), bn.cA, bn.cB, bn.cC, G32("conv_stem.weight"), N,
                                           spec.in_chans, self.H, self.W, spec.stem, 3, 2, 1, dt)))
        bwd = self._patch_workspace([op for op in bwd if op is not None])
        self._upload_fin_descs()

        def base_name(n):
            for suf in ("_train", "_evalonly", "_sync"):
                if n.endswith(suf):
                    return n[:-len(suf)]
            return n

        for n, a in fwd + bwd:      # arity / type check of the plan against the ABI table
            if n.startswith("ALLREDUCE"):
                continue
            codes = _lib.SIGNATURES[base_name(n)]
            if len(a) != len(codes) - 1:
                raise AssertionError("%s: %d args for signature %r" % (n, len(a), codes))
            for v, c in zip(a, codes):
                if isinstance(v, tuple) and v[0] == "TRAIN_ONLY":
                    v = v[1]
                ok = (v is None or isinstance(v, int)) if c == "p" else (
                    isinstance(v, int) if c in "il" else (isinstance(v, (int, float)) or v == "TRAINING"))
                if not (ok or v == "TRAINING"):
                    raise AssertionError("%s: argument %r does not fit code %r" % (n, v, c))
        # `<name>_train` ops run in training mode only (mask generation, dropout); ("TRAIN_ONLY", ptr) operands are NULL in eval
        fwd = [(n, a) for n, a in fwd]
        self.fwd_ops = [(None if n.startswith("ALLREDUCE") else getattr(L, base_name(n)), n, a) for n, a in fwd]
        self.bwd_ops = [(None if n.startswith("ALLREDUCE") else getattr(L, n), n, tuple(a)) for n, a in bwd]
        self.n_launch["fwd"] = len(fwd)
        self.n_launch["bwd"] = len(bwd)

    # ------------------------------------------------------------------------------------------
    # execution
    # ------------------------------------------------------------------------------------------
    def _run(self, ops, stream, training=None, skip_finalize=False):
        if self._plan_only:
            raise _lib.NativeError("plan-only engine cannot execute (no CUDA device)")
        L = self.L
        for fn, name, args in ops:
            if name.startswith("ALLREDUCE"):
                if training:
                    import torch.distributed as dist
                    dist.all_reduce(args[0], op=dist.ReduceOp.SUM if args[1] == "sum" else dist.ReduceOp.AVG)
                continue
            if name == "dfd_bn_finalize_sync":
                args = list(args)
                if training:
                    args[2] = args[2] * self.sync_world          # global element count behind the summed statistics
                name = "dfd_bn_finalize"
            if name.startswith("dfd_bn_finalize"):
                # `_evalonly`: in training the producing kernel's last CTA finalised this BatchNorm already
                if skip_finalize or (training and name.endswith("_evalonly")):
                    continue
                args = tuple((1 if training else 0) if a == "TRAINING" else a for a in args)
                if not training:
                    args = (None, None) + args[2:]
            elif name.endswith("_train"):
                if not training:
                    continue
            elif name == "dfd_bn_act" and any(isinstance(a, tuple) for a in args):
                args = tuple((a[1] if training else None) if isinstance(a, tuple) else a for a in args)
            elif not training and name in ("dfd_gemm_tn", "dfd_gemm_tn_rowpack", "dfd_dwconv_fwd"):
                args = tuple(args[:-3]) + (None, None, None)      # eval: no batch statistics, no finalisation
            elif not training and name in ("dfd_gemm_tn_mma", "dfd_stem_fwd"):
                args = tuple(args[:-2]) + (None, None)
            rc = fn(*args, stream)
            _lib.N_CALLS[0] += 1
            if rc != 0:
                raise _lib.NativeError("%s failed (%d): %s" % (name, rc, L.last_error()))

    def set_input(self, x):
        """x: [N, C, H, W] (NCHW, any float dtype / device)."""
        if tuple(x.shape) != tuple(self.x_in.shape):
            raise ValueError("input shape %s != engine shape %s" % (tuple(x.shape), tuple(self.x_in.shape)))
        self.x_in.copy_(x, non_blocking=True)

    def set_target(self, target):
        if target.dtype.is_floating_point:
            self.target_f.copy_(target, non_blocking=True)
            self._soft = True
        else:
            self.target_i.copy_(target, non_blocking=True)
            self._soft = False

    def zero_step_scratch(self, stream, grads=True):
        _lib.call("dfd_memset_async", _ptr(self.stats), 0, self.stats.numel() * 8, stream)
        _lib.call("dfd_memset_async", _ptr(self.scalars), 0, self.scalars.numel() * 4, stream)
        if grads:
            _lib.call("dfd_memset_async", _ptr(self.grads32), 0, self.grads32.numel() * 4, stream)

    def forward(self, training=True, stream=None):
        """Runs the network on self.x_in; logits land in self.logits ([N, num_classes] fp32)."""
        st = stream if stream is not None else torch.cuda.current_stream().cuda_stream
        ar = self.arena
        if training:
            ar.state_version += 1            # running statistics move
            self._run(self.fwd_ops, st, True)
        else:
            # inference: BN is an affine map with constants (running statistics). Its per-channel scale / shift - the
            # "folded" form every consumer kernel applies on load - is computed ONCE per weight state and kept, so a
            # steady-state eval forward launches no BN kernel at all (test_img, validate; dfd/runners/test.py:29-60)
            frozen = self._eval_version == ar.state_version
            self._run(self.fwd_ops, st, False, skip_finalize=frozen)
            self._eval_version = ar.state_version
        return self.logits

    def head(self, with_loss, smoothing=0.0, loss_scale=1.0, soft=False, stream=None, loss_scale_dev=None):
        """classifier (+ fused softmax cross-entropy, top-1 count and dL/dlogits when with_loss; needs num_classes >= 2)."""
        st = stream if stream is not None else torch.cuda.current_stream().cuda_stream
        spec = self.spec
        pw = _ptr(self.params32, self.p_off[self.cls_name + ".weight"][0])
        pb = _ptr(self.params32, self.p_off[self.cls_name + ".bias"][0])
        if with_loss:
            _lib.call("dfd_head_fwd", _ptr(self.pooled), pw, pb, _ptr(self.logits), self.N, spec.num_features,
                      spec.num_classes, None if soft else _ptr(self.target_i), _ptr(self.target_f) if soft else None,
                      float(smoothing), float(loss_scale), loss_scale_dev, _ptr(self.scalars), _ptr(self.scalars, 1),
                      _ptr(self.dlogits), st)
        else:
            _lib.call("dfd_head_fwd", _ptr(self.pooled), pw, pb, _ptr(self.logits), self.N, spec.num_features,
                      spec.num_classes, None, None, 0.0, 1.0, None, None, None, None, st)

    def backward(self, stream=None):
        """Back-propagates self.dlogits; gradients are ACCUMULATED into self.grads32 (zero it per step)."""
        st = stream if stream is not None else torch.cuda.current_stream().cuda_stream
        self._run(self.bwd_ops, st, True)

    @property
    def loss(self):
        return self.scalars[0]

    @property
    def correct(self):
        return self.scalars[1]
