"""Drop-in model objects for the runner: `create_model` / `create_deepfake_model_v4` return an `nn.Module` whose
forward / backward run on the native engine.

Boundary being mirrored (SURVEY.md section 8b):
  * `create_model(model_name, pretrained=False, num_classes=1000, in_chans=3, checkpoint_path='', **kwargs)`
        dfd/timm/models/factory.py:8-64
  * `create_deepfake_model_v4(model_name, ..., num_classes, in_chans, checkpoint_path, strict)`  factory.py:190-252
  * the model object protocol the runner relies on: `model(input) -> logits [N, num_classes]` (train.py:621,719),
    `.train()/.eval()`, `.named_parameters()` (optim_factory.py:14), `.state_dict()/.load_state_dict()` with the
    reference key names / OIHW fp32 tensors (utils.py:32-33,101; helpers.py:44,57), `.default_cfg`, `.cuda()`.

The kernels need static shapes, so the engine (kernel plan + activation arenas) is built lazily for each
(batch, H, W) that reaches `forward`; all plans share one set of weights, gradients and running statistics.
"""
from collections import OrderedDict

import torch
import torch.nn as nn

from . import _lib
from .arch import SUPPORTED_ARCHS, get_spec, state_entries
from .engine import Engine, check_num_classes

_DEFAULT_CFG = dict(num_classes=1000, pool_size=(7, 7), crop_pct=0.875, interpolation="bicubic",
                    mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225))


class _NativeForward(torch.autograd.Function):
    """logits = net(input) on the engine; backward hands dL/dlogits to the engine's backward plan, which accumulates
    into the flat gradient arena that the parameters' `.grad` tensors alias."""

    @staticmethod
    def forward(ctx, anchor, model, engine, training):
        ctx.engine = engine
        ctx.model = model
        st = torch.cuda.current_stream().cuda_stream
        engine.zero_step_scratch(st, grads=False)
        engine.forward(training=training, stream=st)
        engine.head(False, stream=st)
        return engine.logits.clone()

    @staticmethod
    def backward(ctx, dlogits):
        e = ctx.engine
        e.dlogits.copy_(dlogits)
        red = ctx.model._reducer
        if red is not None:
            # data-parallel run: the backward of the plan that ran this forward, with the bucketed gradient mean
            # overlapped on the reducer's side stream (what the reference's DDP wrapper does in its backward hooks)
            red.backward_and_reduce(e)
        else:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1 and not ctx.model.allow_local_grads:
                raise _lib.NativeError("NativeModel.backward in a %d-rank job without a gradient reducer: wrap the model in "
                                       "deepfake_detection_b200.ddp.NativeDDP (train.py:402-406) so that replicas do not "
                                       "diverge silently" % dist.get_world_size())
            e.backward()
        return None, None, None, None


def init_state_dict(spec, seed=None):
    """Random-init state in the reference's key order with the reference's initialisers:
    EfficientNet: efficientnet_builder.py:537-575 (`_init_weight_goog`: conv N(0, 2/fan_out), depthwise fan_out / groups,
    Linear U(+-1/sqrt(fan_out)), BN 1 / 0);
    ResNet: resnet.py:410-420 (conv kaiming_normal fan_out, BN 1 / 0, the LAST BN gamma of every residual block ZERO -
    `zero_init_last_bn=True` is the constructor default, :353 - and nn.Linear's default U(+-1/sqrt(fan_in)) for fc)."""
    import math
    g = torch.Generator(device="cpu").manual_seed((torch.initial_seed() if seed is None else seed) % (2 ** 31))
    sd = OrderedDict()
    resnet = spec.family == "resnet"
    last_bn = set()
    if resnet:
        for b in spec.blocks:
            last_bn.add(b.name + (".bn2.weight" if b.kind == "basic" else ".bn3.weight"))       # resnet.py:147-148,212-213
    for name, shape, role in state_entries(spec):
        if resnet and role in ("fc_w", "fc_b"):
            r = 1.0 / math.sqrt(spec.num_features)
            sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * r
            continue
        if name in last_bn:
            sd[name] = torch.zeros(shape)
            continue
        if role in ("conv_w", "dw_w", "se_w"):
            fan_out = shape[0] * shape[2] * shape[3]
            if role == "dw_w":
                fan_out = shape[2] * shape[3]           # fan_out //= groups
            sd[name] = torch.randn(shape, generator=g) * math.sqrt(2.0 / fan_out)
        elif role == "bn_w":
            sd[name] = torch.ones(shape)
        elif role in ("bn_b", "se_b", "fc_b", "bn_rm"):
            sd[name] = torch.zeros(shape)
        elif role == "bn_rv":
            sd[name] = torch.ones(shape)
        elif role == "bn_nbt":
            sd[name] = torch.zeros((), dtype=torch.int64)
        elif role == "fc_w":
            r = 1.0 / math.sqrt(shape[0])               # fan_out of the Linear, _init_weight_goog
            sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * r
    return sd


class NativeModel(nn.Module):
    def __init__(self, arch, num_classes=2, in_chans=3, dtype="bf16", bn_momentum=None, bn_eps=None, bn_tf=False,
                 drop_rate=0.0, drop_path_rate=0.0, gemm_impl="tc", **unused):
        super().__init__()
        if bn_tf:       # efficientnet_blocks.py:13-30
            bn_momentum = 1 - 0.99 if bn_momentum is None else bn_momentum
            bn_eps = 1e-3 if bn_eps is None else bn_eps
        check_num_classes(num_classes)
        self.arch = arch
        self.num_classes = num_classes
        self.in_chans = in_chans
        self.dtype_name = dtype
        self.bn_momentum = 0.1 if bn_momentum is None else bn_momentum
        self.bn_eps = 1e-5 if bn_eps is None else bn_eps
        self.gemm_impl = gemm_impl
        self.drop_rate = float(drop_rate)              # efficientnet.py:346-347 (classifier dropout)
        self.drop_path_rate = float(drop_path_rate)    # efficientnet_builder.py:322-323 (linear ramp over the blocks)
        self.max_plans = 4                             # execution plans kept alive (LRU); each owns an activation arena
        self.allow_local_grads = False
        self.sync_bn = False                           # set by ddp.convert_syncbn_model (train.py:388-394)
        self._reducer = None
        self.spec = get_spec(arch, num_classes=num_classes, in_chans=in_chans)
        if self.spec.family != "efficientnet" and (self.drop_rate or self.drop_path_rate):
            raise _lib.NativeError("drop_rate / drop_path_rate are implemented for the EfficientNet family only")
        self.default_cfg = dict(_DEFAULT_CFG, input_size=self.spec.input_size,
                                first_conv="conv_stem" if self.spec.family == "efficientnet" else "conv1",
                                classifier="classifier" if self.spec.family == "efficientnet" else "fc")
        self._engines = OrderedDict()
        self._primary = None
        self._pending_state = None
        self._anchor = nn.Parameter(torch.zeros(()), requires_grad=True)   # gives the output a grad_fn
        self._named = None

    # ---- engines ------------------------------------------------------------------------------------
    def _engine_kwargs(self):
        return dict(num_classes=self.num_classes, in_chans=self.in_chans, dtype=self.dtype_name, bn_momentum=self.bn_momentum,
                    bn_eps=self.bn_eps, gemm_impl=self.gemm_impl, drop_rate=self.drop_rate, drop_path_rate=self.drop_path_rate,
                    sync_bn=self.sync_bn)

    @property
    def engine(self):
        """the ARENA engine: owner of the weights, gradients, running statistics and derived weight layouts. It holds no
        activation buffers and no kernel plan (those are built per input shape by `engine_for`), so touching it - which
        `create_optimizer`, `named_parameters` and `state_dict` do - costs parameter memory only."""
        if self._primary is None:
            self._primary = Engine(self.arch, 1, params_only=True, **self._engine_kwargs())
            if self._pending_state is not None:
                self._primary.load_state_dict(self._pending_state, strict=False)
                self._pending_state = None
            else:
                self._init_weights(self._primary)
        return self._primary

    def engine_for(self, n, h, w):
        """the execution plan for a (batch, H, W) input: built on first use, at most `max_plans` kept (least recently used
        evicted together with every CUDA graph / trainer view captured over it)"""
        key = (int(n), int(h), int(w))
        e = self._engines.get(key)
        if e is None:
            arena = self.engine
            while len(self._engines) >= self.max_plans:
                old_key, old = self._engines.popitem(last=False)
                for tk in [k for k in self.__dict__.get("_trainers", {}) if k[0] == id(old)]:
                    del self.__dict__["_trainers"][tk]
                if self._reducer is not None:
                    self._reducer._plans.pop(id(old), None)
            e = Engine(self.arch, key[0], key[1], key[2], share_from=arena, **self._engine_kwargs())
            self._engines[key] = e
        else:
            self._engines.move_to_end(key)
        return e

    def _init_weights(self, e):
        e.load_state_dict(init_state_dict(self.spec))

    # ---- nn.Module protocol ---------------------------------------------------------------------------
    def forward(self, x):
        if x.dim() != 4:
            raise ValueError("expected NCHW input")
        if self.__dict__.get("_weights_dirty", False):
            self.engine.sync_weights()          # fp32 master changed out of band (ModelEma.update): refresh the 16-bit copies
            self._weights_dirty = False
        e = self.engine_for(x.shape[0], x.shape[2], x.shape[3])
        e.set_input(x)
        if torch.is_grad_enabled() and self.training:
            return _NativeForward.apply(self._anchor, self, e, True)
        st = torch.cuda.current_stream().cuda_stream
        e.zero_step_scratch(st, grads=False)
        e.forward(training=self.training, stream=st)
        e.head(False, stream=st)
        return e.logits.clone()

    def named_parameters(self, prefix="", recurse=True, remove_duplicate=True):
        if self._named is None:
            e = self.engine
            self._named = []
            for n in e.param_names:
                p = nn.Parameter(e.param_view(n), requires_grad=True)
                p.grad = e.grad_view(n)
                self._named.append((n, p))
        for n, p in self._named:
            yield (prefix + ("." if prefix else "") + n, p)

    def parameters(self, recurse=True):
        for _, p in self.named_parameters():
            yield p

    def state_dict(self, *args, **kwargs):
        return self.engine.state_dict()

    def load_state_dict(self, state_dict, strict=True):
        if self._primary is None and not torch.cuda.is_available():
            self._pending_state = state_dict
            return
        missing = self.engine.load_state_dict(state_dict, strict=strict)
        return missing

    def cuda(self, device=None):
        """train.py:346 `model.cuda()`: the arenas are created on the current CUDA device; a different index is refused"""
        if device is not None and self._primary is not None:
            idx = torch.device("cuda", device).index if isinstance(device, int) else torch.device(device).index
            if idx is not None and idx != self._primary.device.index:
                raise _lib.NativeError("NativeModel lives on %s; cannot move it to cuda:%d" % (self._primary.device, idx))
        return self

    def half(self):
        """test.py:47 `model.half()`: switches the compute dtype to fp16 (only before the first plan exists)"""
        if self.dtype_name not in ("fp16", "float16", "half", torch.float16):
            if self._primary is not None:
                raise _lib.NativeError("NativeModel.half(): the model was already materialised in %r; pass dtype='fp16' to the "
                                       "factory instead" % (self.dtype_name,))
            self.dtype_name = "fp16"
        return self

    def get_classifier(self):
        """efficientnet.py:307-308 / resnet.py:426-427: the classifier as an nn.Linear whose tensors alias the arenas"""
        e = self.engine
        fc = nn.Linear(self.spec.num_features, self.num_classes)
        fc.weight = nn.Parameter(e.param_view(e.cls_name + ".weight"))
        fc.bias = nn.Parameter(e.param_view(e.cls_name + ".bias"))
        return fc

    def __deepcopy__(self, memo):
        """ModelEma deep-copies the model (utils.py:300): the copy owns fresh arenas holding the same state"""
        kw = dict(num_classes=self.num_classes, in_chans=self.in_chans, dtype=self.dtype_name, bn_momentum=self.bn_momentum,
                  bn_eps=self.bn_eps, drop_rate=self.drop_rate, drop_path_rate=self.drop_path_rate, gemm_impl=self.gemm_impl)
        m = NativeModel(self.arch, **kw)
        m.training = self.training
        if self._primary is not None:
            m.load_state_dict(self.state_dict())
        elif self._pending_state is not None:
            m._pending_state = self._pending_state
        return m


def create_model(model_name, pretrained=False, num_classes=1000, in_chans=3, checkpoint_path="", **kwargs):
    """dfd/timm/models/factory.py:8-64 for the architectures on the native hot path."""
    if pretrained:
        raise _lib.NativeError("pretrained weights need network access; load a checkpoint instead")
    if model_name not in SUPPORTED_ARCHS:
        raise RuntimeError("Unknown model (%s)" % model_name)       # factory.py:56
    kwargs.pop("global_pool", None)
    model = NativeModel(model_name, num_classes=num_classes, in_chans=in_chans, **kwargs)
    if checkpoint_path:
        from .helpers import load_checkpoint
        load_checkpoint(model, checkpoint_path)
    return model


def create_deepfake_model_v4(model_name, pretrained=False, num_classes=1000, in_chans=3, checkpoint_path="",
                             strict=True, **kwargs):
    """dfd/timm/models/factory.py:190-252 (asserts the model name, :213)."""
    assert model_name in ["efficientnet_deepfake_v4"]
    kwargs.pop("global_pool", None)
    model = NativeModel(model_name, num_classes=num_classes, in_chans=in_chans, **kwargs)
    if checkpoint_path:
        from .helpers import load_checkpoint
        load_checkpoint(model, checkpoint_path, strict=strict)
    return model
