"""`train_epoch` / `validate` with the reference's signatures and return values (dfd/runners/train.py:594-766),
driving the native engine.

What is kept: the argument lists, the `args` fields read inside the step (`prefetcher, mixup, mixup_off_epoch,
num_classes, smoothing, distributed, world_size, local_rank, log_interval, recovery_interval, tta`), the metric
definitions (`loss` = mean of per-batch (all-reduced) losses weighted by batch size, `prec1` = top-1 %), the lr read
from `optimizer.param_groups` for logging, recovery checkpoints, `lr_scheduler.step_update`.

What is NOT kept, on purpose: the per-step `torch.cuda.synchronize()` + two `.item()` host reads
(train.py:639-645).  The loss / correct-count of every step stay on the device; they are read back (one small copy)
only at `log_interval` boundaries and at the end of the epoch, which is what lets the CPU run ahead of the GPU.
The reported numbers are identical.

Two step flavours:
  * fused   : model is a NativeModel, loss_fn one of deepfake_detection_b200.loss.* and optimizer an ArenaOptimizer
              -> one Trainer step (forward, cross-entropy head, backward, [all-reduce], update), CUDA-graph replayed;
  * protocol: anything else that follows the reference's object protocol (model(input), loss_fn(out, target),
              loss.backward(), optimizer.step()) — the NativeModel autograd bridge makes this work unchanged.
"""
import logging
import time
from collections import OrderedDict

import torch


class AverageMeter:
    """dfd/timm/utils.py:152-167"""

    def __init__(self):
        self.reset()

    def reset(self):
        self.val = self.avg = self.sum = self.count = 0

    def update(self, val, n=1):
        self.val = val
        self.sum += val * n
        self.count += n
        self.avg = self.sum / self.count


def accuracy(output, target, topk=(1,)):
    """dfd/timm/utils.py:170-186 (top-1 only is used on the hot path; soft targets compare against their argmax)"""
    if target.shape == output.shape:
        target = target.argmax(dim=1)
    pred = output.argmax(dim=1)
    return (pred == target).float().sum() * 100.0 / target.size(0)


def _fused_ok(model, optimizer, loss_fn):
    from ..models import NativeModel
    from ..optim import ArenaOptimizer
    m = model.module if hasattr(model, "module") else model
    return isinstance(m, NativeModel) and isinstance(optimizer, ArenaOptimizer) and hasattr(loss_fn, "native_smoothing")


def train_epoch(epoch, model, loader, optimizer, loss_fn, args, lr_scheduler=None, saver=None, output_dir="",
                use_amp=False, model_ema=None):
    if args.prefetcher and args.mixup > 0 and getattr(loader, "mixup_enabled", False):
        if args.mixup_off_epoch and epoch >= args.mixup_off_epoch:
            loader.mixup_enabled = False
    batch_time_m, data_time_m, losses_m, prec1_m = AverageMeter(), AverageMeter(), AverageMeter(), AverageMeter()
    model.train()
    m = model.module if hasattr(model, "module") else model
    fused = _fused_ok(model, optimizer, loss_fn)
    world = args.world_size if args.distributed else 1
    pending = []            # (device tensor [loss, correct], batch size): read back lazily
    end = time.time()
    last_idx = len(loader) - 1
    num_updates = epoch * len(loader)
    lr = None

    def drain():
        for stats, n in pending:
            vals = stats.tolist()
            if vals[0] == vals[0]:                 # train.py:642-643: a NaN loss is not averaged in
                losses_m.update(vals[0], n)
            prec1_m.update(vals[1], n)
        del pending[:]

    for batch_idx, (input, target) in enumerate(loader):
        last_batch = batch_idx == last_idx
        data_time_m.update(time.time() - end)
        if not args.prefetcher:
            input, target = input.cuda(non_blocking=True), target.cuda(non_blocking=True)
            if args.mixup > 0.:                                                    # train.py:615-619
                input, target = mixup_batch(input, target, alpha=args.mixup, num_classes=args.num_classes,
                                            smoothing=args.smoothing,
                                            disable=bool(args.mixup_off_epoch and epoch >= args.mixup_off_epoch))
        n = input.size(0)
        if fused:
            e = m.engine_for(n, input.shape[2], input.shape[3])
            tr = _trainer_for(m, e, optimizer, loss_fn)
            loss_t, correct_t = tr.train_step(input, target)
            stats = torch.stack([loss_t, correct_t * (100.0 / n)])
        else:
            output = model(input)
            loss = loss_fn(output, target)
            prec1 = accuracy(output.detach(), target)
            optimizer.zero_grad()
            loss.backward()
            optimizer.step()
            stats = torch.stack([loss.detach().float(), prec1])
        if args.distributed:
            from ..ddp import reduce_tensor
            stats = reduce_tensor(stats, world)          # loss and prec1 in ONE 2-float all-reduce (train.py:626-627)
        pending.append((stats, n))
        if model_ema is not None:
            model_ema.update(model)
        num_updates += 1
        batch_time_m.update(time.time() - end)
        if last_batch or batch_idx % args.log_interval == 0:
            drain()
            lrl = [g["lr"] for g in optimizer.param_groups]
            lr = sum(lrl) / len(lrl)
            if args.local_rank == 0:
                logging.info("Train:%d [%4d/%d] Loss:%.5f(%.5f) Prec@1:%7.4f(%7.4f) Time:%.3f(%.3f)s/batch LR:%.3e Data:%.3f(%.3f)s/batch",
                             epoch, batch_idx, len(loader), losses_m.val, losses_m.avg, prec1_m.val, prec1_m.avg,
                             batch_time_m.val, batch_time_m.avg, lr, data_time_m.val, data_time_m.avg)
        if saver is not None and args.recovery_interval and (last_batch or (batch_idx + 1) % args.recovery_interval == 0):
            saver.save_recovery(model, optimizer, args, epoch, model_ema=model_ema, use_amp=use_amp, batch_idx=batch_idx)
        if lr_scheduler is not None:
            # the metric the reference passes is the running loss average (train.py:695); it is only as fresh as the last
            # drain - none of the reference's per-update schedulers (cosine / step / tanh) reads it
            lr_scheduler.step_update(num_updates=num_updates, metric=losses_m.avg)
        end = time.time()
    drain()
    if hasattr(optimizer, "sync_lookahead"):
        optimizer.sync_lookahead()
    return OrderedDict([("loss", losses_m.avg), ("prec1", prec1_m.avg), ("learning_rate", lr)])


def mixup_batch(input, target, alpha=0.2, num_classes=1000, smoothing=0.1, disable=False):
    """dfd/timm/data/mixup.py:10-24: one lambda per batch, images mixed with the flipped batch, float [N, C] targets"""
    import numpy as np
    lam = 1.0
    if not disable:
        lam = float(np.random.beta(alpha, alpha))
    input = input.mul(lam).add_(input.flip(0), alpha=1.0 - lam)
    off = smoothing / num_classes
    on = 1.0 - smoothing + off
    y1 = torch.full((target.size(0), num_classes), off, device=target.device).scatter_(1, target.long().view(-1, 1), on)
    y2 = torch.full((target.size(0), num_classes), off, device=target.device).scatter_(1, target.flip(0).long().view(-1, 1), on)
    return input, lam * y1 + (1.0 - lam) * y2


def _trainer_for(model, engine, optimizer, loss_fn):
    """A Trainer view over an existing (model engine, optimizer) pair, cached on the model per engine."""
    from ..trainer import Trainer
    cache = model.__dict__.setdefault("_trainers", {})
    key = (id(engine), id(optimizer), float(loss_fn.native_smoothing), bool(loss_fn.native_soft))
    tr = cache.get(key)
    if tr is None:
        tr = Trainer.__new__(Trainer)
        tr.engine, tr.optimizer = engine, optimizer
        tr.smoothing = float(loss_fn.native_smoothing)
        tr.use_graph = True
        tr._graph = tr._graph_key = None
        tr.n_captures = 0
        tr.scale_window = 2000
        tr.dynamic_scale = model.dtype_name in ("fp16", "float16", "half", torch.float16)      # apex O1 semantics for half precision
        if tr.dynamic_scale and optimizer.gscale_dev is None:
            from ..engine import _ptr
            e0 = model.engine
            e0.loss_scale_state.copy_(torch.tensor([65536.0, 1.0 / 65536.0]))
            optimizer.gscale_dev = _ptr(e0.loss_scale_state, 1)
            optimizer.skip_flag = _ptr(e0.flags, 0)
        tr.reducer = getattr(model, "_reducer", None)
        cache[key] = tr
    return tr


def validate(model, loader, loss_fn, args, log_suffix=""):
    batch_time_m, losses_m, prec1_m = AverageMeter(), AverageMeter(), AverageMeter()
    model.eval()
    world = args.world_size if args.distributed else 1
    pending = []
    end = time.time()
    last_idx = len(loader) - 1
    with torch.no_grad():
        for batch_idx, (input, target) in enumerate(loader):
            if not args.prefetcher:
                input, target = input.cuda(non_blocking=True), target.cuda(non_blocking=True)
            output = model(input)
            if isinstance(output, (tuple, list)):
                output = output[0]
            rf = args.tta
            if rf > 1:                                                     # train.py:724-727
                output = output.unfold(0, rf, rf).mean(dim=2)
                target = target[0:target.size(0):rf]
            loss = loss_fn(output, target)
            prec1 = accuracy(output, target)
            stats = torch.stack([loss.float(), prec1])
            if args.distributed:
                from ..ddp import reduce_tensor
                stats = reduce_tensor(stats, world)
            pending.append((stats, input.size(0)))
            batch_time_m.update(time.time() - end)
            end = time.time()
            if args.local_rank == 0 and (batch_idx == last_idx or batch_idx % args.log_interval == 0):
                for s, n in pending:
                    v = s.tolist()
                    losses_m.update(v[0], n)
                    prec1_m.update(v[1], n)
                del pending[:]
                logging.info("Test%s:[%4d/%d] Loss:%.4f(%.4f) Prec@1:%.4f(%.4f) Time:%.3f(%.3f)s/batch", log_suffix, batch_idx,
                             last_idx, losses_m.val, losses_m.avg, prec1_m.val, prec1_m.avg, batch_time_m.val, batch_time_m.avg)
    for s, n in pending:
        v = s.tolist()
        losses_m.update(v[0], n)
        prec1_m.update(v[1], n)
    return OrderedDict([("loss", losses_m.avg), ("prec1", prec1_m.avg)])
