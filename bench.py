#!/usr/bin/env python
"""Benchmark of the data-parallel train step (BASELINE.json metric: images/sec, device-timed, max over ranks).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--arch efficientnet_b0] [--batch 256]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...        # the reference's arithmetic (oracle port) on the host cores
    python bench.py --impl library ...          # the same module graph under stock PyTorch eager (autocast, channels_last,
                                                # cuDNN / cuBLAS, torch DDP over NCCL): the bar SURVEY.md 8(d) names
    python bench.py --dump-outputs DIR ...      # also write what the last timed step computed as DIR/<name>.npy

One "step" = one full train iteration of the reference's hot loop (dfd/runners/train.py:621-637) on a synthetic
batch: forward, 2-class CE (sigmoid-BCE) loss + top-1, zero_grad, backward, [gradient all-reduce], SGD-nesterov
update, on per-GPU batch 256 x 3 x 224 x 224 (weak scaling).  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# algorithmic work per image per train step (SURVEY.md 8d / BASELINE.md section 3)
WORK = {
    "efficientnet_b0": dict(gflop=2.286, act_mb=68.00, bound="hbm", res=224),
    "efficientnet_b4": dict(gflop=26.258, act_mb=495.94, bound="hbm", res=380),
    "resnet50": dict(gflop=24.287, act_mb=108.44, bound="tensor", res=224),
    "resnet18": dict(gflop=10.645, act_mb=23.03, bound="tensor", res=224),
}


BASELINE_CFG = {("efficientnet_b0", 256, "bf16"): "BASELINE configs[1]/[2]", ("resnet50", 256, "bf16"): "BASELINE configs[3]",
                ("efficientnet_b4", 128, "fp16"): "BASELINE configs[4]"}


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], source="measured")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


DUMP_BYTES = 60 << 20      # all dumped arrays together, leaving room for the .npy headers under 64 MB


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Write each tensor as out_dir/<name>.npy (float64 stays float64, everything else becomes float32).

    The arrays are taken smallest first and each may use an equal share of what is left of `budget`.  One larger than its
    share is replaced by a sample of its flattened elements at positions drawn from a fixed seed, so the same array size
    always gives the same positions and two builds can be compared element for element."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    left = budget
    for i, (name, t) in enumerate(items):
        t = t.detach().cpu()
        a = (t.double() if t.dtype == torch.float64 else t.float()).numpy()
        share = left // (len(items) - i)
        if a.nbytes > share:
            idx = np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes


class ClockSampler(threading.Thread):
    """nvidia-smi clock / throttle sampling DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([s.strip() for s in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        sm, mx, reasons = [], 0.0, set()
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx = max(mx, float(s[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx or None, reasons=sorted(reasons), samples=len(sm))


# ---------------------------------------------------------------------------------------------------
# algorithmic bytes of one launch of each kernel family (ideal: every operand once, 2 B / element)
# ---------------------------------------------------------------------------------------------------
def conv_out(h, k, s):
    return (h + 2 * ((k - 1) // 2) - k) // s + 1


def op_bytes(name, a):
    if name in ("dfd_gemm_tn", "dfd_gemm_tn_rowpack"):
        M, N, K = a[3], a[4], a[5]
        return 2 * (M * K + N * K + M * N)
    if name == "dfd_gemm_tn_mma":
        M, N, K = a[4], a[5], a[6]
        return 2 * (M * K + N * K + M * N)
    if name in ("dfd_gemm_wgrad_mma", "dfd_gemm_wgrad"):
        M, Nw, Kw = a[3], a[4], a[5]
        return 2 * M * (Nw + Kw) + 4 * Nw * Kw
    if name == "dfd_conv_dgrad_s2_tc":
        N, H, W, Cin, Cout = a[3:8]
        return 2 * (N * (H * W * Cin + conv_out(H, 3, 2) * conv_out(W, 3, 2) * Cout) + 9 * Cin * Cout)
    if name == "dfd_conv_tc":                              # input once, output once, weights once (no im2col matrix)
        N, H, W, Cin, Cout, k, S = a[3:10]
        return 2 * (N * (H * W * Cin + conv_out(H, k, S) * conv_out(W, k, S) * Cout) + k * k * Cin * Cout)
    if name == "dfd_conv_wgrad_tc":
        N, H, W, Cin, Cout, k, S = a[3:10]
        return 2 * N * (H * W * Cin + conv_out(H, k, S) * conv_out(W, k, S) * Cout) + 4 * k * k * Cin * Cout
    if name == "dfd_dwconv_fwd":
        N, H, W, C, k, s = a[5:11]
        return 2 * N * C * (H * W + ((H + s - 1) // s) * ((W + s - 1) // s))
    if name == "dfd_dwconv_dgrad":
        N, H, W, C, k, s, mode = a[13:20]
        o = ((H + s - 1) // s) * ((W + s - 1) // s)
        return 2 * N * C * ((2 * o if a[2] else o) + (2 if mode == 1 else 1) * H * W + (H * W if a[11] else 0))
    if name == "dfd_dwconv_bwd":
        # dy operand(s) once, pre-activation input once, input gradient once (the k*k weight gradient is negligible)
        N, H, W, C, k, s = a[14:20]
        o = ((H + s - 1) // s) * ((W + s - 1) // s)
        return 2 * N * C * ((2 * o if a[2] else o) + 2 * H * W + (H * W if a[11] else 0))
    if name == "dfd_dwconv_wgrad":
        N, H, W, C, k, s = a[9:15]
        o = ((H + s - 1) // s) * ((W + s - 1) // s)
        return 2 * N * C * (H * W + (2 * o if a[5] else o))
    if name in ("dfd_bn_act",):
        n, hw, C = a[6], a[7], a[8]
        return 2 * n * hw * C * (2 + (1 if a[4] else 0))
    if name in ("dfd_pool", "dfd_colstats"):
        idx = 4 if name == "dfd_pool" else 1
        n, hw, C = a[idx], a[idx + 1], a[idx + 2]
        return 2 * n * hw * C
    if name == "dfd_relu_bn_bwd_reduce":                  # g (+ g2), y, out read; masked gradient written
        n, hw, C = a[7], a[8], a[9]
        return 2 * n * hw * C * (5 if a[1] else 4)
    if name in ("dfd_bn_bwd_reduce", "dfd_se_bwd_reduce"):
        n, hw, C = a[5], a[6], a[7]
        return 2 * n * hw * C * 2
    if name == "dfd_bn_bwd_apply":
        n, hw, C = a[7], a[8], a[9]
        return 2 * n * hw * C * 3
    if name == "dfd_act_bwd":
        n, hw, C = a[9], a[10], a[11]
        return 2 * n * hw * C * (3 if a[0] else 2)
    if name == "dfd_add_inplace":
        return 2 * a[2] * 3
    if name == "dfd_stem_fwd":
        N, Cin, H, W, Cout = a[3:8]
        return 2 * N * (Cin * H * W + Cout * ((H + 1) // 2) * ((W + 1) // 2))
    if name == "dfd_stem_wgrad":
        N, Cin, H, W, Cout = a[7:12]
        return 2 * N * (Cin * H * W + 2 * Cout * ((H + 1) // 2) * ((W + 1) // 2))
    return 0


def op_flops(name, a):
    """algorithmic FLOPs of one launch of the tensor-core kernels (2 * M * N * K)"""
    if name in ("dfd_gemm_tn", "dfd_gemm_tn_rowpack"):
        return 2 * a[3] * a[4] * a[5]
    if name == "dfd_gemm_tn_mma":
        return 2 * a[4] * a[5] * a[6]
    if name in ("dfd_gemm_wgrad_mma", "dfd_gemm_wgrad"):
        return 2 * a[3] * a[4] * a[5]
    if name == "dfd_conv1x1_dgrad_add":
        N, H, W, Cin, Cout, S = a[3:9]
        return 2 * N * conv_out(H, 1, S) * conv_out(W, 1, S) * Cin * Cout
    if name == "dfd_conv_dgrad_s2_tc":                     # 9 taps x Cout per 4 input pixels
        N, H, W, Cin, Cout = a[3:8]
        return 2 * N * conv_out(H, 3, 2) * conv_out(W, 3, 2) * 9 * Cin * Cout
    if name in ("dfd_conv_tc", "dfd_conv_wgrad_tc"):       # implicit GEMM: M = N*Ho*Wo pixels, K = k*k*Cin, N = Cout
        N, H, W, Cin, Cout, k, S = a[3:10]
        return 2 * N * conv_out(H, k, S) * conv_out(W, k, S) * Cout * k * k * Cin
    return 0


def profile_plan(trainer, torch):
    """Per-launch CUDA-event timing of one eager step (each kernel bracketed on the launching stream)."""
    e = trainer.engine
    stream = torch.cuda.current_stream()
    st = stream.cuda_stream
    e.zero_step_scratch(st, grads=True)
    fam = {}
    per_op = []
    for ops, training in ((e.fwd_ops, True), (e.bwd_ops, True)):
        for op in ops:
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(stream)
            e._run([op], st, training)
            t1.record(stream)
            t1.synchronize()
            ms = t0.elapsed_time(t1)
            f = fam.setdefault(op[1], dict(ms=0.0, bytes=0, launches=0, flops=0))
            f["ms"] += ms
            nb = op_bytes(op[1], op[2])
            f["bytes"] += nb
            f["flops"] += op_flops(op[1], op[2])
            f["launches"] += 1
            per_op.append((op[1], [a for a in op[2] if isinstance(a, int) and 0 <= a < (1 << 31)], round(ms, 4),
                           round(nb / max(ms, 1e-9) / 1e6, 1)))
        if ops is e.fwd_ops:
            e.head(True, stream=st)
    out = os.environ.get("DFD_PROFILE_OUT")
    if out:
        with open(out, "w") as f:
            for name, dims, ms, gbs in per_op:
                f.write("%-22s ms=%8.4f GB/s=%8.1f dims=%s\n" % (name, ms, gbs, dims))
    return fam


def run_native(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from deepfake_detection_b200.trainer import Trainer
    from deepfake_detection_b200.arch import get_spec
    from deepfake_detection_b200.models import init_state_dict
    arch, B = args.arch, args.batch
    res = args.res or WORK[arch]["res"]
    # args.lr = batch * world * basic_lr (train.py:814). basic_lr = 1e-5: random labels + nesterov momentum 0.9 make the
    # synthetic problem unstable above lr ~ 0.1 (round 1 used 1e-4: loss_final 1.18 at N = 8, lr 0.2 - the optimisation
    # diverging, not the reduction: tests/ddp_worker.py holds the 2-rank weights to the oracle); throughput is unaffected
    lr = 0.00001 * B * world
    tr = Trainer(arch, B, res, res, dtype=args.dtype, opt=args.opt, lr=lr, momentum=0.9, weight_decay=1e-4,
                 use_graph=not args.no_graph, gemm_impl=args.gemm)
    spec = get_spec(arch)
    torch.manual_seed(42)
    tr.load_state_dict(init_state_dict(spec, seed=42))        # random init with the reference's initialisers
    if tr.reducer is not None:
        tr.reducer.broadcast_parameters()
    e = tr.engine
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    x = torch.randn(B, spec.in_chans, res, res, device="cuda", generator=g)
    y = torch.randint(0, 2, (B,), device="cuda", generator=g)
    e.set_input(x)
    e.set_target(y)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # C-ABI calls of ONE step, counted (not derived): an eager step with the call counter of the binding read before / after
    # (on every rank, before the timed region: the step contains the gradient collectives)
    from deepfake_detection_b200 import _lib as _L
    c0 = _L.N_CALLS[0]
    tr.optimizer.push_hyper()
    tr._launch_step(False)
    torch.cuda.synchronize()
    n_launch = _L.N_CALLS[0] - c0
    for _ in range(max(args.warmup, 3)):
        tr.step_resident()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        tr.step_resident()
    t1.record()
    barrier()
    ms = t0.elapsed_time(t1)
    loss_final = float(e.loss)
    clocks = sampler.stop() if sampler else None
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    if args.dump_outputs and rank == 0:
        # what a caller of the step receives after the last timed step: loss, correct count, logits, the reference-layout
        # state dict (updated weights, running statistics) and the gradients, flattened in parameter order
        sd = tr.state_dict()
        dump_outputs(args.dump_outputs, dict(
            loss=e.loss.reshape(1), correct=e.correct.reshape(1), logits=e.logits,
            state=torch.cat([v.reshape(-1).float() for v in sd.values()]),
            grads=torch.cat([e.grad_view(n).reshape(-1) for n in e.param_names])))

    # ---- end to end through the public API with HOST buffers (H2D of the batch + D2H of the loss every step) ----
    # the batch is what the reference's fast_collate hands its prefetcher: uint8 NCHW in pinned host memory
    # (loader.py:14-41); Trainer.train_step_host uploads it on a copy stream (double-buffered) and normalises it on the device
    xh = torch.empty(B, spec.in_chans, res, res, dtype=torch.uint8).pin_memory()
    xh.copy_((x * 58.0 + 120.0).clamp_(0, 255).to(torch.uint8))
    yh = torch.empty(B, dtype=torch.int64).pin_memory()
    yh.copy_(y)
    for _ in range(3):
        out = tr.train_step_host(xh, yh)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2e_steps = max(3, args.steps // 2)
    e0.record()
    for _ in range(e2e_steps):
        out = tr.train_step_host(xh, yh)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([e2e_ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t)
    if world > 1:
        # every rank leaves together and without tearing NCCL down (a destroy while a peer still holds captured
        # collectives can block for minutes): rank 0 first finishes its report
        torch.cuda.synchronize()
    if rank != 0:
        sys.stdout.flush()
        os._exit(0)

    peaks = load_peaks()
    img_s = B * world * args.steps / (ms / 1e3)
    e2e_img_s = B * world * e2e_steps / (e2e_ms / 1e3)
    w = WORK[arch]
    fam = profile_plan(tr, torch)
    tot_ms = sum(f["ms"] for f in fam.values())
    top = max(fam.items(), key=lambda kv: kv[1]["ms"])
    top_name, tf = top
    ach = tf["bytes"] / (tf["ms"] / 1e3) / 1e9 if tf["ms"] > 0 else 0.0
    # measured DRAM bytes per launch of that kernel (dram__bytes_read.sum + dram__bytes_write.sum of the committed ncu
    # launch list, same workload: profiles/r01_ncu_launches.md), valid for the default workload only
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if os.path.exists(tpath) and arch == "efficientnet_b0" and B == 256 and args.dtype == "bf16":
        try:
            with open(tpath) as f:
                tj = json.load(f)
            ent = tj.get(top_name[len("dfd_"):] + "_kernel")
            if ent and ent["launches"] == tf["launches"]:
                traffic, traffic_src = ent["dram_bytes_per_launch"], "profiles/r02_ncu_traffic.json (ncu capture of this build, see its 'build' field)"
        except Exception:  # noqa: BLE001
            pass
    if w["bound"] == "tensor":
        # dense-conv models (SURVEY.md 8d): the dominant family is the tcgen05 GEMM; achieved = its algorithmic FLOPs / its time,
        # against the SUSTAINED bf16 matmul rate of MEASURED_PEAKS.json (the kernel runs inside a long step)
        top_name = max((k for k in fam if fam[k]["flops"]), key=lambda k: fam[k]["ms"])
        tf = fam[top_name]
        ach = tf["flops"] / (tf["ms"] / 1e3) / 1e12 if tf["ms"] > 0 else 0.0
        roofline = dict(bound="tensor", kernel=top_name, achieved=round(ach, 1), peak=peaks["tf_sustained"], unit="TFLOP/s",
                        frac=round(ach / peaks["tf_sustained"], 4), peak_burst=peaks["tf_burst"],
                        frac_of_burst=round(ach / peaks["tf_burst"], 4), traffic=None,
                        algorithmic_flops_per_launch=int(tf["flops"] / max(tf["launches"], 1)), peak_source=peaks["source"],
                        kernel_share_of_step=round(tf["ms"] / tot_ms, 4), launches=tf["launches"],
                        step_frac_of_ideal_fusion_roofline=round(img_s / world * w["act_mb"] * 1e6 / (peaks["hbm_gbs"] * 1e9), 4),
                        step_frac_of_tensor_roofline=round(img_s / world * w["gflop"] * 1e9 / (peaks["tf_sustained"] * 1e12), 4),
                        families={k: dict(ms=round(v["ms"], 3), gbs=round(v["bytes"] / max(v["ms"], 1e-9) / 1e6, 1),
                                          tflops=round(v["flops"] / max(v["ms"], 1e-9) / 1e9, 1), n=v["launches"])
                                  for k, v in sorted(fam.items(), key=lambda kv: -kv[1]["ms"])[:8]})
    else:
      roofline = dict(bound="hbm", kernel=top_name, achieved=round(ach, 1), peak=peaks["hbm_gbs"], unit="GB/s",
                    frac=round(ach / peaks["hbm_gbs"], 4), traffic=traffic, traffic_source=traffic_src,
                    algorithmic_bytes_per_launch=int(tf["bytes"] / max(tf["launches"], 1)), peak_source=peaks["source"],
                    kernel_share_of_step=round(tf["ms"] / tot_ms, 4), launches=tf["launches"],
                    step_frac_of_ideal_fusion_roofline=round(img_s / world * w["act_mb"] * 1e6 / (peaks["hbm_gbs"] * 1e9), 4),
                    step_frac_of_tensor_roofline=round(img_s / world * w["gflop"] * 1e9 / (peaks["tf_sustained"] * 1e12), 4),
                    families={k: dict(ms=round(v["ms"], 3), gbs=round(v["bytes"] / max(v["ms"], 1e-9) / 1e6, 1), n=v["launches"])
                              for k, v in sorted(fam.items(), key=lambda kv: -kv[1]["ms"])[:8]})
    cpu = cpu_baseline(arch, sample_steps=args.cpu_steps) if world == 1 and not args.no_cpu else None
    line = dict(metric="images/sec (device-timed, max over ranks) %s 3x%dx%d train step" % (arch, res, res),
                value=round(img_s, 1), unit="images/sec", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                ms_per_step=round(ms / args.steps, 4), higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype=args.dtype, data="synthetic",
                config=dict(workload="%s %s train step, synthetic 3x%dx%d, per-GPU batch %d (%s%s)" % (
                    arch, args.dtype, res, res, B, BASELINE_CFG.get((arch, B, args.dtype), "not a BASELINE.json configuration"),
                    "; DDP weak scaling" if world > 1 else ""), global_batch=B * world,
                    optimizer=args.opt, l2_policy="working set (activations ~6 GB/step) far exceeds the 126 MB L2",
                    cuda_graph=tr._graph is not None, gemm=args.gemm, loss_final=loss_final),
                roofline=roofline, cpu_baseline=cpu,
                e2e=dict(value=round(e2e_img_s, 1), unit="images/sec",
                         h2d_bytes_per_step=int(xh.numel() * xh.element_size() + yh.numel() * 8), d2h_bytes_per_step=16,
                         input="uint8 NCHW pinned host batch, uploaded on a copy stream (2 staging slots) and normalised on the device"),
                gpu_launches=n_launch * args.steps, gpu_launches_per_step=n_launch, clocks=clocks)
    print(json.dumps(line))
    sys.stdout.flush()
    if world > 1:
        os._exit(0)


def cpu_baseline(arch, sample_steps=4, batch=None, world=1):
    """The reference's arithmetic (oracle port: torch fp32 CPU, reference module semantics) timed on the host cores."""
    import torch
    from deepfake_detection_b200.arch import get_spec
    from oracle import train as OT
    from oracle.weights import synth_batch, synth_state
    spec = get_spec(arch)
    res = WORK[arch]["res"]
    b = batch or {"efficientnet_b0": 16, "efficientnet_b4": 4, "resnet50": 8, "resnet18": 8}[arch]
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    sd = synth_state(spec, seed=42)
    opt = OT.OptState(kind="sgd", lr=0.01, momentum=0.9, weight_decay=1e-4)
    x, y = synth_batch(b, 3, res, res, seed=1234)
    # "all the host threads it can use": torch's intra-op pool degrades badly when oversubscribed on shared hosts, so
    # probe a few pool sizes on one step each and keep the fastest (bounded: stop as soon as it gets slower)
    best_t, best_dt = None, None
    for t in [c for c in (8, 16, 32, 64) if c <= avail] or [avail]:
        torch.set_num_threads(t)
        t0 = time.perf_counter()
        OT.train_step(spec, sd, x, y, opt)
        dt = time.perf_counter() - t0
        if best_dt is None or dt < best_dt:
            best_t, best_dt = t, dt
        elif dt > 1.3 * best_dt:
            break
    torch.set_num_threads(best_t)
    done, t0 = 0, time.perf_counter()
    while done < sample_steps and (done == 0 or time.perf_counter() - t0 < 20.0):
        OT.train_step(spec, sd, x, y, opt)
        done += 1
    dt = time.perf_counter() - t0
    return dict(value=round(b * done / dt, 2), unit="images/sec", cores=best_t, host_cpus=avail, cpu_model=cpu_model(), kind="port",
                sample="%d train steps of %s fp32, batch %d, 3x%dx%d, torch CPU ops (oracle port of the reference's dfd.timm "
                       "modules + SGD), %d intra-op threads (fastest of a probe over pool sizes)" % (done, arch, b, res, res, best_t),
                ms_per_step=round(dt / done * 1e3, 1))


def _cpu_ddp_worker(rank, world, arch, b, threads, steps, port, out):
    """one rank of the CPU data-parallel leg: the oracle step with a gloo mean-all-reduce of the gradients (the reference's
    torch DDP on gloo, train.py:402-406), `threads` intra-op threads per rank"""
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from deepfake_detection_b200.arch import get_spec
    from oracle import train as OT
    from oracle.weights import synth_batch, synth_state
    torch.set_num_threads(threads)
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    spec = get_spec(arch)
    res = WORK[arch]["res"]
    sd = synth_state(spec, seed=42)
    opt = OT.OptState(kind="sgd", lr=0.01, momentum=0.9, weight_decay=1e-4)
    x, y = synth_batch(b, 3, res, res, seed=1234 + rank)

    def mean_hook(grads):
        flat = torch.cat([g.reshape(-1) for g in grads.values()])
        dist.all_reduce(flat)
        flat /= world
        o = 0
        for g in grads.values():
            g.copy_(flat[o:o + g.numel()].view_as(g))
            o += g.numel()

    OT.train_step(spec, sd, x, y, opt, grad_hook=mean_hook)          # warm-up
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        OT.train_step(spec, sd, x, y, opt, grad_hook=mean_hook)
    dist.barrier()
    dt = time.perf_counter() - t0
    if rank == 0:
        out.put(dt)
    dist.destroy_process_group()


def cpu_ddp_baseline(arch, world, threads_total, steps=3):
    """SURVEY 8(d): the reference's CPU DDP path - `world` gloo ranks on the host cores, the threads split evenly"""
    import torch.multiprocessing as mp
    b = {"efficientnet_b0": 16, "efficientnet_b4": 4, "resnet50": 8, "resnet18": 8}[arch]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 200
    threads = max(1, threads_total // world)
    procs = [ctx.Process(target=_cpu_ddp_worker, args=(r, world, arch, b, threads, steps, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    dt = q.get(timeout=600)
    for p in procs:
        p.join(timeout=60)
    return dict(value=round(world * b * steps / dt, 2), unit="images/sec", world_size=world, threads_per_rank=threads, backend="gloo",
                per_rank_batch=b, steps=steps, ms_per_step=round(dt / steps * 1e3, 1))


def run_library(args):
    """Stock PyTorch eager on the same B200: the reference's module graph as torch.nn modules (baseline/library_model.py),
    autocast to the benchmark dtype, channels_last, SGD-nesterov, torch DDP over NCCL when launched under torchrun.
    No kernel, plan or engine of this repository is on this path."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from baseline.library_model import build
    from deepfake_detection_b200.arch import get_spec
    arch, B = args.arch, args.batch
    res = args.res or WORK[arch]["res"]
    spec = get_spec(arch)
    torch.manual_seed(42)
    torch.backends.cudnn.benchmark = True
    model = build(spec).cuda().to(memory_format=torch.channels_last)
    if world > 1:
        model = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local_rank])
    decay = [p for n, p in model.named_parameters() if p.dim() > 1 and not n.endswith(".bias")]
    no_decay = [p for n, p in model.named_parameters() if not (p.dim() > 1 and not n.endswith(".bias"))]
    opt = torch.optim.SGD([dict(params=no_decay, weight_decay=0.0), dict(params=decay, weight_decay=1e-4)],
                          lr=0.00001 * B * world, momentum=0.9, nesterov=True)
    adt = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    scaler = torch.amp.GradScaler("cuda", enabled=adt == torch.float16)
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    x = torch.randn(B, spec.in_chans, res, res, device="cuda", generator=g).to(memory_format=torch.channels_last)
    y = torch.randint(0, 2, (B,), device="cuda", generator=g)
    loss_fn = torch.nn.CrossEntropyLoss()

    def step(xb, yb):
        with torch.autocast("cuda", dtype=adt):
            out = model(xb)
            loss = loss_fn(out.float(), yb)
        opt.zero_grad(set_to_none=True)
        scaler.scale(loss).backward()
        scaler.step(opt)
        scaler.update()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step(x, y)
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        loss = step(x, y)
    t1.record()
    barrier()
    ms = t0.elapsed_time(t1)
    # end to end: uint8 pinned host batch, uploaded and normalised with the reference's own prefetcher expressions
    xh = (x * 58.0 + 120.0).clamp_(0, 255).to(torch.uint8).contiguous(memory_format=torch.contiguous_format).cpu().pin_memory()
    yh = y.cpu().pin_memory()
    mean = torch.tensor([v * 255 for v in (0.485, 0.456, 0.406)], device="cuda").view(1, 3, 1, 1)
    std = torch.tensor([v * 255 for v in (0.229, 0.224, 0.225)], device="cuda").view(1, 3, 1, 1)
    pin_out = torch.empty(1).pin_memory()

    def host_step():
        xb = xh.cuda(non_blocking=True).float().sub_(mean).div_(std).contiguous(memory_format=torch.channels_last)
        yb = yh.cuda(non_blocking=True)
        pin_out.copy_(step(xb, yb).detach().float().reshape(1), non_blocking=True)

    for _ in range(3):
        host_step()
    barrier()
    e2e_steps = max(3, args.steps // 2)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(e2e_steps):
        host_step()
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms, e2e_ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(t[0]), float(t[1])
        torch.cuda.synchronize()
    if rank != 0:
        sys.stdout.flush()
        os._exit(0)
    img_s = B * world * args.steps / (ms / 1e3)
    line = dict(impl="library", metric="images/sec (device-timed, max over ranks) %s 3x%dx%d train step" % (arch, res, res),
                value=round(img_s, 1), unit="images/sec", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                ms_per_step=round(ms / args.steps, 4), higher_is_better=True, scaling="weak", vs_baseline=None, dtype=args.dtype,
                data="synthetic",
                config=dict(workload="%s %s train step, synthetic 3x%dx%d, per-GPU batch %d, stock PyTorch %s eager: autocast, "
                                     "channels_last, cudnn.benchmark, SGD-nesterov%s" % (arch, args.dtype, res, res, B, torch.__version__,
                                                                                         ", torch DDP/NCCL" if world > 1 else ""),
                            global_batch=B * world, loss_final=float(loss)),
                e2e=dict(value=round(B * world * e2e_steps / (e2e_ms / 1e3), 1), unit="images/sec",
                         h2d_bytes_per_step=int(xh.numel() + yh.numel() * 8), d2h_bytes_per_step=4), gpu_launches=0)
    print(json.dumps(line))
    sys.stdout.flush()
    if world > 1:
        os._exit(0)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arch = args.arch
    res = WORK[arch]["res"]
    steps = min(args.steps, 6)
    cb = cpu_baseline(arch, sample_steps=steps)
    if args.cpu_world > 1:
        # optional: the same arithmetic as `cpu_world` gloo ranks with the thread pool split (the reference's CPU DDP scaling)
        cb["ddp"] = cpu_ddp_baseline(arch, args.cpu_world, cb["cores"], steps=min(steps, 3))
    line = dict(impl="reference", metric="images/sec (device-timed, max over ranks) %s 3x%dx%d train step" % (arch, res, res),
                value=cb["value"], unit="images/sec", n_gpus=int(os.environ.get("WORLD_SIZE", "1")), steps=steps,
                warmup=1, ms_per_step=cb["ms_per_step"], higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", config=dict(workload="%s train step on host cores, bounded sample (%s)" % (arch, cb["sample"])),
                cpu_baseline=cb, e2e=dict(value=cb["value"], unit="images/sec", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native")
    ap.add_argument("--arch", default="efficientnet_b0")
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--res", type=int, default=0)
    ap.add_argument("--dtype", default="bf16")
    ap.add_argument("--gemm", default="tc")
    ap.add_argument("--opt", default="sgd")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=4)
    ap.add_argument("--cpu-world", type=int, default=1, help="--impl reference: also time N gloo ranks on the host cores")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--impl native: write the outputs of the last timed step as DIR/<name>.npy (64 MB at most)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs is only implemented for --impl native")
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "library":
        run_library(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
