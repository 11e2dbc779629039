"""Benchmark of the UNet-ConvLSTM training step (BASELINE.json metric: train sequences/s, fwd+bwd).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): Moving-MNIST-shaped sequences 64x64, T=20, batch 256 per GPU,
TemporalUNetDualView(base_ch=64, use_skip_lstm=True) -- the authors' width (reference main.py:225-226) --
bf16 tensor-core mode.  One step = forward + backward + AdamW update (fused) on one batch; with N GPUs
the batch of sequences is sharded data-parallel (weak scaling, 256 sequences per GPU) and gradients
are all-reduced over NCCL, overlapped with backward.

Prints ONE JSON line (rank 0).  `value`: inputs resident in HBM.  `e2e`: same step through the public
nn.Module API with the batch in pinned host memory (H2D inside the timed region, loss read back).
`roofline`: the fused ConvLSTM gate-conv kernel, timed per launch with CUDA events inside the timed
region.  `cpu_baseline` / `--impl reference`: the UNMODIFIED reference (its train/unet.py model and main.py
compute_loss, from the checkout B200_REFERENCE_DIR names; kind "reference") on this box's host cores, on a bounded
sample; oracle/torch_port.py (kind "port") when no checkout is named.
`--dump-outputs DIR`: after the timed steps, what the last of them computed is written to DIR as float32 .npy files
(see dump_outputs); the inputs depend only on the arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "train sequences/sec (fwd+bwd)"
UNIT = "sequences/s"


# ------------------------------------------------------------------------------------------------
# synthetic Moving-MNIST-shaped data (mirrors digits/build_moving_mnist.py:5-58 without the download):
# two 28x28 blobs with integer velocities bouncing off the borders; channel 1 is the same frame as
# seen one pixel to the right ("second satellite"); target = per-pixel x-velocity of the blobs / 10
# ------------------------------------------------------------------------------------------------
def make_batch(B, T, S, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:28, 0:28]
    X = np.zeros((B, T, 2, S, S), dtype=np.float32)
    Y = np.zeros((B, T, 1, S, S), dtype=np.float32)
    for b in range(B):
        for _ in range(2):
            cx, cy, sg = rng.uniform(9, 19), rng.uniform(9, 19), rng.uniform(3, 6)
            blob = np.exp(-((xx - cx) ** 2 + (yy - cy) ** 2) / (2 * sg * sg)).astype(np.float32)
            blob[blob < 0.35] = 0.0
            px, py = rng.integers(0, S - 28, size=2)
            vx, vy = rng.integers(-5, 6, size=2)
            for t in range(T):
                X[b, t, 0, py:py + 28, px:px + 28] = np.maximum(X[b, t, 0, py:py + 28, px:px + 28], blob)
                Y[b, t, 0, py:py + 28, px:px + 28] += (blob > 0) * (vx / 10.0)
                nx, ny = px + vx, py + vy
                if nx < 0 or nx > S - 28:
                    vx = -vx
                    nx = px + vx
                if ny < 0 or ny > S - 28:
                    vy = -vy
                    ny = py + vy
                px, py = int(nx), int(ny)
    X[:, :, 1, :, 1:] = X[:, :, 0, :, :-1]
    M = (X[:, :, :1] > 0).astype(np.float32)  # "cloud mask": the pixels the target is defined on (unet.py:279)
    return torch.from_numpy(X), torch.from_numpy(np.clip(Y, -1, 1)), torch.from_numpy(M)


def loss_torch(y_pred, y, mask):
    """The reference's training loss (main.py:28-72: weighted L1 + 0.005 x spatial-gradient loss, masked means)
    written with torch operators -- the CPU reference arm's loss; the B200 arm uses the fused kernels of
    unet_convlstm_b200.loss on the same formula (both pinned by tests/golden/loss_main_compute_loss.npz)."""
    w = 1.0 + 4.0 * y.abs() ** 3
    d = y_pred - y
    l1 = (d.abs() * mask * w).sum() / ((mask * w).sum() + 1e-8)
    dxe = d[..., :-1, 1:] - d[..., :-1, :-1]
    dye = d[..., 1:, :-1] - d[..., :-1, :-1]
    mc = mask[..., :-1, :-1]
    return l1 + 0.005 * ((dxe.abs() + dye.abs()) * mc).sum() / (mc.sum() + 1e-8)


# ------------------------------------------------------------------------------------------------
def clocks_sampler_start(gpu_index):
    q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    try:
        f = tempfile.TemporaryFile("w+")  # not in the tree: bench.py writes nothing there
        return subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200",
                                 "-i", str(gpu_index)], stdout=f, stderr=subprocess.DEVNULL), f
    except OSError:
        return None, None


def clocks_summary(proc, f):
    if proc is None:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    proc.terminate()
    try:
        proc.wait(timeout=5)
    except subprocess.TimeoutExpired:
        proc.kill()
    f.seek(0)
    lines = f.readlines()
    f.close()
    sm, smax, reasons = [], None, set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for line in lines:
        c = [v.strip() for v in line.split(",")]
        if len(c) < 9:
            continue
        try:
            sm.append(float(c[1]))
            smax = float(c[2])
        except ValueError:
            continue
        for nm, v in zip(names, c[5:9]):
            if v.lower().startswith("active"):
                reasons.add(nm)
    # "under load": the upper half of the samples (the sampler also sees idle gaps around the region)
    sm.sort()
    load = sm[len(sm) // 2:] if sm else []
    return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
            "samples": len(sm)}


def host_info():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return model, len(os.sched_getaffinity(0))


# ------------------------------------------------------------------------------------------------
# the reference's CPU path (oracle/torch_port.py) -- cpu_baseline leg and --impl reference
# ------------------------------------------------------------------------------------------------
def load_reference():
    """The UNMODIFIED reference (train/unet.py's TemporalUNetDualView, main.py's compute_loss) from the checkout
    B200_REFERENCE_DIR names.  Loaded by file path under private module names, so this repository's own `train.unet`
    stays what `import train.unet` means.  Returns (model class, compute_loss, source dir) or None without a checkout."""
    import importlib.util
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import run_reference as RR
        ref = RR.reference_root()
    except Exception:  # noqa: BLE001
        return None
    finally:
        sys.path.pop(0)
    RR.install_stubs()  # train/resnet18.py (imported by main.py) needs segmentation_models_pytorch

    def load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(ref, rel))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
        return mod

    ref_unet = load("b200_reference_unet", "train/unet.py")
    if ref not in sys.path:
        sys.path.append(ref)  # main.py: `from train.resnet18 import ...` (namespace package `train`)
    ref_main = load("b200_reference_main", "main.py")
    return ref_unet.TemporalUNetDualView, ref_main.compute_loss, ref


def cpu_reference_run(args, steps, warmup, batch):
    """The reference's training step (main.py:94-108) on the host cores.  kind "reference": the reference's own
    modules (load_reference); kind "port": oracle/torch_port.py, only when no copy of the reference is available."""
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    x, y, mask = make_batch(batch, args.seq_len, args.size, 1234)
    loaded = load_reference()
    if loaded is not None:
        Model, ref_loss, src = loaded
        model = Model(base_ch=args.base_ch, use_skip_lstm=True).train()
        params = list(model.parameters())
        kind = "reference"

        def fwd_loss():
            out, _ = model(x)
            return ref_loss(torch.stack(out, dim=1), y, mask)
    else:
        from oracle import torch_port as TP
        from train.unet import TemporalUNetDualView
        sd = TemporalUNetDualView(base_ch=args.base_ch, use_skip_lstm=True).state_dict()
        p = TP.params_from_state_dict(sd, torch.float32)
        params = [v for v in p.values() if v.requires_grad]
        kind, src = "port", "oracle/torch_port.py"

        def fwd_loss():
            out, _ = TP.temporal_unet(p, x, None, training=True)
            return loss_torch(torch.stack(out, dim=1), y, mask)
    opt = torch.optim.AdamW(params, lr=1e-3, weight_decay=1e-4)

    def step():
        opt.zero_grad(set_to_none=True)
        loss = fwd_loss()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()
        return loss.item()

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return batch / dt, dt, cores, kind, src


def run_reference_arm(args, out):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # bounded sample: 4 sequences per step (2 when many steps are asked for) so the run ends in minutes
    batch = 4 if args.steps + args.warmup <= 10 else 2
    value, dt, cores, kind, src = cpu_reference_run(args, args.steps, args.warmup, batch)
    cpu_model, _ = host_info()
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, batch_per_step=batch),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "cpu": cpu_model, "source": src,
                         "sample": f"{batch} sequence(s) per step (T={args.seq_len}, {args.size}x{args.size}, base_ch "
                                   f"{args.base_ch} + skip LSTMs), fwd + compute_loss + bwd + clip + AdamW, fp32, torch {torch.__version__} CPU "
                                   f"(oneDNN), {args.steps} timed steps"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=out, flush=True)


def workload_config(args, batch_per_step=None):
    shape = (args.size, args.seq_len, args.batch, args.base_ch)
    which = {(64, 20, 256, 64): "BASELINE.json configs[1]", (128, 10, 32, 64): "BASELINE.json configs[2] shape",
             (256, 16, 8, 128): "BASELINE.json configs[3] shape"}.get(shape, "custom shape")
    kind = "Moving-MNIST-shaped" if args.size == 64 else "cloud-sequence-shaped (synthetic blobs)"
    return {
        "workload": f"{kind} UNet-ConvLSTM {args.size}x{args.size}, T={args.seq_len}, "
                    f"batch {args.batch} per GPU, base_ch {args.base_ch} + skip ConvLSTMs ({which})",
        "batch_per_gpu": args.batch if batch_per_step is None else batch_per_step, "seq_len": args.seq_len,
        "image": args.size, "base_ch": args.base_ch, "use_skip_lstm": True, "precision": args.precision,
        "step": "the reference's training step (main.py:94-108): forward, compute_loss (weighted L1 + gradient loss, "
                "masked), backward, clip_grad_norm_(1.0) + AdamW (multi-tensor kernels) update; gradient all-reduce overlapped when N > 1",
        "parallelism": f"dp{args.gpus}",
        "l2": "per-step working set (tens of GB of activations, 168 MB of inputs at configs[1]) far exceeds the 126 MB L2",
    }


# ------------------------------------------------------------------------------------------------
def run_b200_arm(args, out):
    import torch.distributed as dist
    import unet_convlstm_b200 as pkg
    from train.unet import TemporalUNetDualView
    from unet_convlstm_b200 import _lib, ops
    from unet_convlstm_b200.dist import GradReducer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    pkg.set_precision(args.precision)
    _lib.lib()  # fail loudly if the CUDA library is missing
    ops.enable_background_wgrad()  # this step reads gradients after backward() (own optimizer / GradReducer)

    torch.manual_seed(0)  # identical replicas
    model = TemporalUNetDualView(base_ch=args.base_ch, use_skip_lstm=True).to(dev)
    model.train()
    # B200_OPTIM=torch: torch's foreach clip_grad_norm_ + fused AdamW instead of the multi-tensor kernels of
    # unet_convlstm_b200/optim.py (A/B switch)
    own_optim = os.environ.get("B200_OPTIM", "b200") != "torch"
    if own_optim:
        from unet_convlstm_b200.optim import AdamW as B200AdamW
        opt = B200AdamW(model.parameters(), lr=1e-3, weight_decay=1e-4)
    else:
        opt = torch.optim.AdamW(model.parameters(), lr=1e-3, weight_decay=1e-4, fused=True)
    reducer = GradReducer(model.parameters()) if world > 1 else None

    from unet_convlstm_b200.loss import compute_loss
    x_host, y_host, m_host = make_batch(args.batch, args.seq_len, args.size, 1234 + rank)
    x_host, y_host, m_host = x_host.pin_memory(), y_host.pin_memory(), m_host.pin_memory()
    x_dev, y_dev, m_dev = x_host.to(dev), y_host.to(dev), m_host.to(dev)
    params = [q for q in model.parameters() if q.requires_grad]
    last = {}  # with --dump-outputs: the predictions and loss of the last timed step

    def step(x, y, m, with_opt=True, keep=False):
        # the reference's training step (main.py:94-108): forward, compute_loss, backward, clip_grad_norm_(1.0),
        # optimizer step
        opt.zero_grad(set_to_none=True)
        out, _ = model(x)
        y_pred = torch.stack(out, dim=1)
        loss = compute_loss(y_pred, y, m)
        if keep:
            last.update(pred=y_pred.detach(), loss=loss.detach())
        loss.backward()
        if reducer is not None:
            reducer.finish()
        if with_opt and own_optim:
            opt.step(clip_max_norm=1.0)        # global-norm clip folded into the multi-tensor AdamW kernel
        elif with_opt:
            torch.nn.utils.clip_grad_norm_(params, 1.0)
            opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_profile = {}

    def timed(fn, steps, tag=None):
        """K steps between two barriers, timed on the device with CUDA events, max over ranks.  One extra event per step
        gives the per-step durations of this rank (`tag`: kept in step_profile, gathered over the ranks for the JSON line)."""
        import gc
        barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        st0 = torch.cuda.memory_stats(dev)
        gc0 = [g["collections"] for g in gc.get_stats()]
        host = [time.perf_counter()]
        ev[0].record()
        for i in range(steps):
            fn()
            ev[i + 1].record()
            host.append(time.perf_counter())
        barrier()
        st1 = torch.cuda.memory_stats(dev)
        gc1 = [g["collections"] for g in gc.get_stats()]
        ms = torch.tensor([ev[0].elapsed_time(ev[-1])], device=dev)
        if tag is not None:
            step_profile[tag + "_host"] = {
                "cudaMalloc_calls": st1.get("num_device_alloc", 0) - st0.get("num_device_alloc", 0),
                "cudaFree_calls": st1.get("num_device_free", 0) - st0.get("num_device_free", 0),
                "alloc_retries": st1.get("num_alloc_retries", 0) - st0.get("num_alloc_retries", 0),
                "gc_collections": [b - a for a, b in zip(gc0, gc1)],
                "rank0_host_ms_per_step": [round((host[i + 1] - host[i]) * 1e3, 1) for i in range(steps)]}
            per = torch.tensor([ev[i].elapsed_time(ev[i + 1]) for i in range(steps)], device=dev)
            if world > 1:
                allp = [torch.empty_like(per) for _ in range(world)]
                dist.all_gather(allp, per)
            else:
                allp = [per]
            step_profile[tag] = {"per_rank_median_ms": [round(float(q.median()), 2) for q in allp],
                                 "per_rank_max_ms": [round(float(q.max()), 2) for q in allp],
                                 "rank0_steps_ms": [round(float(v), 1) for v in per.tolist()]}
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps

    if args.profile_steps:
        # for `ncu`: one warm-up step (packs weights, sizes the caching allocator) + N plain steps, no timing
        for _ in range(1 + args.profile_steps):
            step(x_dev, y_dev, m_dev)
        torch.cuda.synchronize()
        return

    for _ in range(args.warmup):
        step(x_dev, y_dev, m_dev)

    if args.breakdown:
        # one instrumented step: CUDA events around every C-ABI call (adds event overhead; the per-kernel
        # numbers it prints are for orientation, the judged ones come from the plain timed region + ncu)
        _lib.TIMER = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step(x_dev, y_dev, m_dev)
        e1.record()
        torch.cuda.synchronize()
        ev, _lib.TIMER = _lib.TIMER, None
        agg = {}
        if args.timeline:
            # start / end of every C-ABI call relative to the start of the step, with the stream it ran on
            streams = {}
            with open(args.timeline, "w") as tf:
                tf.write("start_ms,end_ms,stream,label\n")
                for label, a, b, work, st in ev:
                    tf.write(f"{e0.elapsed_time(a):.4f},{e0.elapsed_time(b):.4f},{streams.setdefault(st, len(streams))},{label}\n")
        for label, a, b, work, _st in ev:
            d = agg.setdefault(label, [0, 0.0, 0.0, 0.0])
            d[0] += 1
            d[1] += a.elapsed_time(b)
            if work is not None:
                d[2] += work[0] or 0.0
                d[3] += work[1] or 0.0
        tot = sum(d[1] for d in agg.values())
        print(f"# breakdown of one step: {e0.elapsed_time(e1):.1f} ms wall, {tot:.1f} ms inside {len(ev)} C-ABI calls",
              file=sys.stderr)
        for label, d in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            rate = ""
            if d[2]:
                rate = f"{d[2] / d[1] / 1e9:8.1f} TFLOP/s"
            elif d[3]:
                rate = f"{d[3] / d[1] / 1e6:8.1f} GB/s"
            print(f"# {d[1]:9.3f} ms {100 * d[1] / tot:5.1f}% x{d[0]:<4d} {rate:>18s}  {label}", file=sys.stderr)

    proc, f = clocks_sampler_start(local) if rank == 0 else (None, None)

    # ---- eager region: every launch from Python, CUDA events around each fused cell launch (roofline) ----
    ops.CELL_TIMER = []
    calls0 = _lib.kernel_launches()
    steps_done = [0]

    def value_step():
        steps_done[0] += 1
        return step(x_dev, y_dev, m_dev, keep=bool(args.dump_outputs) and rank == 0 and steps_done[0] == args.steps)

    ms_eager = timed(value_step, args.steps, tag="value")
    launches = _lib.kernel_launches() - calls0
    cell_events, ops.CELL_TIMER = ops.CELL_TIMER, None
    torch.cuda.synchronize()
    if last:
        dump_outputs(args.dump_outputs, last, model)
        last.clear()
    cell_ms = [a.elapsed_time(b) for a, b, _ in cell_events]
    cell_flops = [fl for _, _, fl in cell_events]

    # ---- fwd+bwd only (no optimizer), for the record --------------------------------------------
    ms_fb = timed(lambda: step(x_dev, y_dev, m_dev, with_opt=False), max(1, args.steps // 2), tag="fwd_bwd_only")
    # ---- timed region 1: inputs resident in HBM = the eager region above.  (Round 1 could also replay the step from
    #      a CUDA graph; measured 232.7 ms graphed vs 233.3 ms eager -- the step is GPU-bound, the host runs ahead --
    #      so the graph path was removed in round 2.) ----
    ms_step = ms_eager

    # ---- timed region 2: end to end through the module API, batch in pinned host memory ----------
    # Every step copies its own batch from pinned host memory (K copies inside the timed region) and reads
    # the loss back; the copy of batch i+1 runs on a side stream while batch i computes
    # (unet_convlstm_b200.data.DevicePrefetcher), so only the first copy of the region is exposed.
    from unet_convlstm_b200.data import DevicePrefetcher
    pf = DevicePrefetcher(dev)

    def e2e_region(steps):
        pf.start(x_host, y_host, m_host)
        for i in range(steps):
            x, y, m = pf.get()
            if i + 1 < steps:
                pf.start(x_host, y_host, m_host)
            step(x, y, m).item()

    e2e_region(2)
    ms_e2e = timed(lambda: e2e_region(args.steps), 1) / args.steps

    clocks = clocks_summary(proc, f) if rank == 0 else None
    peak_mem = torch.cuda.max_memory_allocated(dev)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except (OSError, ValueError):
            pass
        peak_tf = peaks.get("bf16_tflops_sustained")
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)"
        if peak_tf is None:
            peak_tf, peak_src = 1400.0, "fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained)"
        full = [(m, fl) for m, fl in zip(cell_ms, cell_flops) if fl == max(cell_flops)] if cell_flops else []
        ach = (sum(fl for _, fl in full) / (sum(m for m, _ in full) * 1e-3) / 1e12) if full else None
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json"))).get("cell_fwd_bytes_per_launch")
        except (OSError, ValueError):
            pass
        line = {
            "metric": METRIC, "value": world * args.batch / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": workload_config(args),
            "e2e": {"value": world * args.batch / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": (x_host.numel() + y_host.numel() + m_host.numel()) * 4,
                    "d2h_bytes_per_step": 4},
            "fwd_bwd_only": {"value": world * args.batch / (ms_fb * 1e-3), "unit": UNIT, "ms_per_step": ms_fb},
            "eager": {"value": world * args.batch / (ms_eager * 1e-3), "unit": UNIT, "ms_per_step": ms_eager,
                      "note": "same step launched kernel by kernel from Python (no CUDA graph)"},
            "cuda_graph": False,
            "gpu_launches": launches,
            "roofline": {"kernel": "conv_tc2_kernel<256, EPI_LSTM>: fused ConvLSTM gate conv + gate math + c/h update, "
                                   "forward, CTA pairs (tcgen05 cta_group::2), one timestep-persistent launch per "
                                   "layer (T steps)",
                         "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": (ach / peak_tf) if ach else None, "traffic": traffic, "peak_source": peak_src,
                         "launches_timed": len(full),
                         "avg_launch_ms": (sum(m for m, _ in full) / len(full)) if full else None,
                         "flops_per_launch": max(cell_flops) if cell_flops else None,
                         "share_of_step": (sum(cell_ms) / args.steps / ms_eager) if cell_ms else None},
            "clocks": clocks,
            "step_profile": step_profile,
            "peak_mem_gb": peak_mem / 2 ** 30,
        }
        if world == 1 and not args.no_cpu_baseline:
            v, dt, cores, kind, src = cpu_reference_run(args, 2, 1, args.cpu_sample)
            cpu_model, _ = host_info()
            line["cpu_baseline"] = {
                "value": v, "unit": UNIT, "cores": cores, "kind": kind, "cpu": cpu_model, "source": src,
                "sample": f"{args.cpu_sample} sequence(s) per step, 1 warm-up + 2 timed training steps (fwd, compute_loss, bwd, clip, AdamW) "
                          f"of the same model and shapes (T={args.seq_len}, {args.size}x{args.size}), fp32, torch "
                          f"{torch.__version__} CPU (oneDNN), {dt:.1f} s per step"}
        print(json.dumps(line), file=out, flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 64_000_000
DUMP_PARAM_SAMPLE = 4096
NPY_HEADER = 256  # upper bound of the header np.save writes in front of the data


def dump_outputs(path, last, model):
    """Writes what the last timed step computed to `path`, float32: loss.npy (the scalar loss), pred.npy (the predictions
    [B', T, 1, H, W] of B' of the B sequences, a seeded choice so the files stay under DUMP_BYTES) and
    param.<name>.npy (each parameter after the optimizer step, or a seeded sample of DUMP_PARAM_SAMPLE of its elements
    in flat order)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    rng = np.random.default_rng(0)
    arrays = {"loss": last["loss"].detach().float().reshape(())}
    for name, p in model.named_parameters():
        flat = p.detach().float().reshape(-1)
        if flat.numel() > DUMP_PARAM_SAMPLE:
            idx = np.sort(rng.choice(flat.numel(), DUMP_PARAM_SAMPLE, replace=False))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        arrays[f"param.{name}"] = flat
    pred = last["pred"].detach().float()
    room = DUMP_BYTES - sum(a.numel() * 4 + NPY_HEADER for a in arrays.values()) - NPY_HEADER
    keep = min(pred.shape[0], room // (pred[0].numel() * 4))
    if keep < pred.shape[0]:
        idx = np.sort(rng.choice(pred.shape[0], keep, replace=False))
        pred = pred[torch.from_numpy(idx).to(pred.device)]
    arrays["pred"] = pred
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a.cpu().numpy())


def _claim_stdout():
    """The contract is ONE JSON line on stdout: libraries that print there (NCCL's version banner on
    rank 0) are sent to stderr; the JSON line goes to the saved descriptor."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="sequences per GPU and step")
    ap.add_argument("--seq-len", type=int, default=20)
    ap.add_argument("--size", type=int, default=64)
    ap.add_argument("--base-ch", type=int, default=64)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "tf32", "fp32"])
    ap.add_argument("--cpu-sample", type=int, default=4, help="sequences in the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--breakdown", action="store_true", help="print a per-entry-point time table to stderr")
    ap.add_argument("--timeline", default="", help="with --breakdown: write start/end/stream of every C-ABI call to this CSV")
    ap.add_argument("--profile-steps", type=int, default=0, help="run 1 warm-up + N untimed steps and exit (for ncu)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the loss, predictions and updated parameters of the last timed step to DIR as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the B200 path computed: not with --impl reference")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3  # timing rule: at least 3 warm-up steps
    out = _claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args, out)
    else:
        try:
            run_b200_arm(args, out)
        except BaseException:
            # a device-side watchdog (csrc/ptx.cuh mbar_wait) names the barrier it timed out on
            try:
                from unet_convlstm_b200 import _lib
                print(f"bench.py: b200_device_error() = {_lib.lib().b200_device_error()}", file=sys.stderr, flush=True)
            except Exception:  # noqa: BLE001
                pass
            raise
    out.flush()


if __name__ == "__main__":
    main()
