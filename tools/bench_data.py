"""Input pipeline of the training loop: host loaders against the device-resident dataset.

    python tools/bench_data.py [--steps 6] [--warmup 2] [--rounds 2] [--out FILE]

For each shape -- BASELINE.json configs[1] (64x64, T = 20, batch 256) and the configs[2] shape (128x128, T = 10,
batch 32), both with TemporalUNetDualView(base_ch=64, use_skip_lstm=True) in the bf16 mode -- on a synthetic NPZ
generated from a seed (N sequences, the reference's keys X [N,T,2,H,W] / Y [N,T,1,H,W], default explicit constants
and asinh):

  * training throughput of loop.train_one_epoch over `--steps` batches, fed (a) by the host DataLoaders of
    loop.make_loaders (NPZSequenceDataset.__getitem__ + collate + pin + side-stream copy) and (b) by
    make_loaders(device=...) (one b200_sequence_batch launch per batch), alternating a / b for `--rounds` rounds after
    `--warmup` steps of each; host clock around each call, which ends in a device synchronisation;
  * each loader alone, without training: batches drawn epoch after epoch for at least ALONE_SECONDS;
  * the kernel: CUDA events around KERNEL_LAUNCHES launches, each on its own random batch of indices (the rows read
    change from launch to launch; the dataset, 2.0 / 1.3 GB, is far larger than the 126 MB L2), and its bytes (12 read
    + 16 written per pixel-timestep) over that time against the data-sheet 7.7 TB/s of a B200.

The card, its power limit and the host CPU are printed with the numbers.  Needs a CUDA device; writes only the NPZ
(to a temporary directory) and --out.
"""
from __future__ import annotations

import argparse
import itertools
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

HBM_PEAK = 7.7e12  # bytes/s, NVIDIA HGX B200 data sheet, one GPU
SHAPES = [("configs[1]", 64, 20, 256, 2048), ("configs[2] shape", 128, 10, 32, 1024)]  # (label, size, T, batch, N)
ALONE_SECONDS = 2.0   # least time each loader is drained for without training
KERNEL_LAUNCHES = 200


class _Take:
    """The first k batches of one pass over `loader`."""

    def __init__(self, loader, k):
        self.loader, self.k = loader, k

    def __iter__(self):
        return itertools.islice(iter(self.loader), self.k)


def card():
    name = torch.cuda.get_device_name()
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def host_cpu():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return model, len(os.sched_getaffinity(0)), os.cpu_count()


def synthetic_npz(path, N, T, S, seed):
    rng = np.random.default_rng(seed)
    X = rng.random((N, T, 2, S, S), dtype=np.float32) * np.float32(3.0)
    Y = rng.standard_normal((N, T, 1, S, S), dtype=np.float32) * np.float32(4.0)
    np.savez(path, X=X, Y=Y)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def run_shape(label, S, T, B, N, args, log):
    import unet_convlstm_b200 as pkg
    from train.unet import NPZSequenceDataset, TemporalUNetDualView
    from unet_convlstm_b200.loop import make_loaders, train_one_epoch
    from unet_convlstm_b200.optim import AdamW

    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "seq.npz")
        synthetic_npz(path, N, T, S, seed=1234)
        ds = NPZSequenceDataset(path)
    dev = torch.device("cuda", torch.cuda.current_device())
    torch.manual_seed(0)
    host_tr, _ = make_loaders(ds, B)
    torch.manual_seed(0)
    dev_tr, _ = make_loaders(ds, B, device=dev)
    steps = min(args.steps, len(host_tr))

    arms = {"host": host_tr, "device": dev_tr}
    pkg.set_precision("bf16")
    torch.manual_seed(0)
    model = TemporalUNetDualView(base_ch=64, use_skip_lstm=True).to(dev)
    opt = AdamW(model.parameters(), lr=1e-3, weight_decay=1e-4)
    for loader in arms.values():  # warm-up: module loads, workspaces, allocator
        timed(lambda: train_one_epoch(model, _Take(loader, args.warmup), opt, dev, ds))
    train = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, loader in arms.items():
            train[k].append(steps * B / timed(lambda: train_one_epoch(model, _Take(loader, steps), opt, dev, ds)))
    del model, opt

    def drain(loader):
        """Batches of `loader`, epoch after epoch, for at least ALONE_SECONDS (then a device synchronisation):
        (batches, sequences, seconds).  Each epoch ends in a partial batch, so sequences are counted, not batches."""
        n = seqs = 0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < ALONE_SECONDS:
            for b in loader:
                b[0].to(dev, non_blocking=True)  # host batches: the copy the training loop would make
                n += 1
                seqs += b[0].shape[0]
                if time.perf_counter() - t0 >= ALONE_SECONDS:
                    break
        torch.cuda.synchronize()
        return n, seqs, time.perf_counter() - t0
    alone = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, loader in arms.items():
            alone[k].append(drain(loader))

    data = dev_tr.data
    g = torch.Generator().manual_seed(5)
    idx = [data.device_indices(torch.randint(0, N, (B,), generator=g)) for _ in range(KERNEL_LAUNCHES)]
    for i in range(5):
        data._batch(idx[i])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in idx:
        data._batch(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / KERNEL_LAUNCHES
    nbytes = B * T * S * S * 28

    log(f"\n== {label}: {S}x{S}, T = {T}, batch {B}, N = {N} synthetic sequences")
    log(f"training (base_ch 64 + skip ConvLSTMs, bf16), loop.train_one_epoch over {steps} batches, alternating "
        f"host / device, {args.rounds} rounds after {args.warmup} warm-up batches each (sequences/s):")
    for k in arms:
        log(f"  {k:6s} loaders: " + "  ".join(f"{v:8.1f}" for v in train[k]))
    log(f"  device / host: {np.median(train['device']) / np.median(train['host']):.2f}x (medians)")
    log(f"loaders alone, no training, batches drawn for at least {ALONE_SECONDS:g} s per round (sequences/s):")
    for k in arms:
        log(f"  {k:6s} loaders: " + "  ".join(f"{q / t:9.1f} ({n} batches in {t:.2f} s)" for n, q, t in alone[k]))
    log(f"b200_sequence_batch: {ms * 1e3:.1f} us per batch (CUDA events, {KERNEL_LAUNCHES} launches, a new random "
        f"batch of {B} indices each); "
        f"{nbytes / 1e6:.1f} MB moved (28 B per pixel-timestep) = {nbytes / ms / 1e9:.2f} TB/s, "
        f"{100 * nbytes / (ms * 1e-3) / HBM_PEAK:.1f} % of the 7.7 TB/s data-sheet HBM bandwidth")


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    ap.add_argument("--shape", type=int, default=None, help=argparse.SUPPRESS)  # one entry of SHAPES, in this process
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_data.py needs a CUDA device")
    if args.shape is not None:
        run_shape(*SHAPES[args.shape], args, lambda s: print(s, flush=True))
        return
    name, power = card()
    cpu, usable, total = host_cpu()
    lines = [f"card: {name}, power limit {power}; host CPU: {cpu}, {usable} usable of {total} logical cores; "
             f"torch {torch.__version__}, NumPy {np.__version__}; host loaders with num_workers = 0 (as main.py); "
             "each shape in a process of its own"]
    print(lines[0], flush=True)
    for i in range(len(SHAPES)):
        # one model per process, like bench.py's runs of each configuration
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--shape", str(i), "--steps", str(args.steps),
                            "--warmup", str(args.warmup), "--rounds", str(args.rounds)], capture_output=True, text=True)
        sys.stderr.write(r.stderr[-4000:])
        if r.returncode != 0:
            raise SystemExit(f"bench_data.py: shape {SHAPES[i][0]} failed (exit {r.returncode})")
        out = [ln for ln in r.stdout.splitlines() if not ln.startswith("[")]   # the dataset's [INFO] lines
        print("\n".join(out), flush=True)
        lines += out
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
