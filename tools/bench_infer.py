"""Inference of the UNet-ConvLSTM (SURVEY.md section 8 f3) on one GPU, bf16.

    python tools/bench_infer.py [B T size base_ch]      whole sequences: folded-BatchNorm no_grad forward against the
                                                        unfused eval path (autograd enabled)
    python tools/bench_infer.py --stream [T size base_ch]
        online use, frames arriving one at a time, per-frame latency at B = 1, 8, 64 of
          (a) prefix  the exact O(T^2) method of the reference's test.py: model(x[:, :t+1]) for every new frame
          (b) forward model(x[:, t:t+1], state): carries only the temporal state (the skip cells restart from zero), not exact
          (c) stream  TemporalUNetDualView.stream(): every state carried, CUDA-graph replay, split K -- exact
              (c0 = the same without split K; "replayed" = frames 2.. of the sequence, which are graph replays)
        device time from CUDA events around each whole sequence, host time from a wall clock around it (ends in a
        synchronize); then the kernel A/B of split against unsplit K at the single-frame cell and folded-conv shapes.
The card name and power limit are printed first: they are part of every number below them."""
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import unet_convlstm_b200 as pkg  # noqa: E402
from train.unet import TemporalUNetDualView  # noqa: E402
from unet_convlstm_b200 import _lib, ops  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return f"{torch.cuda.get_device_name(0)} | nvidia-smi: {q}"


def timeit(fn, iters=3, warm=2):
    """(device ms, host ms) per call: CUDA events and a wall clock around `iters` calls, after `warm` calls."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, (time.perf_counter() - t0) * 1e3 / iters


def whole_sequences(B, T, S, b):
    torch.manual_seed(0)
    m = TemporalUNetDualView(base_ch=b, use_skip_lstm=True).cuda().eval()
    x = torch.rand(B, T, 2, S, S, device="cuda")

    def folded():
        with torch.no_grad():
            m(x)

    ms_f, _ = timeit(folded)
    ms_u, _ = timeit(lambda: m(x))
    print(f"inference B{B} T{T} {S}x{S} base_ch{b}: folded-BN no_grad {ms_f:8.2f} ms = {B / ms_f * 1e3:8.1f} seq/s | "
          f"unfused eval {ms_u:8.2f} ms = {B / ms_u * 1e3:8.1f} seq/s", flush=True)


def streaming(T, S, b):
    torch.manual_seed(0)
    m = TemporalUNetDualView(base_ch=b, use_skip_lstm=True).cuda().eval()
    print(f"\nper-frame latency, {S}x{S} T={T} base_ch={b} + skip LSTMs, bf16 (ms per frame: device | host)", flush=True)
    for B in (1, 8, 64):
        x = torch.rand(B, T, 2, S, S, device="cuda")

        def prefix():
            with torch.no_grad():
                for t in range(T):
                    m(x[:, :t + 1])

        def fwd():
            with torch.no_grad():
                st = None
                for t in range(T):
                    _, st = m(x[:, t:t + 1], st)

        def stream_of(fs):
            def run():      # one sequence: reset() keeps the captured graph of the previous one
                fs.reset()
                for t in range(T):
                    fs.step(x[:, t])
            return run

        res = {"(a) prefix": timeit(prefix, 1, 1), "(b) forward": timeit(fwd), "(c) stream": timeit(stream_of(m.stream()))}
        # steady state of a stream: frames 2.. are graph replays
        s = m.stream()
        for t in range(3):
            s.step(x[:, t])
        res["(c) replayed"] = tuple(v * T for v in timeit(lambda: s.step(x[:, 5]), 3 * T, 2))
        split = ops.splitk_splits
        ops.splitk_splits = lambda *a: 1
        try:
            res["(c0) stream no split"] = timeit(stream_of(m.stream()))
            s = m.stream()
            for t in range(3):
                s.step(x[:, t])
            res["(c0) replayed no split"] = tuple(v * T for v in timeit(lambda: s.step(x[:, 5]), 3 * T, 2))
        finally:
            ops.splitk_splits = split
        print(f"  B={B:3d}  " + "  ".join(f"{k} {d / T:7.3f} | {h / T:7.3f}" for k, (d, h) in res.items()), flush=True)


def kernel_ab():
    """Split against unsplit K on identical operands, one frame.  The unsplit legs are what forward runs at T = 1: the
    timestep-persistent cell launch and the folded-BatchNorm conv.  Weights and activations of one layer fit in the
    126 MB L2 except the temporal cell's (151 MB): repeated launches read them from L2, a cold frame from HBM."""
    print("\nkernel A/B, bf16, one frame, us per call (CUDA events over 200 calls); S* = b200_splitk_splits", flush=True)
    lib = _lib.lib()
    dev = "cuda"
    for B in (1, 8):
        for H, Ch in ((4, 1024), (8, 512), (16, 256)):
            torch.manual_seed(0)
            w = (torch.randn(4 * Ch, 2 * Ch, 3, 3, device=dev) * (1.0 / (18 * Ch) ** 0.5))
            wp, bp = ops.pack_lstm_weight(w, (0.1 * torch.randn(4 * Ch, device=dev)), torch.bfloat16)
            x = torch.randn(1, B, H, H, Ch, device=dev).bfloat16()
            h_all = torch.randn(2, B, H, H, Ch, device=dev).bfloat16()
            c_all = torch.randn(2, B, H, H, Ch, device=dev)
            gates = torch.empty(1, B, H, H, 4 * Ch, device=dev, dtype=torch.bfloat16)
            s_rule = lib.b200_splitk_splits(B, H, H, Ch, Ch, 4 * Ch, 3)
            un, _ = timeit(lambda: ops.lstm_seq_fwd_fused(x, h_all, c_all, wp, bp, gates, True, 3), 200, 5)
            row = [f"unsplit {un * 1e3:7.1f}"]
            for S in sorted({2, 4, 8, 16, s_rule} - {1}):
                sp, _ = timeit(lambda: ops.lstm_cell_fwd_splitk(x[0], h_all[0], c_all[0], wp, bp, c_all[1], h_all[1], 3, S),
                               200, 5)
                row.append(f"S={S}{'*' if S == s_rule else ''} {sp * 1e3:7.1f} ({un / sp:4.2f}x)")
            wmb = wp.numel() * 2 / 1e6
            print(f"  cell   B={B} {H:2d}x{H:<2d} Ch={Ch:4d} (weights {wmb:6.1f} MB, S*={s_rule:2d}): " + "  ".join(row),
                  flush=True)
        for name, H, C0, C1, N in (("bottleneck.conv1", 4, 512, 0, 1024), ("bottleneck.conv2", 4, 1024, 0, 1024),
                                   ("up3.conv1", 8, 512, 512, 512), ("up3.conv2", 8, 512, 0, 512)):
            torch.manual_seed(0)
            w = torch.randn(N, C0 + C1, 3, 3, device=dev) * (1.0 / (9 * (C0 + C1)) ** 0.5)
            wp = ops.pack_conv_weight(w, torch.bfloat16)
            x0 = torch.randn(1, B, H, H, C0, device=dev).bfloat16()
            x1 = torch.randn(1, B, H, H, C1, device=dev).bfloat16() if C1 else None
            sc, sh = torch.rand(N, device=dev) + 0.5, torch.randn(N, device=dev)
            s_rule = lib.b200_splitk_splits(B, H, H, C0, C1, N, 3)
            un, _ = timeit(lambda: ops.conv_affine_relu(x0, x1, wp, sc, sh, 3), 200, 5)
            row = [f"unsplit {un * 1e3:7.1f}"]
            for S in sorted({2, 4, 8, 16, s_rule} - {1}):
                sp, _ = timeit(lambda: ops.conv_affine_relu_splitk(x0, x1, wp, sc, sh, 3, S), 200, 5)
                row.append(f"S={S}{'*' if S == s_rule else ''} {sp * 1e3:7.1f} ({un / sp:4.2f}x)")
            print(f"  conv   B={B} {name:16s} {H}x{H} K{C0 + C1:5d} N{N:5d} (S*={s_rule:2d}): " + "  ".join(row), flush=True)


if __name__ == "__main__":
    pkg.set_precision("bf16")
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    print(card(), flush=True)
    if "--stream" in sys.argv:
        T, S, b = ([int(v) for v in args[:3]] + [20, 64, 64][len(args[:3]):])[:3]
        streaming(T, S, b)
        kernel_ab()
    else:
        B, T, S, b = ([int(v) for v in args[:4]] + [256, 20, 64, 64][len(args[:4]):])[:4]
        whole_sequences(B, T, S, b)
    if _lib.lib().b200_device_error() != 0:
        raise RuntimeError("device watchdog flag set")
