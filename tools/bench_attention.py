"""SpatialAttention (TemporalUNetDualView(use_attention=True)) on the B200: kernel time, achieved bandwidth and
training throughput, one GPU command.

    python tools/bench_attention.py --out profiles/attention_b200.txt

1. Kernel time, forward + backward, at the bottleneck shapes of the benchmark configurations in bf16
   (configs[1] [20, 256, 4, 4, 1024], configs[2] [10, 32, 8, 8, 1024], configs[3] [16, 8, 16, 16, 2048]):
   b200_spatial_attention_fwd + _bwd against the previous ATen path (permute to NCHW, fp32, mean / amax / cat, cuDNN
   7x7 convolution, sigmoid, mul, permute back, cast; backward by autograd), alternated in rounds, CUDA events over
   many launches.  x of configs[1] (168 MB) and configs[3] (134 MB) exceed the 126 MB L2; configs[2] (42 MB) fits, so
   its back-to-back launches read partly from L2.
2. Achieved bandwidth: algorithmic bytes over kernel time, against the data sheet's 7.7 TB/s.  Forward reads x and
   writes y once; backward reads dy and x and writes dx once.  (The kernels read x twice forward and x, dy twice
   backward; those extra passes count as time, not as bytes.)
3. Training throughput, sequences/s: the bench.py step (forward, compute_loss, backward, clipped AdamW) at configs[1]
   (64x64, T = 20, batch 256, base_ch 64, skip ConvLSTMs) for use_attention False and True, alternated.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

SHAPES = {"configs[1]": (20, 256, 4, 4, 1024), "configs[2]": (10, 32, 8, 8, 1024), "configs[3]": (16, 8, 16, 16, 2048)}
PEAK_TBS = 7.7


def algorithmic_bytes(shape, esize=2):
    n = 1
    for d in shape:
        n *= d
    return 2 * n * esize, 3 * n * esize      # forward (x, y), backward (dy, x, dx)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name()


def ours(x, w, dy):
    from unet_convlstm_b200 import ops
    y, pooled, a = ops.spatial_attention_fwd(x, w)
    dx, dw = ops.spatial_attention_bwd(x, dy, w, pooled, a)
    return y, dx, dw


def aten(x, w, dy):
    """The previous path of train/unet.py (_encode + the nn.Module SpatialAttention), forward and autograd backward."""
    T, B, H, W, C = x.shape
    xr = x.detach().requires_grad_(True)
    wr = w.detach().requires_grad_(True)
    xf = xr.reshape(T * B, H, W, C).permute(0, 3, 1, 2).float()
    pooled = torch.cat([xf.mean(dim=1, keepdim=True), xf.amax(dim=1, keepdim=True)], dim=1)
    a = xf * torch.sigmoid(torch.nn.functional.conv2d(pooled, wr, padding=w.shape[-1] // 2))
    y = a.permute(0, 2, 3, 1).reshape(T, B, H, W, C).to(x.dtype).contiguous()
    y.backward(dy)
    return y, xr.grad, wr.grad


def time_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def graphed(fn, calls=10):
    """A CUDA graph of `calls` back-to-back calls of fn (warmed up on the capture stream first)."""
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        fn()
    torch.cuda.current_stream().wait_stream(st)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        for _ in range(calls):
            fn()
    return g


def kernel_section(lines, rounds, iters):
    import unet_convlstm_b200 as pkg
    pkg.set_precision("bf16")
    lines.append("## 1-2. Kernel time (forward + backward) and achieved bandwidth, bf16, k = 7")
    lines.append(f"CUDA events around {iters} back-to-back fwd+bwd calls, {rounds} rounds alternating ours / ATen; "
                 "min and max over rounds.")
    for name, shape in SHAPES.items():
        g = torch.Generator(device="cuda").manual_seed(0)
        x = torch.relu(torch.randn(shape, device="cuda", generator=g)).bfloat16()
        dy = torch.randn(shape, device="cuda", generator=g).bfloat16()
        w = (torch.randn(1, 2, 7, 7, device="cuda", generator=g) * 0.1)
        from unet_convlstm_b200 import ops
        # forward alone and backward alone for the bandwidth split
        y, pooled, a = ops.spatial_attention_fwd(x, w)
        ours(x, w, dy), aten(x, w, dy)                       # warm-up (cuDNN algorithm choice, module load)
        t_o, t_a, t_f, t_b = [], [], [], []
        for _ in range(rounds):
            t_o.append(time_ms(lambda: ours(x, w, dy), iters))
            t_a.append(time_ms(lambda: aten(x, w, dy), iters))
            t_f.append(time_ms(lambda: ops.spatial_attention_fwd(x, w), iters))
            t_b.append(time_ms(lambda: ops.spatial_attention_bwd(x, dy, w, pooled, a), iters))
        # the same calls replayed from CUDA graphs (10 calls per graph): no host-side work between the kernels
        g_fb, g_f = graphed(lambda: ours(x, w, dy)), graphed(lambda: ops.spatial_attention_fwd(x, w))
        tg_fb = min(time_ms(g_fb.replay, max(1, iters // 10)) / 10 for _ in range(rounds))
        tg_f = min(time_ms(g_f.replay, max(1, iters // 10)) / 10 for _ in range(rounds))
        del g_fb, g_f
        yo, dxo, dwo = ours(x, w, dy)
        ya, dxa, dwa = aten(x, w, dy)
        diff_y = float((yo.float() - ya.float()).abs().max())
        bf, bb = algorithmic_bytes(shape)
        mb = bf / 2 / 1e6
        lines.append(f"\n{name} x {list(shape)} bf16 ({mb:.0f} MB)")
        lines.append(f"  ours fwd+bwd   {min(t_o) * 1e3:8.1f} - {max(t_o) * 1e3:8.1f} us")
        lines.append(f"  ATen fwd+bwd   {min(t_a) * 1e3:8.1f} - {max(t_a) * 1e3:8.1f} us   "
                     f"(ours {min(t_a) / min(t_o):.1f}x faster, best against best)")
        lines.append(f"  ours fwd       {min(t_f) * 1e3:8.1f} us   {bf / (min(t_f) * 1e-3) / 1e12:5.2f} TB/s algorithmic "
                     f"= {100 * bf / (min(t_f) * 1e-3) / 1e12 / PEAK_TBS:4.1f} % of {PEAK_TBS} TB/s")
        lines.append(f"  ours bwd       {min(t_b) * 1e3:8.1f} us   {bb / (min(t_b) * 1e-3) / 1e12:5.2f} TB/s algorithmic "
                     f"= {100 * bb / (min(t_b) * 1e-3) / 1e12 / PEAK_TBS:4.1f} % of {PEAK_TBS} TB/s")
        lines.append(f"  ours fwd+bwd   {(bf + bb) / (min(t_o) * 1e-3) / 1e12:5.2f} TB/s algorithmic")
        lines.append(f"  from CUDA graphs (no host work between calls): fwd+bwd {tg_fb * 1e3:.1f} us, fwd {tg_f * 1e3:.1f} us "
                     f"= {bf / (tg_f * 1e-3) / 1e12:.2f} TB/s, bwd (difference) {(tg_fb - tg_f) * 1e3:.1f} us "
                     f"= {bb / ((tg_fb - tg_f) * 1e-3) / 1e12:.2f} TB/s algorithmic")
        lines.append(f"  max |y_ours - y_ATen| = {diff_y:.3g}; dw rel diff "
                     f"{float((dwo - dwa).abs().max() / dwa.abs().max()):.2e}")
        del x, dy, y, pooled, a, yo, dxo, ya, dxa
        torch.cuda.empty_cache()


def training_section(lines, steps, warmup, rounds):
    import bench
    import unet_convlstm_b200 as pkg
    from train.unet import TemporalUNetDualView
    from unet_convlstm_b200 import ops
    from unet_convlstm_b200.loss import compute_loss
    from unet_convlstm_b200.optim import AdamW
    pkg.set_precision("bf16")
    ops.enable_background_wgrad()
    B, T, S = 256, 20, 64
    xh, yh, mh = bench.make_batch(B, T, S, 1234)
    x, y, m = xh.cuda(), yh.cuda(), mh.cuda()
    arms = {}
    for att in (False, True):
        torch.manual_seed(0)
        model = TemporalUNetDualView(base_ch=64, use_skip_lstm=True, use_attention=att).cuda().train()
        opt = AdamW(model.parameters(), lr=1e-3, weight_decay=1e-4)

        def step(model=model, opt=opt):
            opt.zero_grad(set_to_none=True)
            out, _ = model(x)
            compute_loss(torch.stack(out, dim=1), y, m).backward()
            opt.step(clip_max_norm=1.0)

        for _ in range(warmup):
            step()
        arms[att] = step
    torch.cuda.synchronize()
    res = {False: [], True: []}
    for _ in range(rounds):
        for att in (False, True):
            res[att].append(B * steps / (time_ms(arms[att], steps) * steps / 1e3))
    lines.append("\n## 3. Training throughput, bench.py step at configs[1] (64x64, T = 20, batch 256, base_ch 64, skip "
                 "ConvLSTMs, bf16)")
    lines.append(f"{steps} timed steps after {warmup} warm-up steps per arm, {rounds} rounds alternating.")
    for att in (False, True):
        lines.append(f"  use_attention={att!s:5}  " + "  ".join(f"{v:7.1f}" for v in res[att]) + "  sequences/s")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--train-rounds", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("bench_attention.py needs a CUDA device")
    from unet_convlstm_b200 import _lib
    _lib.lib()
    lines = [f"# SpatialAttention on {card()} (name, power limit, max SM clock)",
             f"torch {torch.__version__}, torch.backends.cudnn.allow_tf32 = {torch.backends.cudnn.allow_tf32} "
             "(the ATen path's convolution runs in TF32, as it did in the model)"]
    kernel_section(lines, args.rounds, args.iters)
    training_section(lines, args.steps, args.warmup, args.train_rounds)
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
