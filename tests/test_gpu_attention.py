"""SpatialAttention kernels (csrc/attention.cu) on the GPU, against fp64.

Op level: y, dx and dw of b200_spatial_attention_fwd / _bwd in the fp32, tf32 and bf16 modes at the benchmarks'
bottleneck shapes (T*B scaled down), ragged and 1x1 images, the scalar path (C = 20, C = 9) and k = 7 / 3, on post-ReLU
inputs with all-zero pixels and duplicated maxima (torch.amax's backward splits the gradient evenly among ties).  The
bf16 outputs are held to one bf16 ulp of the fp64 value on the same bf16 inputs; fp32 arithmetic to 1e-5.
Determinism over calls, streams and a CUDA-graph replay.  Model level: TemporalUNetDualView(use_attention=True)
against the fp64 port (tests/attention_port.py), GradReducer and loop.train_one_epoch, two optimizer steps, streaming inference, and a
profiler trace that shows the attention adds our kernels and nothing else."""
import collections

import pytest
import torch

from attention_port import port_attention, temporal_unet as port_temporal_unet

pytestmark = pytest.mark.gpu


@pytest.fixture
def precision():
    import unet_convlstm_b200 as pkg
    old = pkg.get_precision()
    yield pkg.set_precision
    pkg.set_precision(old)


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


def _rel2(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / max(float(b.norm()), 1e-30))


def _bf16_ulp(v):
    """One bf16 unit in the last place of each |v| (8 significant bits)."""
    mag = v.abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(mag)) - 7)


def _inputs(T, B, H, W, C, dtype, seed):
    """Post-ReLU x with an all-zero pixel and a pixel with two tied maxima per image, and a gradient dy."""
    g = torch.Generator().manual_seed(seed)
    x = torch.relu(torch.randn(T, B, H, W, C, generator=g))
    x[:, :, 0, 0, :] = 0.0
    if H * W > 1:
        py, px = (H - 1, W - 1)
        top = x[:, :, py, px, :].amax(-1, keepdim=True) + 0.5
        x[:, :, py, px, 0:1] = top
        x[:, :, py, px, C // 2:C // 2 + 1] = top
    dy = torch.randn(T, B, H, W, C, generator=g)
    return x.to(dtype).cuda(), dy.to(dtype).cuda()


def _fp64(x, dy, w):
    """fp64 y, dx, dw of the reference's formula on exactly the stored inputs (NHWC sequence -> NCHW images)."""
    T, B, H, W, C = x.shape
    xd = x.detach().double().cpu().reshape(T * B, H, W, C).permute(0, 3, 1, 2).requires_grad_(True)
    wd = w.detach().double().cpu().requires_grad_(True)
    y = port_attention(wd, xd)
    g = dy.double().cpu().reshape(T * B, H, W, C).permute(0, 3, 1, 2)
    (y * g).sum().backward()
    back = lambda t: t.permute(0, 2, 3, 1).reshape(T, B, H, W, C)  # noqa: E731
    return back(y.detach()), back(xd.grad), wd.grad


def _parent_aten(x, w):
    """The parent's path: permute to NCHW, fp32, ATen mean / amax / cat / cuDNN conv / sigmoid / mul, back, cast."""
    T, B, H, W, C = x.shape
    xf = x.reshape(T * B, H, W, C).permute(0, 3, 1, 2).float()
    pooled = torch.cat([xf.mean(dim=1, keepdim=True), xf.amax(dim=1, keepdim=True)], dim=1)
    a = xf * torch.sigmoid(torch.nn.functional.conv2d(pooled, w, padding=w.shape[-1] // 2))
    return a.permute(0, 2, 3, 1).reshape(T, B, H, W, C).to(x.dtype)


SHAPES = [  # (T, B, H, W, C, k)
    (2, 4, 4, 4, 1024, 7),     # configs[1] bottleneck [20, 256, 4, 4, 1024], T*B scaled down
    (2, 2, 8, 8, 1024, 7),     # configs[2] [10, 32, 8, 8, 1024]
    (2, 2, 16, 16, 2048, 7),   # configs[3] [16, 8, 16, 16, 2048]
    (1, 3, 5, 3, 64, 7),       # ragged image
    (2, 2, 1, 1, 64, 7),       # 1x1: only the centre tap
    (2, 2, 6, 6, 20, 7),       # C = 20: scalar path in bf16 (40 bytes a pixel)
    (2, 2, 6, 7, 9, 3),        # C = 9: scalar path in fp32 too
    (2, 3, 8, 8, 256, 3),      # k = 3
]


def _weight(k, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(1, 2, k, k, generator=g) * (2.0 / (2 * k * k)) ** 0.5).cuda()


@pytest.mark.parametrize("mode", ["fp32", "tf32", "bf16"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_op_against_fp64(precision, mode, shape):
    from unet_convlstm_b200 import ops
    precision(mode)
    T, B, H, W, C, k = shape
    act = ops.act_dtype()
    x, dy = _inputs(T, B, H, W, C, act, seed=C + k)
    w = _weight(k, seed=k)
    y, pooled, a = ops.spatial_attention_fwd(x, w)
    dx, dw = ops.spatial_attention_bwd(x, dy, w, pooled, a)
    torch.cuda.synchronize()
    y64, dx64, dw64 = _fp64(x, dy, w)
    if act == torch.float32:
        assert _rel(y, y64) < 1e-5, _rel(y, y64)
        assert _rel(dx, dx64) < 1e-5, _rel(dx, dx64)
    else:
        # one bf16 rounding of the fp32 result: within one ulp of the fp64 value (exact zeros stay exact)
        assert ((y.double().cpu() - y64).abs() <= _bf16_ulp(y64)).all(), float(((y.double().cpu() - y64).abs() / _bf16_ulp(y64)).max())
        # dx sums three fp32 terms before its rounding: one ulp of the value, plus the fp32 sums' 2^-20 of the largest
        err = (dx.double().cpu() - dx64).abs()
        assert (err <= _bf16_ulp(dx64) + 2.0 ** -20 * dx64.abs().max()).all(), float((err / _bf16_ulp(dx64)).max())
        ref = _parent_aten(x, w)
        assert ((y.double() - ref.double()).abs().cpu() <= _bf16_ulp(ref.double().cpu())).all()
    assert _rel(dw, dw64) < 1e-5, _rel(dw, dw64)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_ties_split_the_max_gradient_evenly(precision, mode):
    """Post-ReLU input where most channels of many pixels are zero: all-zero pixels (every channel tied) and pixels with
    2 and 3 equal maxima.  dx against fp64 torch.amax backward, at the tied pixels."""
    from unet_convlstm_b200 import ops
    precision(mode)
    act = ops.act_dtype()
    T, B, H, W, C = 2, 2, 6, 6, 64
    g = torch.Generator().manual_seed(5)
    x = torch.relu(torch.randn(T, B, H, W, C, generator=g) - 1.5)     # ~93 % zeros
    x[:, :, 0:3, :, :] = 0.0                                         # whole rows of all-zero pixels
    x[:, :, 4, 1, 3] = x[:, :, 4, 1, 40] = 3.0
    x[:, :, 4, 2, 7] = x[:, :, 4, 2, 8] = x[:, :, 4, 2, 63] = 4.0
    x, dy = x.to(act).cuda(), torch.randn(T, B, H, W, C, generator=g).to(act).cuda()
    w = _weight(7, seed=1)
    y, pooled, a = ops.spatial_attention_fwd(x, w)
    dx, dw = ops.spatial_attention_bwd(x, dy, w, pooled, a)
    _, dx64, dw64 = _fp64(x, dy, w)
    tied = [(slice(None), slice(None), slice(0, 3)), (slice(None), slice(None), 4, 1), (slice(None), slice(None), 4, 2)]
    for s in tied:
        got, ref = dx[s].double().cpu(), dx64[s]
        if act == torch.float32:
            assert float((got - ref).abs().max()) <= 1e-5 * float(dx64.abs().max()), s
        else:
            assert ((got - ref).abs() <= _bf16_ulp(ref) + 2.0 ** -20 * dx64.abs().max()).all(), s
    assert _rel(dw, dw64) < 1e-5


def _run_op(x, dy, w):
    from unet_convlstm_b200 import ops
    y, pooled, a = ops.spatial_attention_fwd(x, w)
    dx, dw = ops.spatial_attention_bwd(x, dy, w, pooled, a)
    return y, dx, dw


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_deterministic_over_calls_streams_and_graph_replay(precision, mode):
    from unet_convlstm_b200 import ops
    precision(mode)
    x, dy = _inputs(4, 8, 8, 8, 1024, ops.act_dtype(), seed=9)
    w = _weight(7, seed=2)
    ref = _run_op(x, dy, w)
    for _ in range(2):
        assert all(torch.equal(a, b) for a, b in zip(_run_op(x, dy, w), ref))
    # on a side stream while a large matrix product runs on the current one
    big = torch.randn(8192, 8192, device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    big @ big
    with torch.cuda.stream(side):
        got = _run_op(x, dy, w)
    torch.cuda.current_stream().wait_stream(side)
    assert all(torch.equal(a, b) for a, b in zip(got, ref))
    # captured into a CUDA graph and replayed
    cs = torch.cuda.Stream()
    cs.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(cs):
        _run_op(x, dy, w)
    torch.cuda.current_stream().wait_stream(cs)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=cs):
        out = _run_op(x, dy, w)
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(out, ref))


def _model(base_ch=16, seed=0, **kw):
    from train.unet import TemporalUNetDualView
    torch.manual_seed(seed)
    m = TemporalUNetDualView(base_ch=base_ch, use_skip_lstm=True, use_attention=True, **kw)
    g = torch.Generator().manual_seed(seed + 1)
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.running_mean.copy_(0.05 * torch.randn(mod.num_features, generator=g))
            mod.running_var.copy_(0.5 + torch.rand(mod.num_features, generator=g))
    return m


def _port(sd, x, dy, dtype, training):
    from oracle import torch_port as TP
    p = TP.params_from_state_dict(sd, dtype)
    xt = x.to(dtype).requires_grad_(True)
    out, _ = port_temporal_unet(p, xt, None, training=training, track=False)
    y = torch.stack(out, dim=1)
    (y * dy.to(dtype)).sum().backward()
    r = {"y": y.detach(), "dx": xt.grad}
    r.update({"g." + k: v.grad for k, v in p.items() if v.requires_grad})
    return r


@pytest.mark.parametrize("training", [False, True])
def test_model_fp32_against_the_fp64_port(precision, training):
    """fp32 check mode: eval-mode y within 1e-5; train mode, every gradient (attention.conv.weight included) within
    max(1e-5, 4 x the port's own fp32 error) max-relative, the criterion of the use_attention=False model tests."""
    precision("fp32")
    B, T, S = 2, 3, 32
    m = _model()
    g = torch.Generator().manual_seed(3)
    x, dy = torch.rand(B, T, 2, S, S, generator=g), torch.randn(B, T, 1, S, S, generator=g)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    ref = _port(sd, x, dy, torch.float64, training)
    m = m.cuda().train(training)
    xg = x.cuda().requires_grad_(True)
    y = torch.stack(m(xg)[0], dim=1)
    (y * dy.cuda()).sum().backward()
    got = {"y": y, "dx": xg.grad}
    got.update({"g." + k: p.grad for k, p in m.named_parameters()})
    assert got["g.attention.conv.weight"] is not None
    if not training:
        assert _rel(got["y"], ref["y"]) < 1e-5, _rel(got["y"], ref["y"])
        return
    r32 = _port(sd, x, dy, torch.float32, training)
    zero_scale = float(dy.abs().max()) * 100
    bad = []
    for k, v in ref.items():
        if float(v.abs().max()) < 1e-7 * zero_scale:
            # mathematically zero (conv bias feeding a train-mode BatchNorm): absolute comparison, as
            # tests/test_gpu_parity.py::_check_grads does
            if not float(got[k].abs().max()) < 10 * 1e-5 * zero_scale:
                bad.append((k, "zero", float(got[k].abs().max())))
            continue
        floor = _rel(r32[k], v)
        if not _rel(got[k], v) < max(1e-5, 4 * floor):
            bad.append((k, _rel(got[k], v), floor))
    assert not bad, bad


def test_grad_reducer_and_train_one_epoch_take_the_attention_path(precision):
    """GradReducer (single process: its bucketing and hooks, with the background weight-gradient stream on) leaves every
    gradient of an attention model bit-identical to a plain backward, and loop.train_one_epoch trains the model like
    the reference's loop restated step by step, the attention weight included."""
    import copy
    import types
    from unet_convlstm_b200 import _lib, loop, ops
    from unet_convlstm_b200.dist import GradReducer
    from unet_convlstm_b200.loss import compute_loss
    precision("fp32")
    m1 = _model(base_ch=8, seed=12).cuda()
    m2 = copy.deepcopy(m1)
    g = torch.Generator().manual_seed(13)
    x = torch.rand(2, 3, 2, 32, 32, generator=g).cuda()
    dy = torch.randn(2, 3, 1, 32, 32, generator=g).cuda()
    bg = ops.WGRAD_STREAM
    ops.enable_background_wgrad()
    try:
        red = GradReducer(m1.parameters())
        for _ in range(2):
            m1.zero_grad(set_to_none=True), m2.zero_grad(set_to_none=True)
            calls = _lib.CALLS.get("b200_spatial_attention_bwd", 0)
            (torch.stack(m1(x)[0], dim=1) * dy).sum().backward()
            red.finish()
            assert _lib.CALLS["b200_spatial_attention_bwd"] == calls + 1
            (torch.stack(m2(x)[0], dim=1) * dy).sum().backward()
            for (k, a), b in zip(m1.named_parameters(), m2.parameters()):
                assert torch.equal(a.grad, b.grad), k
        m1 = _model(base_ch=8, seed=14).cuda()
        m2 = copy.deepcopy(m1)
        batches = []
        for b in (3, 2):
            xb = torch.rand(b, 3, 2, 32, 32, generator=g) * 2
            yb = torch.clamp(torch.randn(b, 3, 1, 32, 32, generator=g), -1, 1)
            batches.append((xb, yb, (xb[:, :, 0:1] > 1.1).float()))
        ds = types.SimpleNamespace(trans_min=-1.05, trans_max=1.17, y_scale=6.0, y_transform="asinh")
        o1 = torch.optim.AdamW(m1.parameters(), lr=1e-3)
        o2 = torch.optim.AdamW(m2.parameters(), lr=1e-3)
        w0 = m1.attention.conv.weight.detach().clone()
        got = loop.train_one_epoch(m1, batches, o1, "cuda", ds)
        m2.train()
        tot, n = 0.0, 0
        for xb, yb, mb in batches:
            xb, yb, mb = xb.cuda(), yb.cuda(), mb.cuda()
            o2.zero_grad(set_to_none=True)
            loss = compute_loss(torch.stack(m2(xb)[0], dim=1), yb, mb, True)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(m2.parameters(), 1.0)
            o2.step()
            tot += loss.item() * xb.size(0)
            n += xb.size(0)
        assert abs(got[0] - tot / n) <= 2e-4 * abs(tot / n), (got[0], tot / n)
        assert not torch.equal(m1.attention.conv.weight, w0)
        for (k, a), b in zip(m1.state_dict().items(), m2.state_dict().values()):
            assert _rel2(a.float(), b.float()) < 1e-3, k
    finally:
        ops.WGRAD_STREAM = bg


def test_model_bf16_against_the_fp64_port(precision):
    precision("bf16")
    B, T, S = 2, 3, 64
    m = _model()
    g = torch.Generator().manual_seed(4)
    x = torch.rand(B, T, 2, S, S, generator=g)
    from oracle import torch_port as TP
    p = TP.params_from_state_dict(m.state_dict(), torch.float64, requires_grad=False)
    out64, _ = port_temporal_unet(p, x.double(), None, training=False, track=False)
    m = m.cuda().eval()
    with torch.no_grad():
        y = torch.stack(m(x.cuda())[0], dim=1)
    assert _rel2(y, torch.stack(out64, dim=1)) < 2e-2


def test_two_optimizer_steps_equal_a_fresh_model(precision):
    import copy
    from unet_convlstm_b200 import optim
    precision("bf16")
    m = _model(seed=8).cuda()
    fresh = _model(seed=99).cuda()
    g = torch.Generator(device="cuda").manual_seed(2)
    x = torch.rand(2, 3, 2, 32, 32, device="cuda", generator=g) * 2
    dy = torch.randn(2, 3, 1, 32, 32, device="cuda", generator=g)
    opt = optim.AdamW(m.parameters(), lr=3e-2)
    w0 = m.attention.conv.weight.detach().clone()
    m.train()
    for _ in range(2):
        opt.zero_grad(set_to_none=True)
        (torch.stack(m(x)[0], dim=1) * dy).sum().backward()
        opt.step()
    assert not torch.equal(m.attention.conv.weight, w0)
    fresh.load_state_dict(copy.deepcopy(m.state_dict()))
    m.eval(), fresh.eval()
    with torch.no_grad():
        assert torch.equal(torch.stack(m(x)[0], dim=1), torch.stack(fresh(x)[0], dim=1))
    m.train(), fresh.train()
    m.zero_grad(set_to_none=True)
    a, b = torch.stack(m(x)[0], dim=1), torch.stack(fresh(x)[0], dim=1)
    assert torch.equal(a, b)
    (a * dy).sum().backward()
    (b * dy).sum().backward()
    assert torch.equal(m.attention.conv.weight.grad, fresh.attention.conv.weight.grad)


@pytest.mark.parametrize("mode,tol", [("fp32", 0.0), ("tf32", 1e-5), ("bf16", 1e-2)])
def test_stream_equals_the_sequence(precision, mode, tol):
    precision(mode)
    m = _model().cuda().eval()
    T = 5
    x = torch.rand(2, T, 2, 64, 64, generator=torch.Generator().manual_seed(6)).cuda()
    with torch.no_grad():
        ref, ref_state = m(x)
    s = m.stream()
    ys = [s.step(x[:, t]) for t in range(T)]
    for t in range(T):
        if tol == 0.0:
            assert torch.equal(ys[t], ref[t]), t
        else:
            assert _rel2(ys[t], ref[t]) < tol, (t, _rel2(ys[t], ref[t]))
    for a, b in zip(s.state[0], ref_state[0]):
        assert torch.equal(a, b) if tol == 0.0 else _rel2(a, b) < tol


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return collections.Counter(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                               and not e.name.startswith(("Memset", "Memcpy", "[memset]", "[memcpy]")))


def trace_kernels(mode):
    """{use_attention: (kernels of one training step, kernels of one stream frame)} for a base_ch-16 model, by name."""
    import unet_convlstm_b200 as pkg
    from train.unet import TemporalUNetDualView
    pkg.set_precision(mode)
    g = torch.Generator().manual_seed(7)
    x = torch.rand(2, 3, 2, 32, 32, generator=g).cuda()
    dy = torch.randn(2, 3, 1, 32, 32, generator=g).cuda()
    counts = {}
    for att in (False, True):
        torch.manual_seed(0)
        m = TemporalUNetDualView(base_ch=16, use_skip_lstm=True, use_attention=att).cuda()

        def step():
            m.zero_grad(set_to_none=True)      # gradients stored, not accumulated (an accumulation is an ATen add)
            (torch.stack(m(x)[0], dim=1) * dy).sum().backward()

        step()                                  # warm-up: weight packing, workspaces
        train = _kernels(step)
        m.eval()
        s = m.stream()
        with torch.no_grad():
            s.step(x[:, 0])
        frame = _kernels(lambda: s.step(x[:, 1]))
        counts[att] = (train, frame)
    return counts


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_attention_adds_only_its_own_kernels(mode):
    """The trace is taken in a child process: a profiler session leaves CUPTI state behind in the process, and the
    sessions of later test modules (tests/test_gpu_wgrad.py) then record no kernels."""
    import json
    import os
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    code = ("import json, sys; sys.path[:0] = [sys.argv[1], sys.argv[2]]; import test_gpu_attention as t; "
            "c = t.trace_kernels(sys.argv[3]); "
            "print(json.dumps({str(k): [dict(v[0]), dict(v[1])] for k, v in c.items()}))")
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", code, os.path.dirname(here), here, mode], capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    raw = json.loads(r.stdout.strip().splitlines()[-1])
    counts = {att: tuple(collections.Counter(d) for d in raw[str(att)]) for att in (False, True)}
    for i, what in enumerate(("training step", "stream frame")):
        extra = counts[True][i] - counts[False][i]
        missing = counts[False][i] - counts[True][i]
        assert not missing, (what, missing)
        names = sorted(extra)
        assert all("attn_" in n or "splitk_reduce_kernel" in n for n in names), (what, names)
        want = ({"attn_pool_kernel": 1, "attn_apply_kernel": 1, "attn_bwd_reduce_kernel": 1, "attn_bwd_dx_kernel": 1,
                 "attn_wgrad_kernel": 1, "splitk_reduce_kernel": 1} if i == 0 else
                {"attn_pool_kernel": 1, "attn_apply_kernel": 1})
        got = collections.Counter()
        for n, c in extra.items():
            got[next(k for k in want if k in n)] += c
        assert dict(got) == want, (what, dict(extra))
