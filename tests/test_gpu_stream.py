"""Streaming inference on the GPU (TemporalUNetDualView.stream, unet_convlstm_b200/stream.py): frame by frame with every
ConvLSTM state carried, against model(x) of the whole sequence (eval mode, no_grad) and the fp64 port; the split-K
kernels against the unsplit ones on identical operands; determinism; the refusal after a weight change."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def rel2(a, b):
    a = a.detach().double().cpu().numpy()
    b = b.detach().double().cpu().numpy()
    return float(np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-30))


@pytest.fixture
def precision():
    import unet_convlstm_b200 as pkg
    old = pkg.get_precision()
    yield pkg.set_precision
    pkg.set_precision(old)


def _model(base_ch, seed=0):
    from train.unet import TemporalUNetDualView
    torch.manual_seed(seed)
    m = TemporalUNetDualView(base_ch=base_ch, use_skip_lstm=True)
    g = torch.Generator().manual_seed(seed + 1)
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):      # non-trivial folded BatchNorm
            mod.running_mean.copy_(0.05 * torch.randn(mod.num_features, generator=g))
            mod.running_var.copy_(0.5 + torch.rand(mod.num_features, generator=g))
    return m.cuda().eval()


def _stream(m, x, state=None):
    s = m.stream(state)
    ys = [s.step(x[:, t]) for t in range(x.shape[1])]
    return ys, s.state


def _inputs(B, T, H, W, seed=3):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(B, T, 2, H, W, generator=g).cuda()


@pytest.mark.parametrize("with_state", [False, True])
def test_fp32_stream_is_bit_identical_to_the_sequence(precision, with_state):
    precision("fp32")
    m = _model(16)
    x = _inputs(2, 6, 32, 32)
    state = None
    if with_state:
        g = torch.Generator().manual_seed(9)
        state = [(0.5 * torch.randn(2, 256, 2, 2, generator=g).cuda(), torch.randn(2, 256, 2, 2, generator=g).cuda())]
    with torch.no_grad():
        ref, ref_state = m(x, state)
    ys, st = _stream(m, x, state)
    for t in range(6):
        assert torch.equal(ys[t], ref[t]), t
    assert torch.equal(st[0][0], ref_state[0][0]) and torch.equal(st[0][1], ref_state[0][1])


@pytest.mark.parametrize("B,H,W", [(1, 64, 64), (4, 40, 28)])
def test_bf16_stream_against_the_sequence_and_fp64(precision, B, H, W):
    from oracle import torch_port as TP
    precision("bf16")
    m = _model(64 if B == 1 else 16)
    T = 5
    x = _inputs(B, T, H, W)
    with torch.no_grad():
        ref, ref_state = m(x)
    ys, st = _stream(m, x)
    for t in range(T):
        assert rel2(ys[t], ref[t]) < 1e-2, (t, rel2(ys[t], ref[t]))
    for a, b in zip(st[0], ref_state[0]):
        assert rel2(a, b) < 1e-2
    p = TP.params_from_state_dict({k: v.cpu() for k, v in m.state_dict().items()}, torch.float64, requires_grad=False)
    out64, _ = TP.temporal_unet(p, x.cpu().double(), None, training=False, track=False)
    y = torch.stack(ys, 1)
    assert rel2(y, torch.stack(out64, 1)) < 2e-2


def test_tf32_stream_against_the_sequence(precision):
    precision("tf32")
    m = _model(16)
    x = _inputs(2, 4, 64, 64)
    with torch.no_grad():
        ref, ref_state = m(x)
    ys, st = _stream(m, x)
    for t in range(4):
        assert rel2(ys[t], ref[t]) < 1e-5, t
    assert rel2(st[0][1], ref_state[0][1]) < 1e-5


def _bf16_ulps(a, ref):
    """Per-element |a - ref| in bf16 units in the last place of max(|ref|, 2^-8).  The floor: a value near zero is the
    result of a cancellation (c = f*c + i*g, conv * scale + shift), whose fp32 summation-order noise from the split
    partial sums is an absolute error of the operands' scale, not of the small result."""
    ref = ref.float()
    mag = ref.abs().clamp_min(2.0 ** -8)
    ulp = torch.exp2(torch.floor(torch.log2(mag)) - 7)
    return ((a.float() - ref).abs() / ulp).max().item()


@pytest.mark.parametrize("B", [1, 8])
@pytest.mark.parametrize("H,Ch", [(4, 1024), (8, 512), (16, 256)])
def test_splitk_cell_against_the_fused_cell(precision, B, H, Ch):
    from unet_convlstm_b200 import ops
    precision("bf16")
    torch.manual_seed(5)
    w = (torch.randn(4 * Ch, 2 * Ch, 3, 3) * (1.0 / (18 * Ch) ** 0.5)).cuda()
    b = (0.1 * torch.randn(4 * Ch)).cuda()
    wp, bp = ops.pack_lstm_weight(w, b, torch.bfloat16)
    x = torch.randn(B, H, H, Ch).cuda().bfloat16()
    h = torch.randn(B, H, H, Ch).cuda().bfloat16()
    c = torch.randn(B, H, H, Ch).cuda()
    for h_prev, c_prev in ((h, c), (None, None)):
        cu, hu = torch.empty_like(c), torch.empty_like(h)
        ops.lstm_cell_fwd_fused(x, h_prev, c_prev, wp, bp, cu, hu, None, 3)
        for splits in (2, 7):
            cs, hs = torch.empty_like(c), torch.empty_like(h)
            ops.lstm_cell_fwd_splitk(x, h_prev, c_prev, wp, bp, cs, hs, 3, splits)
            assert rel2(cs, cu) <= 1e-5, (splits, rel2(cs, cu))
            assert _bf16_ulps(hs, hu) <= 1, (splits, _bf16_ulps(hs, hu))


@pytest.mark.parametrize("B", [1, 8])
@pytest.mark.parametrize("H,C0,C1,N", [(4, 512, 0, 1024), (4, 1024, 0, 1024), (8, 512, 512, 512), (8, 512, 0, 512)])
def test_splitk_conv_against_the_unsplit_conv(precision, B, H, C0, C1, N):
    from unet_convlstm_b200 import ops
    precision("bf16")
    torch.manual_seed(6)
    K = C0 + C1
    w = (torch.randn(N, K, 3, 3) * (1.0 / (9 * K) ** 0.5)).cuda()
    wp = ops.pack_conv_weight(w, torch.bfloat16)
    x0 = torch.randn(1, B, H, H, C0).cuda().bfloat16()
    x1 = torch.randn(1, B, H, H, C1).cuda().bfloat16() if C1 else None
    bias = (0.1 * torch.randn(N)).cuda()
    scale = (0.5 + torch.rand(N)).cuda()
    ref32 = torch.empty(1, B, H, H, N, device="cuda")
    ops.conv_fwd(x0, x1, wp, None, 3, ref32)
    ref = ops.conv_affine_relu(x0, x1, wp, scale, bias, 3)
    for splits in (2, 9):
        # the partial sums reduced in split order: summation order only
        z = ops.conv_affine_relu_splitk(x0, x1, wp, None, None, 3, splits, relu=False, out_fp32=True)
        assert rel2(z, ref32) <= 1e-5, (splits, rel2(z, ref32))
        y = ops.conv_affine_relu_splitk(x0, x1, wp, scale, bias, 3, splits)
        assert _bf16_ulps(y, ref) <= 1, (splits, _bf16_ulps(y, ref))


def test_two_streams_are_bit_identical(precision):
    precision("bf16")
    m = _model(64)
    x = _inputs(1, 6, 64, 64)
    ys1, st1 = _stream(m, x)
    s = m.stream()
    ys2 = [s.step(x[:, t]) for t in range(6)]
    st2 = s.state
    for a, b in zip(ys1, ys2):
        assert torch.equal(a, b)
    assert torch.equal(st1[0][0], st2[0][0]) and torch.equal(st1[0][1], st2[0][1])
    # a new sequence on the same stream keeps the captured graph: frames 1.. are replays, same results
    s.reset()
    ys3 = [s.step(x[:, t]) for t in range(6)]
    for a, b in zip(ys1, ys3):
        assert torch.equal(a, b)
    assert torch.equal(st1[0][1], s.state[0][1])


def test_weight_change_refused_until_reset(precision):
    precision("fp32")
    m = _model(8)
    x = _inputs(2, 5, 32, 32)
    s = m.stream()
    for t in range(3):
        s.step(x[:, t])
    m.load_state_dict(_model(8, seed=4).state_dict())
    with pytest.raises(RuntimeError, match="changed since this stream bound it"):
        s.step(x[:, 3])
    s.reset()
    ys = [s.step(x[:, t]) for t in range(5)]
    with torch.no_grad():
        ref, _ = m(x)
    for t in range(5):
        assert torch.equal(ys[t], ref[t]), t
