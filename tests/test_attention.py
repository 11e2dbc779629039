"""SpatialAttention (TemporalUNetDualView(use_attention=True), reference unet.py:113-125) without a GPU.

A host-side dry run on CPU tensors: every C-ABI call a training step and a three-frame stream make is checked against its
prototype in include/b200_convlstm.h and skipped, with ATen's attention operators (conv2d, amax, sigmoid) patched to
raise, so the attention cannot quietly run on them.  Also the fp64 port of the model with attention that the GPU tests
(tests/test_gpu_attention.py) measure against (tests/attention_port.py), checked here against the reference's
nn.Module and against oracle/torch_port.py, and the refusal of kernel sizes the kernels do not have."""
import ctypes

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from attention_port import RefSpatialAttention, port_attention, temporal_unet


@pytest.fixture
def dry(monkeypatch):
    import train.unet as U
    from unet_convlstm_b200 import _lib, loss, ops, optim
    protos = _lib.parse_header()
    seen = {}

    def fake_call(name, *args, tag="", work=None, kernels=None):
        assert name in protos, f"{name} is not declared in include/b200_convlstm.h"
        _, argtypes = protos[name]
        assert len(args) == len(argtypes), (name, len(args), len(argtypes))
        for i, (a, t) in enumerate(zip(args, argtypes)):
            if t is ctypes.c_void_p:
                assert a is None or hasattr(a, "data_ptr") or isinstance(a, (int, ctypes.Array)), (name, i, type(a))
            elif t in (ctypes.c_int, ctypes.c_longlong):
                assert isinstance(a, int) and not isinstance(a, bool), (name, i, type(a), a)
            else:
                assert isinstance(a, (float, int)) and not isinstance(a, bool), (name, i, type(a))
        seen[name] = seen.get(name, 0) + 1
        if name.startswith("b200_spatial_attention"):
            seen.setdefault("attention_args", []).append(args)

    def aten_attention(*a, **k):
        raise AssertionError("an ATen operator of the attention was called")

    monkeypatch.setattr(_lib, "call", fake_call)
    monkeypatch.setattr(_lib, "supported", lambda name, *a: False)
    monkeypatch.setattr(ops, "_chk", lambda t, name="tensor": t)
    monkeypatch.setattr(ops, "_st", lambda: 0)
    monkeypatch.setattr(optim, "_st", lambda: 0)
    monkeypatch.setattr(optim, "_check", lambda ts, what: None)
    monkeypatch.setattr(ops, "copy_", lambda dst, src, accumulate=False: (dst.add_(src) if accumulate else dst.copy_(src)))
    monkeypatch.setattr(ops, "_pack_ok", lambda w, taps: w.dtype == torch.float32 and taps <= 9)
    monkeypatch.setattr(U, "_require_cuda", lambda *a, **k: None)
    monkeypatch.setattr(ops, "WGRAD_STREAM", False)
    if hasattr(loss, "_st"):
        monkeypatch.setattr(loss, "_st", lambda: 0)
    for mod, name in ((F, "conv2d"), (torch, "conv2d"), (torch, "amax"), (torch.Tensor, "amax"), (torch, "sigmoid"),
                      (torch.Tensor, "sigmoid"), (nn.Conv2d, "forward"), (nn.Sigmoid, "forward")):
        monkeypatch.setattr(mod, name, aten_attention)
    old = ops.get_precision()
    yield seen
    ops.set_precision(old)


def _model(**kw):
    from train.unet import TemporalUNetDualView
    torch.manual_seed(0)
    return TemporalUNetDualView(base_ch=16, use_skip_lstm=True, use_attention=True, **kw)


@pytest.mark.parametrize("precision", ["fp32", "bf16", "tf32"])
def test_training_step_and_stream_match_the_header(dry, precision):
    from unet_convlstm_b200 import ops, optim
    ops.set_precision(precision)
    m = _model()
    B, T, S = 2, 3, 32
    x = torch.randn(B, T, 2, S, S, requires_grad=True)
    opt = optim.AdamW(m.parameters(), lr=1e-3)
    for _ in range(2):
        out, _ = m(x)
        torch.stack(out, 1).sum().backward()
        w = m.attention.conv.weight
        assert w.grad is not None and w.grad.shape == (1, 2, 7, 7) and w.grad.dtype == torch.float32
        opt.step()
        opt.zero_grad(set_to_none=True)
    assert dry["b200_spatial_attention_fwd"] == 2 and dry["b200_spatial_attention_bwd"] == 2
    act = torch.float32 if precision != "bf16" else torch.bfloat16
    fwd, bwd = dry["attention_args"][0], dry["attention_args"][1]
    # fwd: x [T, B, h, w, 256] as the bottleneck left it (no permute, no cast), 7x7, the dtype flag of the mode
    assert fwd[0].shape == (T, B, S // 16, S // 16, 256) and fwd[0].dtype == act and fwd[0].is_contiguous()
    assert fwd[2:8] == (T * B, S // 16, S // 16, 256, 7, int(precision != "bf16"))
    assert fwd[1].data_ptr() == m.attention.conv.weight.data_ptr()
    assert bwd[13] is not None and bwd[13].shape == (1, 2, 7, 7)       # dw
    P = T * B * (S // 16) ** 2
    assert bwd[11].numel() == 2 * P + 2 * 49 * -(-P // 2048)            # the workspace the header asks for
    m.eval()
    s = m.stream()
    for t in range(3):
        assert s.step(torch.rand(B, 2, S, S)).shape == (B, 1, S, S)
    assert dry["b200_spatial_attention_fwd"] == 2 + 3 and dry["b200_spatial_attention_bwd"] == 2


def test_module_forward_goes_through_the_kernels(dry):
    from train.unet import SpatialAttention
    from unet_convlstm_b200 import ops
    ops.set_precision("bf16")
    for k in (1, 3, 5, 7):
        m = SpatialAttention(k)
        x = torch.randn(3, 20, 5, 3, requires_grad=True)
        y = m(x)
        assert y.shape == x.shape and y.dtype == torch.float32
        y.sum().backward()
        assert x.grad.shape == x.shape and m.conv.weight.grad.shape == (1, 2, k, k)
        args = dry["attention_args"][-1]
        assert args[5:11] == (3, 5, 3, 20, k, 0)


def test_no_attention_makes_no_attention_call(dry):
    from train.unet import TemporalUNetDualView
    torch.manual_seed(0)
    m = TemporalUNetDualView(base_ch=8, use_skip_lstm=True)
    assert not hasattr(m, "attention")
    out, _ = m(torch.randn(1, 2, 2, 32, 32))
    torch.stack(out, 1).sum().backward()
    assert not any(k.startswith("b200_spatial_attention") for k in dry)


@pytest.mark.parametrize("k", [2, 9])
def test_unsupported_kernel_sizes_raise(dry, k):
    from train.unet import SpatialAttention
    m = SpatialAttention(k)
    with pytest.raises(RuntimeError, match="not supported"):
        m(torch.randn(2, 16, 8, 8))
    assert "b200_spatial_attention_fwd" not in dry


def test_state_dict_and_initialisation_are_the_references():
    from train.unet import DoubleConv, Down, TemporalUNetDualView
    torch.manual_seed(4)
    m = TemporalUNetDualView(base_ch=8, use_attention=True)
    keys = [k for k in m.state_dict() if k.startswith("attention")]
    assert keys == ["attention.conv.weight"] and m.state_dict()[keys[0]].shape == (1, 2, 7, 7)
    # the weight draws from the RNG where the reference's does: after the encoder, as nn.Conv2d(2, 1, 7, padding=3,
    # bias=False)
    torch.manual_seed(4)
    DoubleConv(2, 8), Down(8, 16), Down(16, 32), Down(32, 64), Down(64, 128)
    assert torch.equal(RefSpatialAttention().conv.weight, m.attention.conv.weight)


@pytest.mark.parametrize("k", [1, 3, 7])
def test_port_attention_equals_the_reference_module_in_fp64(k):
    torch.manual_seed(k)
    ref = RefSpatialAttention(k).double()
    x = torch.relu(torch.randn(3, 24, 6, 5, dtype=torch.float64))
    x[0, :, 1, 1] = 0.0                               # a pixel whose channels are all tied at zero
    x[1, 3, 2, 2] = x[1, 5, 2, 2] = x[1, :, 2, 2].max() + 1   # two tied maxima
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    w = ref.conv.weight.detach().clone().requires_grad_(True)
    ya, yb = ref(xa), port_attention(w, xb)
    assert torch.equal(ya, yb)
    g = torch.randn_like(ya)
    (ya * g).sum().backward()
    (yb * g).sum().backward()
    assert torch.equal(xa.grad, xb.grad) and torch.equal(ref.conv.weight.grad, w.grad)


def test_port_with_attention_equals_the_model_structure_in_fp64():
    """The fp64 port applies the reference's module to the bottleneck output of every frame: the same outputs and
    gradients with RefSpatialAttention loaded from the state_dict in its place; without the attention weight it is
    oracle/torch_port.py's forward, bit for bit."""
    from oracle import torch_port as TP
    from train.unet import TemporalUNetDualView
    torch.manual_seed(2)
    m = TemporalUNetDualView(base_ch=4, use_skip_lstm=True, use_attention=True)
    sd = m.state_dict()
    x = torch.rand(2, 3, 2, 32, 32, dtype=torch.float64)
    ref_mod = RefSpatialAttention().double()
    ref_mod.conv.weight.data.copy_(sd["attention.conv.weight"])
    for training in (False, True):
        p = TP.params_from_state_dict(sd, torch.float64)
        out, st = temporal_unet(p, x, None, training=training, track=False)
        p2 = TP.params_from_state_dict(sd, torch.float64)
        ref_mod.conv.weight.data.copy_(p2["attention.conv.weight"])
        out2, st2 = temporal_unet(p2, x, None, training=training, track=False, attention=ref_mod)
        assert all(torch.equal(a, b) for a, b in zip(out, out2))
        assert torch.equal(st[0][0], st2[0][0]) and torch.equal(st[0][1], st2[0][1])
        torch.stack(out, 1).sum().backward()
        ref_mod.zero_grad()
        torch.stack(out2, 1).sum().backward()
        assert torch.equal(p["attention.conv.weight"].grad, ref_mod.conv.weight.grad)
        for k in p:
            if p[k].requires_grad and k != "attention.conv.weight":
                assert torch.equal(p[k].grad, p2[k].grad), k
    # without the attention weight: oracle/torch_port.py, bit for bit
    p = TP.params_from_state_dict(sd, torch.float64, requires_grad=False)
    out_att, _ = temporal_unet(p, x, None, training=False, track=False)
    p.pop("attention.conv.weight")
    out3, st3 = temporal_unet(p, x, None, training=False, track=False)
    out4, st4 = TP.temporal_unet(p, x, None, training=False, track=False)
    assert all(torch.equal(a, b) for a, b in zip(out3, out4))
    assert torch.equal(st3[0][0], st4[0][0]) and torch.equal(st3[0][1], st4[0][1])
    assert not all(torch.equal(a, b) for a, b in zip(out_att, out3))
