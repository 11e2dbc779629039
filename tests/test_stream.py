"""Host-side dry run of streaming inference (TemporalUNetDualView.stream) on CPU tensors: no GPU, no kernels.  Every C-ABI
call the stream makes is checked against its prototype in include/b200_convlstm.h and skipped, with the tensor-core
routes reported as available so that the split-K routing of the bf16 mode is exercised with the library's own
selection rule (b200_splitk_splits).  Also the refusals: training mode, a changed frame, a changed parameter."""
import ctypes

import pytest
import torch


@pytest.fixture
def dry(monkeypatch):
    import train.unet as U
    from unet_convlstm_b200 import _lib, ops
    protos = _lib.parse_header()
    seen = {}

    def fake_call(name, *args, tag="", work=None):
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

    monkeypatch.setattr(_lib, "call", fake_call)
    monkeypatch.setattr(_lib, "supported", lambda name, *a: True)   # each precision mode takes its tensor-core route
    monkeypatch.setattr(ops, "_chk", lambda t, name="tensor": t)
    monkeypatch.setattr(ops, "_st", lambda: 0)
    monkeypatch.setattr(ops, "copy_", lambda dst, src, accumulate=False: (dst.add_(src) if accumulate else dst.copy_(src)))
    monkeypatch.setattr(ops, "_pack_ok", lambda w, taps: w.dtype == torch.float32 and taps <= 9)
    monkeypatch.setattr(U, "_require_cuda", lambda *a, **k: None)
    old = ops.get_precision()
    yield seen
    ops.set_precision(old)


def _model(base_ch=16):
    from train.unet import TemporalUNetDualView
    torch.manual_seed(0)
    return TemporalUNetDualView(base_ch=base_ch, use_skip_lstm=True).eval()


SPLIT = ("b200_convlstm_cell_fwd_splitk_tc", "b200_conv_affine_relu_splitk_tc")


@pytest.mark.parametrize("precision", ["fp32", "bf16", "tf32"])
def test_three_frames_match_the_header(dry, precision):
    from unet_convlstm_b200 import ops
    ops.set_precision(precision)
    m = _model()
    B, S = 1, 64
    h0 = [(torch.zeros(B, 256, S // 16, S // 16), torch.zeros(B, 256, S // 16, S // 16))]
    s = m.stream(h0)
    assert s.state is not None and len(s.state) == 1
    for t in range(3):
        y = s.step(torch.rand(B, 2, S, S))
        assert y.shape == (B, 1, S, S) and y.dtype == torch.float32
    st = s.state
    assert len(st) == 1 and st[0][0].shape == (B, 256, S // 16, S // 16) and st[0][1].dtype == torch.float32
    if precision == "bf16":
        # 64x64, base_ch 16, B = 1: the cells and folded convs of the low-resolution levels have one M tile; those with
        # enough k-blocks (b200_splitk_splits) are split over K in every frame, the others keep the unsplit cell launch
        split = dry["b200_convlstm_cell_fwd_splitk_tc"]
        assert split >= 3 and split + dry.get("b200_convlstm_seq_fwd_tc", 0) == 3 * 3
        assert dry["b200_conv_affine_relu_splitk_tc"] >= 3 * 2
    else:
        assert not any(k in dry for k in SPLIT)


def test_forward_routing_is_unchanged(dry):
    """The split-K kernels are reachable only from a stream: model(x) of the same frames keeps its kernels."""
    from unet_convlstm_b200 import ops
    ops.set_precision("bf16")
    m = _model()
    with torch.no_grad():
        m(torch.rand(1, 3, 2, 64, 64))
        m(torch.rand(1, 1, 2, 64, 64))
    assert not any(k in dry for k in SPLIT)
    assert dry["b200_convlstm_seq_fwd_tc"] == 2 * 3


def test_refusals(dry):
    from unet_convlstm_b200 import ops
    ops.set_precision("bf16")
    m = _model()
    s = m.stream()
    s.step(torch.rand(2, 2, 32, 32))
    with pytest.raises(RuntimeError, match="differs from the first frame"):
        s.step(torch.rand(2, 2, 32, 48))
    with pytest.raises(RuntimeError, match="differs from the first frame"):
        s.step(torch.rand(2, 2, 32, 32, dtype=torch.float64))
    s.step(torch.rand(2, 2, 32, 32))
    with torch.no_grad():
        m.up1.conv.net[0].weight.add_(1.0)
    with pytest.raises(RuntimeError, match="changed since this stream bound it"):
        s.step(torch.rand(2, 2, 32, 32))
    m.load_state_dict(_model().state_dict())
    with pytest.raises(RuntimeError, match="changed since this stream bound it"):
        s.step(torch.rand(2, 2, 32, 32))
    s.reset()
    s.step(torch.rand(2, 2, 32, 48))      # a new sequence binds the new weights and frame shape
    m.train()
    with pytest.raises(RuntimeError, match="training mode"):
        s.step(torch.rand(2, 2, 32, 48))
