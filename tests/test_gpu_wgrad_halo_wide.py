"""wgrad_halo at every image width it accepts (16, 32, 64, 128), for both of its source widths (16 and 64 channels),
against an fp64 reference.

At W = 128 a pixel block is one image row, and the MMAs of the 16-channel mode read source-tile rows up to 7 padded
rows past their taps.  Those rows hold garbage and are never stored, but they must lie inside the shared-memory
allocation.  Before that was sized for (launch_wgrad_halo's `tail`), the last pipeline stage read past the end of
shared memory.  This broke the first layer's weight gradient of every model with 64 base channels at 128x128 (the
configs[2] shape).  The cases use enough pixel blocks per split for every stage of the ring, the last one included.
"""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 2.0 ** -20   # as tests/test_gpu_wgrad.py: bf16 operands are exact, only the fp32 accumulation differs
HALO = 2           # plan[0] of b200_wgrad_plan for wgrad_halo


def _reference(dz, src):
    """(dW, |dW|-sum) in fp64, [9, Nz, Csrc], tap = ky * 3 + kx, zero padding."""
    T, B, H, W, Nz = dz.shape
    dzd = dz.double().cpu().reshape(-1, Nz)
    sp = torch.nn.functional.pad(src.double().cpu(), (0, 0, 1, 1, 1, 1))
    ref, absref = [], []
    for ky in range(3):
        for kx in range(3):
            s = sp[:, :, ky:ky + H, kx:kx + W, :].reshape(-1, src.shape[-1])
            ref.append(dzd.T @ s)
            absref.append(dzd.abs().T @ s.abs())
    return torch.stack(ref), torch.stack(absref)


# (T, B, H, W, Nz, Csrc): 64 pixel blocks for every width
CASES = [(2, 2, 16, 128, 64, 16), (2, 2, 16, 128, 64, 64), (2, 2, 16, 128, 128, 16),
         (2, 2, 32, 64, 64, 16), (2, 2, 32, 64, 64, 64), (2, 4, 32, 32, 64, 16), (2, 4, 64, 16, 64, 16)]


@pytest.mark.parametrize("case", CASES, ids=[f"T{c[0]}B{c[1]}-{c[2]}x{c[3]}-Nz{c[4]}C{c[5]}" for c in CASES])
def test_wgrad_halo_every_width(case):
    from unet_convlstm_b200 import _lib
    T, B, H, W, Nz, Cs = case
    plan = (ctypes.c_int * 2)()
    _lib.call("b200_wgrad_plan", Nz, Cs, T, B, H, W, 3, Cs, 0, 0, ctypes.addressof(plan))
    assert plan[0] == HALO
    # pixel blocks per split: at least the 4 stages of the ring, so that the last stage is read
    assert T * B * H * W // 128 // plan[1] >= 4, plan[1]
    g = torch.Generator().manual_seed(sum(case))
    dz = torch.randn(T, B, H, W, Nz, generator=g).bfloat16().cuda()
    src = torch.randn(T, B, H, W, Cs, generator=g).bfloat16().cuda()
    ref, absref = _reference(dz, src)
    dw = torch.zeros(9, Nz, Cs, device="cuda")
    _lib.call("b200_wgrad_tc", dz, Nz, src, Cs, T, B, H, W, 3, dw, Cs, 0, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert _lib.lib().b200_device_error() == 0
    err = (dw.double().cpu() - ref).abs() / (TOL * absref + 1e-30)
    assert float(err.max()) <= 1.0, (case, float(err.max()))
