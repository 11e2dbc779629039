"""Tensor-level wrappers over the C ABI (include/b200_convlstm.h).

torch is used here for device memory (torch.empty / torch.zeros), strides and the current stream
only; every arithmetic kernel is one of ours.  Activations are NHWC: a sequence tensor is
[T, B, H, W, C] (contiguous); P = B*H*W pixels per timestep.
"""
from __future__ import annotations

import ctypes
import os

import torch

from . import _lib

# ------------------------------------------------------------------------------------------------
# precision mode
# ------------------------------------------------------------------------------------------------
_PRECISION = os.environ.get("B200_PRECISION", "bf16")


def set_precision(mode: str) -> None:
    """'bf16': tcgen05 tensor-core path, bf16 activations, fp32 accumulation and cell state.
    'tf32': fp32 activations and weights, convolutions and the fused cell forward on tcgen05 kind::tf32 (TF32 products,
            fp32 accumulation: the arithmetic of the reference's own GPU runs, cuDNN with torch's default allow_tf32);
            the weight-gradient reductions stay on the CUDA-core fp32 kernels.
    'fp32': check mode -- fp32 storage and CUDA-core FMA convolutions (1e-5 parity with the reference)."""
    global _PRECISION
    if mode not in ("bf16", "tf32", "fp32"):
        raise ValueError(f"unknown precision mode {mode!r}")
    _PRECISION = mode


def get_precision() -> str:
    return _PRECISION


def act_dtype() -> torch.dtype:
    return torch.bfloat16 if _PRECISION == "bf16" else torch.float32


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def _p(t):
    """A pointer argument of a C-ABI call: the tensor itself (unet_convlstm_b200._lib.call hands it to the torch custom op,
    or takes its data_ptr() on the ctypes route)."""
    return t


def bump_version(*tensors):
    """Marks tensors our kernels modified in place through raw pointers (torch cannot see those writes)."""
    for t in tensors:
        if t is not None:
            torch.autograd.graph.increment_version(t)


def _st():
    return torch.cuda.current_stream().cuda_stream


def _f32(t) -> int:
    if t.dtype == torch.float32:
        return 1
    if t.dtype == torch.bfloat16:
        return 0
    raise TypeError(f"unsupported dtype {t.dtype}")


def _chk(t, name="tensor"):
    if not t.is_cuda:
        raise RuntimeError(f"{name}: the B200 kernels need CUDA tensors (there is no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError(f"{name}: expected a contiguous tensor, got strides {t.stride()}")
    return t


_LL5 = ctypes.c_longlong * 5


def _copy_raw(dst, dst_off, src, src_off, dims, accumulate=False):
    """dims: list of (n, src_stride, dst_stride) in elements (strides may be negative)."""
    dims = [d for d in dims if d[0] != 1]
    merged = []
    for n, ss, ds in dims:
        if merged:
            pn, pss, pds = merged[-1]
            if pss == ss * n and pds == ds * n:
                merged[-1] = (pn * n, ss, ds)
                continue
        merged.append((n, ss, ds))
    if len(merged) > 5:
        raise ValueError("copy_: more than 5 non-mergeable dimensions")
    # iterate with the smallest destination stride innermost (coalesced writes)
    merged.sort(key=lambda d: -abs(d[2]))
    while len(merged) < 5:
        merged.insert(0, (1, 0, 0))
    _lib.call("b200_strided_copy", src.data_ptr() + src_off * src.element_size(), _f32(src),
              dst.data_ptr() + dst_off * dst.element_size(), _f32(dst),
              _LL5(*[d[0] for d in merged]), _LL5(*[d[1] for d in merged]), _LL5(*[d[2] for d in merged]),
              int(accumulate), _st())


def copy_(dst: torch.Tensor, src: torch.Tensor, accumulate: bool = False) -> torch.Tensor:
    """dst (+)= src for two equally-shaped, arbitrarily strided views (fp32 / bf16, converting)."""
    if tuple(dst.shape) != tuple(src.shape):
        raise ValueError(f"copy_: shape mismatch {tuple(dst.shape)} vs {tuple(src.shape)}")
    if not (dst.is_cuda and src.is_cuda):
        raise RuntimeError("copy_: the B200 kernels need CUDA tensors (there is no CPU fallback)")
    if dst.numel() == 0:
        return dst
    _copy_raw(dst, 0, src, 0, list(zip(src.shape, src.stride(), dst.stride())), accumulate)
    return dst


# ------------------------------------------------------------------------------------------------
# weight packing (all through the strided-copy kernel)
# ------------------------------------------------------------------------------------------------
def lstm_cht(Ch: int) -> int:
    """Hidden channels per GEMM N tile of the fused cell kernel (conv_tc.cu pick_block_n)."""
    return 64 if Ch % 64 == 0 else (32 if Ch % 32 == 0 else (16 if Ch % 16 == 0 else 0))


def _pack_ok(w: torch.Tensor, taps: int) -> bool:
    return w.dtype == torch.float32 and taps <= 9 and w.is_cuda


# While a functional.WeightCache builds an entry, every packed tensor derived from a parameter is noted here with the
# recipe that produced it -- ("pack", parameter, geometry of b200_pack_weight) or ("redo", parameters, closure) -- so
# that optim.AdamW can emit the packed copies from its update kernel (b200_adamw_pack) instead of leaving them to be
# re-packed at their first use in the next forward pass.
_PACK_RECORDER = None


def _pack(w, A, B, taps, out, a_contig, flip, tap_pitch, row_pitch, perm_ch=0, perm_cht=0):
    """b200_pack_weight: tiled layout change [A][B][taps] fp32 -> GEMM operand (see include/b200_convlstm.h)."""
    src = w.detach()
    if _PACK_RECORDER is not None and src.is_contiguous():
        _PACK_RECORDER.append(("pack", w, (A, B, taps, out, _f32(out), int(a_contig), int(flip), tap_pitch, row_pitch,
                                           perm_ch, perm_cht)))
    src = src if src.is_contiguous() else src.contiguous()
    _lib.call("b200_pack_weight", _p(src), A, B, taps, _p(out), _f32(out), int(a_contig), int(flip), tap_pitch,
              row_pitch, perm_ch, perm_cht, _st())
    return out


def pack_conv_weight(w: torch.Tensor, dtype: torch.dtype, kpad: int | None = None) -> torch.Tensor:
    """OIHW fp32 [N, K, k, k] -> [k*k, N, Kp] (K contiguous: the GEMM B operand, K-major)."""
    N, K, kh, kw = w.shape
    taps = kh * kw
    Kp = K if kpad is None else kpad
    out = (torch.zeros if Kp != K else torch.empty)((taps, N, Kp), device=w.device, dtype=dtype)
    if _pack_ok(w, taps):
        return _pack(w, N, K, taps, out, False, False, N * Kp, Kp)
    copy_(out[:, :, :K], w.detach().reshape(N, K, taps).permute(2, 0, 1))
    return out


def pack_conv_weight_dgrad(w: torch.Tensor, dtype: torch.dtype, kpad: int | None = None) -> torch.Tensor:
    """OIHW [N, K, k, k] -> [k*k (flipped), Kp, N]: the weights of the data-gradient convolution (rows >= K, the
    zero-padded input channels, stay zero)."""
    N, K, kh, kw = w.shape
    taps = kh * kw
    Kp = K if kpad is None else kpad
    out = (torch.zeros if Kp != K else torch.empty)((taps, Kp, N), device=w.device, dtype=dtype)
    if _pack_ok(w, taps):
        return _pack(w, N, K, taps, out, True, True, Kp * N, N)
    # out[taps-1-tap][k][n] = w[n][k][tap]: the tap dimension runs backwards in the destination
    _copy_raw(out, (taps - 1) * Kp * N, w.detach(), 0,
              [(taps, 1, -Kp * N), (K, taps, N), (N, K * taps, 1)])
    return out


def pack_lstm_weight(w: torch.Tensor, b: torch.Tensor | None, dtype: torch.dtype):
    """Gate-interleaved packing for the fused cell kernel: packed row (nt*4 + g)*CHT + j holds
    reference row g*Ch + nt*CHT + j (rows blocked i,f,g,o: unet.py:19,29)."""
    N, K, kh, kw = w.shape
    Ch, taps = N // 4, kh * kw
    cht = lstm_cht(Ch)
    nt = Ch // cht
    out = torch.empty((taps, N, K), device=w.device, dtype=dtype)
    if _pack_ok(w, taps):
        _pack(w, N, K, taps, out, False, False, N * K, K, Ch, cht)
    else:
        # views [taps, nt, g, j, K]
        dst = out.view(taps, nt, 4, cht, K)
        src = w.detach().reshape(4, nt, cht, K, taps).permute(4, 1, 0, 2, 3)
        copy_(dst, src)
    bp = None
    if b is not None:
        bp = torch.empty(N, device=w.device, dtype=torch.float32)

        def pack_bias():
            copy_(bp.view(nt, 4, cht), b.detach().reshape(4, nt, cht).permute(1, 0, 2))

        pack_bias()
        if _PACK_RECORDER is not None:
            _PACK_RECORDER.append(("redo", (b,), pack_bias))
    return out, bp


def pack_convT_weight(w: torch.Tensor, dtype: torch.dtype):
    """ConvTranspose2d weight IOHW [Cin, Cout, 2, 2] -> forward GEMM B operand [1, 4*Cout (tap, co), Cin]
    and data-gradient operand [1, Cin, 4*Cout]."""
    Cin, Cout = w.shape[0], w.shape[1]
    fwd = torch.empty((1, 4 * Cout, Cin), device=w.device, dtype=dtype)
    bwd = torch.empty((1, Cin, 4 * Cout), device=w.device, dtype=dtype)
    if _pack_ok(w, 4):
        _pack(w, Cin, Cout, 4, fwd, True, False, Cout * Cin, Cin)      # fwd[(tap, co)][ci] = w[ci][co][tap]
        _pack(w, Cin, Cout, 4, bwd, False, False, Cout, 4 * Cout)      # bwd[ci][(tap, co)] = w[ci][co][tap]
        return fwd, bwd
    copy_(fwd.view(4, Cout, Cin), w.detach().reshape(Cin, Cout, 4).permute(2, 1, 0))
    copy_(bwd.view(Cin, 4, Cout), w.detach().reshape(Cin, Cout, 4).permute(0, 2, 1))
    return fwd, bwd


def unpack_conv_wgrad(dw: torch.Tensor, K: int) -> torch.Tensor:
    """[taps, N, Kp] fp32 -> OIHW [N, K, k, k] fp32."""
    taps, N, Kp = dw.shape
    k = int(round(taps ** 0.5))
    g = torch.empty((N, K, k, k), device=dw.device, dtype=torch.float32)
    if dw.dtype == torch.float32 and dw.is_contiguous() and taps <= 9:
        _lib.call("b200_unpack_wgrad", _p(dw), N, K, taps, Kp, _p(g), _st())
        return g
    copy_(g.view(N, K, taps), dw[:, :, :K].permute(1, 2, 0))
    return g


# ------------------------------------------------------------------------------------------------
# convolutions
# ------------------------------------------------------------------------------------------------
def tc_conv_ok(x0, x1, N, lstm=False) -> bool:
    if x0.dtype != torch.bfloat16:
        return False
    T, B, H, W, C0 = x0.shape
    C1 = 0 if x1 is None else x1.shape[-1]
    return _lib.supported("b200_conv_tc_supported", B, H, W, C0, C1, N, int(lstm))


def conv_fwd(x0, x1, wp, bias, ksize, out0, out1=None, relu=False, bn_ws=None):
    """out = conv_k([x0 ; x1]) (+bias) (+relu).  x*: [T,B,H,W,C*]; wp: [k*k, N, C0+C1]; the N output
    columns go to out0 (its last dim) and, if given, the rest to out1 (dgrad of a virtual concat).
    bn_ws: optional fp64 [2, T, N] workspace; on the tensor-core path the per-(t, channel) sum and sum of
    squares of the output are accumulated into it by the conv epilogue.  Returns True if they were."""
    _chk(x0, "x0"), _chk(wp, "wp"), _chk(out0, "out0")
    T, B, H, W, C0 = x0.shape
    C1 = 0 if x1 is None else _chk(x1, "x1").shape[-1]
    N = wp.shape[1]
    split = out0.shape[-1]
    if wp.shape[2] != C0 + C1 or wp.dtype != x0.dtype:
        raise ValueError(f"conv_fwd: packed weights {tuple(wp.shape)}/{wp.dtype} do not match C0+C1={C0 + C1}/{x0.dtype}")
    if split + (0 if out1 is None else out1.shape[-1]) != N:
        raise ValueError("conv_fwd: output widths do not add up to N")
    if out1 is not None and out1.dtype != out0.dtype:
        raise ValueError("conv_fwd: out0/out1 dtypes differ")
    ld1 = 0 if out1 is None else out1.shape[-1]
    tag = f"K{C0 + C1} N{N} {H}x{W} k{ksize}"
    work = (2.0 * T * B * H * W * ksize * ksize * (C0 + C1) * N, None)
    tc = tc_conv_ok(x0, x1, N) and split % 16 == 0 and out0.shape[-1] % 8 == 0 and ld1 % 8 == 0
    if (not tc and _PRECISION == "tf32" and x0.dtype == torch.float32 and out0.dtype == torch.float32 and split % 16 == 0
            and out0.shape[-1] % 4 == 0 and ld1 % 4 == 0 and _lib.supported("b200_conv_tf32_supported", B, H, W, C0, C1, N, 0)):
        _lib.call("b200_conv_tf32_fwd", _p(x0), C0, _p(x1), C1, T, B, H, W, _p(wp), _p(bias), N, ksize, _p(out0),
                  out0.shape[-1], split, _p(out1), ld1, int(relu), 0, _st(), tag=tag + " tf32", work=work)
        return False
    if tc and bn_ws is not None and out1 is None and not relu and out0.dtype == torch.bfloat16:
        _lib.call("b200_conv_bnstats_tc_fwd", _p(x0), C0, _p(x1), C1, T, B, H, W, _p(wp), _p(bias), N, ksize,
                  _p(out0), _p(bn_ws[0]), _p(bn_ws[1]), _st(), tag=tag + " +bnstats", work=work)
        return True
    if tc:
        _lib.call("b200_conv_tc_fwd", _p(x0), C0, _p(x1), C1, T, B, H, W, _p(wp), _p(bias), N, ksize, _p(out0),
                  out0.shape[-1], split, _p(out1), ld1, _f32(out0), int(relu), 0, _st(), tag=tag, work=work)
    else:
        _lib.call("b200_conv_simt_fwd", _p(x0), C0, _p(x1), C1, T * B, H, W, _p(wp), _p(bias), N, ksize,
                  _p(out0), out0.shape[-1], split, _p(out1), ld1, _f32(x0), _f32(out0), int(relu), _st(),
                  tag=tag, work=work)
    return False


def conv_affine_relu_ok(x0, x1, N) -> bool:
    return x0.dtype == torch.bfloat16 and tc_conv_ok(x0, x1, N)


def conv_affine_relu(x0, x1, wp, scale, shift, ksize, relu=True):
    """Inference: relu(conv_k([x0 ; x1]) * scale + shift) in one kernel (eval-mode BatchNorm folded into the
    GEMM epilogue, b200_conv_affine_relu_tc_fwd).  Tensor-core path only (see conv_affine_relu_ok).  Under
    split_k_routing(), a single frame with few M tiles is split over K instead (splitk_splits)."""
    _chk(x0, "x0"), _chk(wp, "wp")
    T, B, H, W, C0 = x0.shape
    C1 = 0 if x1 is None else _chk(x1, "x1").shape[-1]
    N = wp.shape[1]
    splits = splitk_splits(x0, x1, N, ksize)
    if splits > 1:
        return conv_affine_relu_splitk(x0, x1, wp, scale, shift, ksize, splits, relu)
    out = torch.empty((T, B, H, W, N), device=x0.device, dtype=x0.dtype)
    _lib.call("b200_conv_affine_relu_tc_fwd", _p(x0), C0, _p(x1), C1, T, B, H, W, _p(wp), _p(scale), _p(shift), N, ksize,
              _p(out), int(relu), _st(), tag=f"K{C0 + C1} N{N} {H}x{W} k{ksize} +bn(eval)+relu",
              work=(2.0 * T * B * H * W * ksize * ksize * (C0 + C1) * N, None))
    return out


# ------------------------------------------------------------------------------------------------
# split K for single-frame problems with few M tiles (b200_splitk_splits).  Only streaming inference
# (unet_convlstm_b200/stream.py) routes here, inside split_k_routing(); every other call keeps its kernels.
# ------------------------------------------------------------------------------------------------
_SPLITK_ROUTING = [False]


class split_k_routing:
    """`with split_k_routing():` single-frame bf16 folded convolutions (conv_affine_relu) and ConvLSTM steps
    (lstm_seq_fwd_fused at T = 1) whose shape b200_splitk_splits selects run split over K."""

    def __enter__(self):
        self.prev, _SPLITK_ROUTING[0] = _SPLITK_ROUTING[0], True
        return self

    def __exit__(self, *exc):
        _SPLITK_ROUTING[0] = self.prev
        return False


def splitk_splits(x0, x1, N, ksize) -> int:
    """K splits for the bf16 convolution of the frame x0 [1,B,H,W,C0] (+ x1) into N channels: 1 = unsplit."""
    if not _SPLITK_ROUTING[0] or x0.dtype != torch.bfloat16 or x0.shape[0] != 1:
        return 1
    _, B, H, W, C0 = x0.shape
    C1 = 0 if x1 is None else x1.shape[-1]
    return int(_lib.lib().b200_splitk_splits(B, H, W, C0, C1, N, ksize))


def conv_affine_relu_splitk(x0, x1, wp, scale, shift, ksize, splits, relu=True, out_fp32=False):
    """conv_affine_relu of one frame (x0 [1,B,H,W,C0]) split over K into `splits` ranges (b200_conv_affine_relu_splitk_tc);
    scale / shift None: the plain convolution.  Returns [1,B,H,W,N], bf16 (fp32 with out_fp32)."""
    _chk(x0, "x0"), _chk(wp, "wp")
    T, B, H, W, C0 = x0.shape
    C1 = 0 if x1 is None else _chk(x1, "x1").shape[-1]
    N = wp.shape[1]
    if T != 1:
        raise ValueError(f"conv_affine_relu_splitk: one frame at a time, got T={T}")
    out = torch.empty((1, B, H, W, N), device=x0.device, dtype=torch.float32 if out_fp32 else x0.dtype)
    _lib.call("b200_conv_affine_relu_splitk_tc", _p(x0), C0, _p(x1), C1, B, H, W, _p(wp), _p(scale), _p(shift), N, ksize,
              _p(out), int(out_fp32), int(relu), int(splits), _st(),
              tag=f"K{C0 + C1} N{N} {H}x{W} k{ksize} +bn(eval)+relu splitK{splits}",
              work=(2.0 * B * H * W * ksize * ksize * (C0 + C1) * N, None))
    return out


def lstm_cell_fwd_splitk(x_t, h_prev, c_prev, wp_il, bias_il, c_next, h_next, ksize, splits):
    """One ConvLSTM step split over K (b200_convlstm_cell_fwd_splitk_tc): the fused cell without its gates output."""
    B, H, W, Cin = x_t.shape
    Ch = c_next.shape[-1]
    kin = Cin + (Ch if h_prev is not None else 0)
    _lib.call("b200_convlstm_cell_fwd_splitk_tc", _p(x_t), Cin, _p(h_prev), Ch, B, H, W, _p(wp_il), _p(bias_il),
              _p(c_prev), _p(c_next), _p(h_next), int(splits), ksize, _st(), tag=f"Ch{Ch} {H}x{W} splitK{splits}",
              work=(2.0 * B * H * W * ksize * ksize * kin * 4 * Ch, None))


def bn_eval_scale_shift(gamma, beta, running_mean, running_var, eps, conv_bias):
    """(scale, shift) of an eval-mode BatchNorm folded behind a conv with bias: y = conv * scale + shift."""
    C = gamma.numel()
    dev = gamma.device
    mean = torch.empty((1, C), device=dev, dtype=torch.float32)
    rstd, scale, shift = torch.empty_like(mean), torch.empty_like(mean), torch.empty_like(mean)
    _lib.call("b200_bn_finalize", None, None, 1, 1, C, _p(gamma), _p(beta), _p(running_mean), _p(running_var), eps, 0.0, 0,
              _p(mean), _p(rstd), _p(scale), _p(shift), _st())
    if conv_bias is not None:
        shift = torch.addcmul(shift, conv_bias.detach().float().view(1, C), scale)  # [C]-sized parameter algebra
    return scale.view(C), shift.view(C)


def conv_wgrad(dz, src, ksize, dw, koff):
    """dw[tap][n][koff + c] += sum_{t,p} dz[t,p,n] * src[t,p+tap,c]; dw fp32 [k*k, Nz, ldk]."""
    _chk(dz, "dz"), _chk(src, "src"), _chk(dw, "dw")
    T, B, H, W, Nz = dz.shape
    Cs = src.shape[-1]
    ldk = dw.shape[2]
    tag = f"Nz{Nz} C{Cs} {H}x{W} k{ksize} T{T}"
    work = (2.0 * T * B * H * W * ksize * ksize * Cs * Nz, None)
    if dz.dtype == torch.bfloat16 and ldk % 4 == 0 and koff % 4 == 0 and \
            _lib.supported("b200_wgrad_tc_supported", B, H, W, Nz, Cs):
        _lib.call("b200_wgrad_tc", _p(dz), Nz, _p(src), Cs, T, B, H, W, ksize, _p(dw), ldk, koff, _st(),
                  tag=tag, work=work)
    elif (_PRECISION == "tf32" and WGRAD_TF32 and dz.dtype == torch.float32 and src.dtype == torch.float32 and ldk % 4 == 0
          and koff % 4 == 0 and _lib.supported("b200_wgrad_tf32_supported", B, H, W, Nz, Cs)):
        _lib.call("b200_wgrad_tf32", _p(dz), Nz, _p(src), Cs, T, B, H, W, ksize, _p(dw), ldk, koff, _st(),
                  tag=tag + " tf32", work=work)
    else:
        _lib.call("b200_wgrad_simt", _p(dz), Nz, _p(src), Cs, T * B, H, W, ksize, _p(dw), ldk, koff, _f32(dz), _st(),
                  tag=tag, work=work)
    return dw


def colsum(x2d_rows: int, x, C: int, out=None, accumulate=False):
    """out[c] (+)= sum over rows of x viewed as [rows, C]."""
    ws = torch.empty(C, device=x.device, dtype=torch.float64)
    if out is None:
        out = torch.empty(C, device=x.device, dtype=torch.float32)
    _lib.call("b200_colsum", _p(x), x2d_rows, C, _f32(x), _p(ws), _p(out), int(accumulate), _st())
    return out


# ------------------------------------------------------------------------------------------------
# BatchNorm + ReLU
# ------------------------------------------------------------------------------------------------
# BatchNorm apply + ReLU + the 2x2 max-pool of the next Down stage in one pass, forward and backward (encoder outputs
# with even H and W): B200_FUSE_BN_POOL=0 goes back to the separate kernels (PoolFork).
FUSE_BN_POOL = os.environ.get("B200_FUSE_BN_POOL", "1") != "0"


def bn_pool_ok(z) -> bool:
    return FUSE_BN_POOL and z.shape[2] % 2 == 0 and z.shape[3] % 2 == 0


# BatchNorm apply + ReLU + the 1x1 OutConv (one output channel) in one pass, forward and backward: the last DoubleConv's
# full-resolution activation and its gradient are never materialised.  B200_FUSE_BN_OUTCONV=0: separate kernels.
FUSE_BN_OUTCONV = os.environ.get("B200_FUSE_BN_OUTCONV", "1") != "0"


def bn_outconv_ok(C: int, dtype, out_channels: int) -> bool:
    """C channels of `dtype` activations into a 1x1 convolution with `out_channels` outputs: can the fused kernels run?"""
    V = 4 if dtype == torch.float32 else 8
    cv = C // V
    return FUSE_BN_OUTCONV and out_channels == 1 and C % V == 0 and 1 <= cv <= 32 and (cv & (cv - 1)) == 0


def bn_relu_fwd(z, gamma, beta, running_mean, running_var, training, eps, momentum, ws=None, pool=False, outconv=None):
    """Returns (y, stats) with stats = (mean, rstd, scale, shift, tstride); statistics per (t, c).
    ws: fp64 [2, T, C] sums already produced by the conv epilogue (conv_fwd(..., bn_ws=ws)).
    pool: returns ((y, maxpool2x2(y)), stats), both outputs written by one kernel (H and W even).
    outconv = (w fp32 [C], b fp32 [1] or None): returns (out fp32 [T,B,H,W,1], stats) with out = outconv1x1(y); y itself
    is not written (bn_outconv_ok)."""
    _chk(z, "z")
    T, B, H, W, C = z.shape
    P = B * H * W
    dev = z.device
    Ts = T if training else 1
    mean = torch.empty((Ts, C), device=dev, dtype=torch.float32)
    rstd = torch.empty_like(mean)
    scale = torch.empty_like(mean)
    shift = torch.empty_like(mean)
    if training:
        if ws is None:
            ws = torch.empty((2, T, C), device=dev, dtype=torch.float64)
            _lib.call("b200_bn_stats", _p(z), T, P, C, _f32(z), _p(ws[0]), _p(ws[1]), _st(),
                      tag=f"C{C} {H}x{W}", work=(None, z.numel() * z.element_size()))
        _lib.call("b200_bn_finalize", _p(ws[0]), _p(ws[1]), T, P, C, _p(gamma), _p(beta), _p(running_mean),
                  _p(running_var), eps, momentum, 1, _p(mean), _p(rstd), _p(scale), _p(shift), _st())
        # the kernel wrote the running estimates through raw pointers: tell autograd's version counters, which
        # the folded-BatchNorm cache of the inference path (and anyone else) relies on
        bump_version(running_mean, running_var)   # (None when track_running_stats=False: nothing to update)
    else:
        _lib.call("b200_bn_finalize", None, None, 1, P, C, _p(gamma), _p(beta), _p(running_mean),
                  _p(running_var), eps, momentum, 0, _p(mean), _p(rstd), _p(scale), _p(shift), _st())
    tstride = C if training else 0
    if outconv is not None:
        w, b = outconv
        out = torch.empty((T, B, H, W, 1), device=dev, dtype=torch.float32)
        _lib.call("b200_bn_relu_outconv_fwd", _p(z), _p(scale), _p(shift), _p(w), _p(b), _p(out), T, P, C, tstride,
                  _f32(z), _st(), tag=f"C{C} {H}x{W}", work=(None, z.numel() * z.element_size() + out.numel() * 4))
        return out, (mean, rstd, scale, shift, tstride)
    y = torch.empty_like(z)
    if pool:
        yp = torch.empty((T, B, H // 2, W // 2, C), device=dev, dtype=z.dtype)
        _lib.call("b200_bn_relu_apply_pool", _p(z), _p(scale), _p(shift), _p(y), _p(yp), T, B, H, W, C, tstride,
                  _f32(z), _st(), tag=f"C{C} {H}x{W}", work=(None, (2 * z.numel() + yp.numel()) * z.element_size()))
        return (y, yp), (mean, rstd, scale, shift, tstride)
    _lib.call("b200_bn_relu_apply", _p(z), _p(scale), _p(shift), _p(y), T, P, C, tstride, 1, _f32(z), _st(),
              tag=f"C{C} {H}x{W}", work=(None, 2 * z.numel() * z.element_size()))
    return y, (mean, rstd, scale, shift, tstride)


def bn_relu_bwd(z, dy, stats, training, want_dbias=False, dpool=None, outconv_w=None):
    """Returns (dz, dgamma, dbeta, dconv_bias).  dpool: the gradient of maxpool2x2(y) (bn_relu_fwd(..., pool=True)); the
    gradient of y is then dy (may be None) + dpool routed to the window maxima, formed inside the two passes.
    outconv_w (fp32 [C]; bn_relu_fwd(..., outconv=...)): dy is the gradient of the 1x1 convolution's OUTPUT, fp32
    [T,B,H,W,1]; returns (dz, dgamma, dbeta, dconv_bias, d outconv_w)."""
    _chk(z, "z")
    mean, rstd, scale, shift, tstride = stats
    T, B, H, W, C = z.shape
    P = B * H * W
    dev = z.device
    ws = torch.empty((2, T, C), device=dev, dtype=torch.float64)
    esz = z.element_size()
    dw_out = None
    if outconv_w is not None:
        _chk(dy, "dout")
        if dy.dtype != torch.float32 or dy.numel() != T * P:
            raise ValueError("bn_relu_bwd(outconv_w=...): dy must be the fp32 [T,B,H,W,1] gradient of the 1x1 convolution")
        wsw = torch.empty(C, device=dev, dtype=torch.float64)
        dw_out = torch.empty(C, device=dev, dtype=torch.float32)
        _lib.call("b200_bn_relu_outconv_bwd_reduce", _p(z), _p(dy), _p(outconv_w), _p(mean), _p(rstd), _p(scale), _p(shift),
                  T, P, C, tstride, _f32(z), _p(ws[0]), _p(ws[1]), _p(wsw), _p(dw_out), _st(), tag=f"C{C} {H}x{W}",
                  work=(None, z.numel() * esz + dy.numel() * 4))
    elif dpool is not None:
        _chk(dpool, "dpool")
        if dy is not None:
            _chk(dy, "dy")
        nb = (1 if dy is None else 2) * z.numel() + dpool.numel()
        _lib.call("b200_bn_relu_pool_bwd_reduce", _p(z), _p(dy), _p(dpool), _p(mean), _p(rstd), _p(scale), _p(shift), T, B,
                  H, W, C, tstride, _f32(z), _p(ws[0]), _p(ws[1]), _st(), tag=f"C{C} {H}x{W}", work=(None, nb * esz))
    else:
        _chk(dy, "dy")
        _lib.call("b200_bn_relu_bwd_reduce", _p(z), _p(dy), _p(mean), _p(rstd), _p(scale), _p(shift), T, P, C, tstride,
                  _f32(z), _p(ws[0]), _p(ws[1]), _st(), tag=f"C{C} {H}x{W}", work=(None, 2 * z.numel() * esz))
    coef = torch.empty((2, T, C), device=dev, dtype=torch.float32)
    dgamma = torch.empty(C, device=dev, dtype=torch.float32)
    dbeta = torch.empty(C, device=dev, dtype=torch.float32)
    dcb = torch.empty(C, device=dev, dtype=torch.float32) if want_dbias else None
    _lib.call("b200_bn_bwd_finalize", _p(ws[0]), _p(ws[1]), T, P, C, int(training), _p(scale), _p(coef[0]),
              _p(coef[1]), _p(dgamma), _p(dbeta), _p(dcb), 0, _st())
    dz = torch.empty_like(z)
    if outconv_w is not None:
        _lib.call("b200_bn_relu_outconv_bwd_apply", _p(z), _p(dy), _p(outconv_w), _p(mean), _p(rstd), _p(scale), _p(shift),
                  _p(coef[0]), _p(coef[1]), _p(dz), T, P, C, tstride, _f32(z), _st(), tag=f"C{C} {H}x{W}",
                  work=(None, 2 * z.numel() * esz + dy.numel() * 4))
        return dz, dgamma, dbeta, dcb, dw_out
    if dpool is not None:
        _lib.call("b200_bn_relu_pool_bwd_apply", _p(z), _p(dy), _p(dpool), _p(mean), _p(rstd), _p(scale), _p(shift),
                  _p(coef[0]), _p(coef[1]), _p(dz), T, B, H, W, C, tstride, _f32(z), _st(), tag=f"C{C} {H}x{W}",
                  work=(None, (nb + z.numel()) * esz))
        return dz, dgamma, dbeta, dcb
    _lib.call("b200_bn_relu_bwd_apply", _p(z), _p(dy), _p(mean), _p(rstd), _p(scale), _p(shift), _p(coef[0]),
              _p(coef[1]), _p(dz), T, P, C, tstride, _f32(z), _st(), tag=f"C{C} {H}x{W}",
              work=(None, 3 * z.numel() * esz))
    return dz, dgamma, dbeta, dcb


# ------------------------------------------------------------------------------------------------
# max-pool, pixel shuffle, 1x1 output conv
# ------------------------------------------------------------------------------------------------
def maxpool2_fwd(x):
    _chk(x, "x")
    T, B, H, W, C = x.shape
    if H < 2 or W < 2:
        # nn.MaxPool2d(2) of the reference raises here too (an image smaller than 16 pixels on a side reaches the fourth Down
        # stage below 2x2); without this the empty tensor would travel on into the convolutions
        raise RuntimeError(f"max_pool2d(2): input {H}x{W} is too small (output size would be {H // 2}x{W // 2})")
    y = torch.empty((T, B, H // 2, W // 2, C), device=x.device, dtype=x.dtype)
    _lib.call("b200_maxpool2_fwd", _p(x), _p(y), T * B, H, W, C, _f32(x), _st())
    return y


def maxpool2_bwd(x, dy, accumulate_into=None):
    """dx = routing of dy to the maxima of x; with accumulate_into (a contiguous tensor like x) the routed gradient is
    ADDED to it in place -- the other gradient of a skip connection -- and it is returned."""
    _chk(x, "x"), _chk(dy, "dy")
    T, B, H, W, C = x.shape
    if accumulate_into is not None:
        _chk(accumulate_into, "accumulate_into")
        _lib.call("b200_maxpool2_bwd", _p(x), _p(dy), _p(accumulate_into), T * B, H, W, C, 1, _f32(x), _st())
        return accumulate_into
    dx = (torch.empty_like if (H % 2 == 0 and W % 2 == 0) else torch.zeros_like)(x)
    _lib.call("b200_maxpool2_bwd", _p(x), _p(dy), _p(dx), T * B, H, W, C, 0, _f32(x), _st())
    return dx


def shuffle2x2(z, bias, Hd, Wd):
    """z [T,B,H,W,4*C] (tap-major columns) -> y [T,B,Hd,Wd,C] (+bias), centred like F.pad (unet.py:95-97)."""
    _chk(z, "z")
    T, B, H, W, C4 = z.shape
    C = C4 // 4
    oy, ox = (Hd - 2 * H) // 2, (Wd - 2 * W) // 2
    exact = (Hd == 2 * H and Wd == 2 * W)
    y = (torch.empty if exact else torch.zeros)((T, B, Hd, Wd, C), device=z.device, dtype=z.dtype)
    _lib.call("b200_shuffle2x2", _p(z), _p(y), _p(bias), T * B, H, W, C, Hd, Wd, oy, ox, 0, _f32(z), _st())
    return y


def convT2x2_fwd(x, wf, bias, Cout, Hd, Wd):
    """ConvTranspose2d(k=2, s=2) + centring pad: on the tensor-core path one kernel (GEMM + pixel shuffle in the
    epilogue), otherwise the GEMM followed by b200_shuffle2x2."""
    _chk(x, "x")
    T, B, H, W, Cin = x.shape
    if CONVT_FUSED and x.dtype == torch.bfloat16 and Cout % 16 == 0 and tc_conv_ok(x, None, 4 * Cout):
        exact = (Hd == 2 * H and Wd == 2 * W)
        y = (torch.empty if exact else torch.zeros)((T, B, Hd, Wd, Cout), device=x.device, dtype=x.dtype)
        _lib.call("b200_convT2x2_tc_fwd", _p(x), Cin, T, B, H, W, _p(wf), _p(bias), Cout, _p(y), Hd, Wd, _st(),
                  tag=f"K{Cin} N{4 * Cout} {H}x{W} convT", work=(2.0 * T * B * H * W * Cin * 4 * Cout, None))
        return y
    z = torch.empty((T, B, H, W, 4 * Cout), device=x.device, dtype=x.dtype)
    conv_fwd(x, None, wf, None, 1, z)
    return shuffle2x2(z, bias, Hd, Wd)


def unshuffle2x2(dy, H, W):
    _chk(dy, "dy")
    T, B, Hd, Wd, C = dy.shape
    oy, ox = (Hd - 2 * H) // 2, (Wd - 2 * W) // 2
    du = torch.empty((T, B, H, W, 4 * C), device=dy.device, dtype=dy.dtype)
    _lib.call("b200_shuffle2x2", _p(dy), _p(du), None, T * B, H, W, C, Hd, Wd, oy, ox, 1, _f32(dy), _st())
    return du


def outconv_fwd(x, w, b):
    """x [T,B,H,W,C], w fp32 [O,C] -> y fp32 [T,B,H,W,O]."""
    _chk(x, "x")
    T, B, H, W, C = x.shape
    O = w.shape[0]
    y = torch.empty((T, B, H, W, O), device=x.device, dtype=torch.float32)
    _lib.call("b200_outconv_fwd", _p(x), _p(w), _p(b), _p(y), T * B * H * W, C, O, _f32(x), _st())
    return y


def outconv_bwd(x, w, dy, need_dx=True):
    _chk(x, "x"), _chk(dy, "dy")
    T, B, H, W, C = x.shape
    O = w.shape[0]
    dx = torch.empty_like(x) if need_dx else None
    ws = torch.empty(max(C, O), device=x.device, dtype=torch.float64)
    dw = torch.empty((O, C), device=x.device, dtype=torch.float32)
    db = torch.empty(O, device=x.device, dtype=torch.float32)
    _lib.call("b200_outconv_bwd", _p(x), _p(w), _p(dy), T * B * H * W, C, O, _f32(x), _p(dx), _p(ws), _p(dw), _p(db),
              0, _st())
    return dx, dw, db


# ------------------------------------------------------------------------------------------------
# SpatialAttention (unet.py:113-125): y = x * sigmoid(conv_k([mean_c x ; amax_c x]))
# ------------------------------------------------------------------------------------------------
ATTENTION_KSIZES = (1, 3, 5, 7)
_ATTN_WGRAD_PIXELS = 2048   # pixels per partial weight-gradient sum of b200_spatial_attention_bwd


def _attn_ksize(w):
    k = w.shape[-1]
    if w.dim() != 4 or tuple(w.shape[:2]) != (1, 2) or w.shape[2] != k or k not in ATTENTION_KSIZES:
        raise RuntimeError(f"spatial attention: weight {tuple(w.shape)} is not supported: the kernels take [1, 2, k, k] with "
                           f"k in {ATTENTION_KSIZES} (there is no fallback)")
    if w.dtype != torch.float32:
        raise RuntimeError(f"spatial attention: weight dtype {w.dtype}, expected torch.float32")
    return k


def spatial_attention_fwd(x, w):
    """x [T,B,H,W,C] (activation dtype), w fp32 [1,2,k,k] -> (y like x, pooled fp32 [T,B,H,W,2], a fp32 [T,B,H,W])."""
    _chk(x, "x"), _chk(w, "w")
    k = _attn_ksize(w)
    T, B, H, W, C = x.shape
    pooled = torch.empty((T, B, H, W, 2), device=x.device, dtype=torch.float32)
    a = torch.empty((T, B, H, W), device=x.device, dtype=torch.float32)
    y = torch.empty_like(x)
    _lib.call("b200_spatial_attention_fwd", _p(x), _p(w), T * B, H, W, C, k, _f32(x), _p(pooled), _p(a), _p(y), _st(),
              tag=f"C{C} {H}x{W} k{k}", work=(None, 3 * x.numel() * x.element_size()))   # x read twice, y written
    return y, pooled, a


def spatial_attention_bwd(x, dy, w, pooled, a, need_dx=True, need_dw=True):
    """Returns (dx like x or None, dw fp32 [1,2,k,k] or None) for y = spatial_attention_fwd(x, w)[0] and dy = dL/dy."""
    _chk(x, "x"), _chk(dy, "dy"), _chk(w, "w"), _chk(pooled, "pooled"), _chk(a, "a")
    k = _attn_ksize(w)
    T, B, H, W, C = x.shape
    P = T * B * H * W
    ws = torch.empty(2 * P + -(-P // _ATTN_WGRAD_PIXELS) * 2 * k * k, device=x.device, dtype=torch.float32)
    dx = torch.empty_like(x) if need_dx else None
    dw = torch.empty((1, 2, k, k), device=x.device, dtype=torch.float32) if need_dw else None
    _lib.call("b200_spatial_attention_bwd", _p(x), _p(dy), _p(w), _p(pooled), _p(a), T * B, H, W, C, k, _f32(x), _p(ws),
              _p(dx), _p(dw), _st(), tag=f"C{C} {H}x{W} k{k}",
              work=(None, (2 + 3 * need_dx) * x.numel() * x.element_size()),   # (x, dy) read once or twice, dx written
              kernels=2 + int(need_dx) + 2 * int(need_dw))
    return dx, dw


# ------------------------------------------------------------------------------------------------
# ConvLSTM cell
# ------------------------------------------------------------------------------------------------
def lstm_tc_ok(x_t, Ch) -> bool:
    B, H, W, Cin = x_t.shape
    if x_t.dtype == torch.float32 and _PRECISION == "tf32":
        return _lib.supported("b200_conv_tf32_supported", B, H, W, Cin, Ch, 4 * Ch, 1)
    if x_t.dtype != torch.bfloat16:
        return False
    return _lib.supported("b200_conv_tc_supported", B, H, W, Cin, Ch, 4 * Ch, 1)


# tf32 mode: weight gradients on tcgen05 kind::tf32 (1) or on the CUDA-core fp32 kernel (0)
WGRAD_TF32 = os.environ.get("B200_WGRAD_TF32", "1") != "0"

# ConvTranspose 2x2: pixel shuffle in the GEMM epilogue (1) or GEMM + separate shuffle kernel (0)
CONVT_FUSED = os.environ.get("B200_CONVT_FUSED", "1") != "0"

# BatchNorm batch statistics in the conv epilogue instead of a separate pass (slower on B200, see functional.py)
FUSE_BN_STATS = os.environ.get("B200_FUSE_BN_STATS", "0") == "1"

# One cooperative timestep-persistent launch per ConvLSTM layer (default) or one launch per timestep
PERSISTENT_LSTM = os.environ.get("B200_PERSISTENT_LSTM", "1") != "0"

# Fused timestep-persistent BPTT kernel (b200_convlstm_seq_bwd_tc) instead of per-step gate-gradient + dgrad
# launches.  Opt-in: measured on B200 (profiles/r01_fused_bptt_measured.txt) the gate-gradient operand traffic
# of the epilogue competes with the L2-bound main loop and the per-step pair of launches is 0-13 % faster.
FUSED_BPTT = os.environ.get("B200_FUSED_BPTT", "0") == "1"

# Weight gradients on a background stream (1) or in line on the current stream (0).  A weight gradient is a leaf of
# backward: nothing downstream waits for it, while the HBM-bound kernels of the NEXT layer's backward (BatchNorm
# sums / apply, gate gradients, pooling) leave the tensor pipes idle.  With the wgrad kernels queued on a second
# stream their CTAs share the SMs with those pointwise blocks (a persistent wgrad CTA leaves ~40 K registers and room
# for two 256-thread blocks per SM).  The current stream re-joins the background stream when backward ends.
#
# OPT-IN (ADVICE r01): a gradient produced on the background stream is only safe if nothing reads it on the current
# stream before backward ends.  _leaf_takes_gradient_as_is() sees tensor hooks and post-accumulate hooks, but hooks on
# the AccumulateGrad NODE -- how torch DistributedDataParallel / FSDP attach their reducers -- cannot be listed from
# Python, so a DDP-wrapped model would copy a gradient that is still being written.  The switch is therefore off
# unless a component that KNOWS the ordering turns it on: this package's GradReducer (dist.py), its training loop
# (loop.py), bench.py and tools/soak.py call enable_background_wgrad(); B200_WGRAD_STREAM=1 / 0 forces it on / off.
_WGRAD_STREAM_ENV = os.environ.get("B200_WGRAD_STREAM", "")
WGRAD_STREAM = _WGRAD_STREAM_ENV == "1"


def enable_background_wgrad(on: bool = True) -> bool:
    """Turns the background weight-gradient stream on (or off) for this process, unless B200_WGRAD_STREAM forces a
    value.  Call it only from a training step that reads parameter gradients AFTER backward() has returned (plain
    optimizers, this package's GradReducer); leave it off under torch DistributedDataParallel / FSDP."""
    global WGRAD_STREAM
    if _WGRAD_STREAM_ENV in ("0", "1"):
        return WGRAD_STREAM
    WGRAD_STREAM = bool(on)
    return WGRAD_STREAM


_BG_DEBUG_DELAY = int(os.environ.get("B200_WGRAD_STREAM_DEBUG_DELAY", "0"))  # spin cycles before every background block (tests)
# ConvLSTM BPTT: timesteps per weight-gradient chunk queued on the background stream while the sweep continues
# (0 = one weight-gradient reduction after the sweep, the default).  Measured (profiles/r01_background_wgrad_ab.txt):
# chunks of 5 steps 207.6-208.5 ms against 206.8-206.9 ms per step, 4 or 10 steps ~212 ms -- the chunk's persistent
# CTAs hold SMs the recurrent (critical-path) dgrad step of the main stream is waiting for.
LSTM_WGRAD_CHUNK = int(os.environ.get("B200_LSTM_WGRAD_CHUNK", "0"))
BG_BLOCKS = [0]  # blocks that actually ran on the background stream (tests)
_bg_streams: dict = {}
_bg_joined_task = [-1]


def background_stream(device=None):
    idx = torch.cuda.current_device() if device is None else torch.device(device).index
    st = _bg_streams.get(idx)
    if st is None:
        st = _bg_streams[idx] = torch.cuda.Stream(idx)
    return st


def background_join():
    """The current stream waits for everything queued on the background stream so far."""
    st = _bg_streams.get(torch.cuda.current_device())
    if st is not None:
        torch.cuda.current_stream().wait_stream(st)


def _leaf_takes_gradient_as_is(p) -> bool:
    """True if autograd will only STORE the new gradient of leaf `p` (no kernel on the current stream reads it during
    backward): .grad is still empty and nobody hooked the tensor -- except hooks that declare themselves aware of the
    background stream (dist.GradReducer sets `_b200_bg_aware`)."""
    if not p.is_leaf or p.grad is not None:
        return False
    if getattr(p, "_backward_hooks", None):
        return False
    if getattr(p, "_post_accumulate_grad_hooks", None) and not getattr(p, "_b200_bg_aware", False):
        return False
    return True


class background:
    """`with background(params, *inputs) as bg:` (params: the leaf or leaves whose gradients the block produces) -- the
    launches inside run on the background stream, ordered
    after everything already queued on the current stream; `inputs` are tensors the block reads (kept away from the
    caching allocator until the background work is done).  Falls back to the current stream (bg.active False) outside
    a backward pass, when the switch is off, when `allow` is False (the caller knows of a second gradient contribution
    to the same parameters), or when autograd would touch the new gradient during backward (_leaf_takes_gradient_as_is)."""

    def __init__(self, grad_target, *inputs, allow=True):
        self.inputs = [t for t in inputs if t is not None]
        self.targets = list(grad_target) if isinstance(grad_target, (tuple, list)) else [grad_target]
        task = torch._C._current_graph_task_id()
        self.active = bool(WGRAD_STREAM and allow and task != -1 and not torch.is_grad_enabled()
                           and all(_leaf_takes_gradient_as_is(p) for p in
                                   (grad_target if isinstance(grad_target, (tuple, list)) else (grad_target,))
                                   if p is not None))
        self.task = task

    def __enter__(self):
        if not self.active:
            return self
        cur = torch.cuda.current_stream()
        self.side = background_stream()
        self.side.wait_stream(cur)
        for t in self.inputs:
            t.record_stream(self.side)
        if _bg_joined_task[0] != self.task:
            # one join per backward pass: whoever reads the gradients after backward() sees them complete
            _bg_joined_task[0] = self.task
            torch.autograd.Variable._execution_engine.queue_callback(_end_of_backward_join)
        BG_BLOCKS[0] += 1
        self.ctx = torch.cuda.stream(self.side)
        self.ctx.__enter__()
        if _BG_DEBUG_DELAY:
            torch.cuda._sleep(_BG_DEBUG_DELAY)
        return self

    def __exit__(self, *exc):
        if self.active:
            self.ctx.__exit__(*exc)
        return False

    def keep(self, *tensors):
        """Tensors created inside the block that the CURRENT stream will own afterwards (returned gradients, in the
        order of the block's parameters)."""
        if self.active:
            cur = torch.cuda.current_stream()
            for t in tensors:
                if t is not None:
                    t.record_stream(cur)
            for p, t in zip(self.targets, tensors):
                if p is not None and t is not None and tuple(t.shape) == tuple(p.shape):
                    _bg_delivered.append((p, t.data_ptr()))


# (parameter, data_ptr of the gradient produced on the background stream) of the running backward pass
_bg_delivered: list = []


# Host lead limit.  Tensors that cross to the background stream (ops.background inputs / outputs: record_stream) return to
# the caching allocator's pool only once the GPU has passed their last use.  A GPU-bound training loop that never
# synchronises (no loss.item()) lets the host run ~2 steps ahead of the GPU: it frees and re-allocates those blocks long
# before they are reusable, the allocator answers with fresh cudaMalloc calls, the reserved pool creeps up to the whole
# HBM and then stalls for 0.1-0.8 s in its out-of-memory retry (free everything, synchronise, malloc again) -- measured
# on B200 in bench.py's non-synchronising regions: 37-199 cudaMalloc calls and 3 retries inside the timed steps, single
# steps of 289-794 ms among 207 ms ones, the whole 8-GPU job waiting for whichever rank stalled
# (profiles/r02_allocator_stalls.md).  So the end of every backward pass that used the background stream waits, on the
# HOST, for the end of the PREVIOUS such backward: the host stays at most one step ahead (the GPU still has a full step
# queued), and the cross-stream working set is bounded by two steps.
_lead_events: dict = {}
HOST_LEAD_LIMIT = os.environ.get("B200_HOST_LEAD_LIMIT", "1") != "0"


def _limit_host_lead():
    if not HOST_LEAD_LIMIT:
        return
    dev = torch.cuda.current_device()
    prev = _lead_events.get(dev)
    if prev is not None:
        prev.synchronize()
    ev = torch.cuda.Event()
    ev.record()
    _lead_events[dev] = ev


def _end_of_backward_join():
    _bg_joined_task[0] = -1
    background_join()
    _limit_host_lead()
    # AccumulateGrad must have STORED each background gradient (same storage).  Had it cloned or accumulated instead
    # (a second reference to the gradient, mismatching strides, a .grad that appeared meanwhile), that kernel ran on
    # the current stream while the background stream was still writing: corrupt, so fail loudly.
    delivered, _bg_delivered[:] = list(_bg_delivered), []
    for p, ptr in delivered:
        g = p.grad
        if g is not None and g.data_ptr() != ptr and not getattr(p, "_b200_bg_aware", False):
            raise RuntimeError("background weight-gradient stream: autograd did not store the gradient of a parameter as "
                               "produced (it was copied or accumulated during backward, on the current stream, while the "
                               "background stream was still writing it).  Call ops.enable_background_wgrad(False).")


# bench.py sets this to a list to time every fused cell launch with CUDA events on the launching stream:
# entries are (start_event, end_event, algorithmic_flops)
CELL_TIMER = None


def lstm_cell_fwd_fused(x_t, h_prev, c_prev, wp_il, bias_il, c_next, h_next, gates, ksize):
    """One fused cell step on the tensor cores (gate conv + gate math + state update)."""
    B, H, W, Cin = x_t.shape
    Ch = c_next.shape[-1]
    timer = CELL_TIMER
    if timer is not None:
        e0 = torch.cuda.Event(enable_timing=True)
        e0.record()
    kin_ = Cin + (Ch if h_prev is not None else 0)
    entry = "b200_convlstm_cell_fwd_tf32" if x_t.dtype == torch.float32 else "b200_convlstm_cell_fwd_tc"
    _lib.call(entry, _p(x_t), Cin, _p(h_prev), Ch, B, H, W, _p(wp_il), _p(bias_il),
              _p(c_prev), _p(c_next), _p(h_next), _p(gates), ksize, _st(), tag=f"Ch{Ch} {H}x{W}",
              work=(2.0 * B * H * W * ksize * ksize * kin_ * 4 * Ch, None))
    if timer is not None:
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        kin = Cin + (Ch if h_prev is not None else 0)
        timer.append((e0, e1, 2.0 * B * H * W * ksize * ksize * kin * 4 * Ch))


def lstm_seq_fwd_fused(x_seq, h_all, c_all, wp_il, bias_il, gates, have_h0, ksize):
    """All T steps of one ConvLSTM layer in one timestep-persistent cooperative launch."""
    T, B, H, W, Cin = x_seq.shape
    Ch = c_all.shape[-1]
    if T == 1:
        splits = splitk_splits(x_seq, h_all[0] if have_h0 else None, 4 * Ch, ksize)
        if splits > 1:   # (split_k_routing only; the gates are not written)
            lstm_cell_fwd_splitk(x_seq[0], h_all[0] if have_h0 else None, c_all[0] if have_h0 else None, wp_il, bias_il,
                                 c_all[1], h_all[1], ksize, splits)
            return
    kin = Cin + Ch
    fl = 2.0 * B * H * W * ksize * ksize * 4 * Ch * (kin * T - (0 if have_h0 else Ch))
    timer = CELL_TIMER
    if timer is not None:
        e0 = torch.cuda.Event(enable_timing=True)
        e0.record()
    _lib.call("b200_convlstm_seq_fwd_tc", _p(x_seq), Cin, _p(h_all), Ch, T, B, H, W, _p(wp_il), _p(bias_il),
              _p(c_all), _p(gates), int(have_h0), ksize, _st(), tag=f"Ch{Ch} {H}x{W} T{T}", work=(fl, None))
    if timer is not None:
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        timer.append((e0, e1, fl))


# Gate recompute (north_star "gate-gradient recompute"): do not keep the activated gates [T, P, 4*Ch] of every ConvLSTM
# layer between forward and backward; BPTT recomputes them for all T steps in one tensor-core launch from the stored
# x_t / h_{t-1} / c_{t-1} (the steps are independent once the states are known) into the buffer the gate-gradient
# kernel then overwrites with dz.  Costs one extra forward gate conv per layer (+1/3 of the cell FLOPs), saves
# T*P*4*Ch*2 bytes of activation memory per layer.  Off by default (speed); B200_GATE_RECOMPUTE=1 or set_gate_recompute().
GATE_RECOMPUTE = os.environ.get("B200_GATE_RECOMPUTE", "0") == "1"


def set_gate_recompute(on: bool) -> None:
    global GATE_RECOMPUTE
    GATE_RECOMPUTE = bool(on)


def lstm_gates_recompute(x_seq, h_all, c_all, wp_il, bias_il, gates_out, ksize):
    """Activated gates of all T steps of a layer from its stored states (BPTT with GATE_RECOMPUTE)."""
    T, B, H, W, Cin = x_seq.shape
    Ch = c_all.shape[-1]
    fl = 2.0 * T * B * H * W * ksize * ksize * 4 * Ch * (Cin + Ch)
    _lib.call("b200_convlstm_gates_recompute_tc", _p(x_seq), Cin, _p(h_all), Ch, T, B, H, W, _p(wp_il), _p(bias_il),
              _p(c_all), _p(gates_out), ksize, _st(), tag=f"Ch{Ch} {H}x{W} T{T}", work=(fl, None))


def lstm_seq_bwd_ok(x_seq, Ch) -> bool:
    """Can the fused timestep-persistent BPTT kernel run this layer?"""
    if x_seq.dtype != torch.bfloat16 or not PERSISTENT_LSTM or not FUSED_BPTT:
        return False
    T, B, H, W, Cin = x_seq.shape
    if T < 2 or Cin % 16 or Ch % 16:
        return False
    return _lib.supported("b200_conv_tc_supported", B, H, W, 4 * Ch, 0, Cin + Ch, 0)


def lstm_seq_bwd_fused(dz_all, wd, gates, c_all, dh_seq, dc_buf, dx_seq, dh0, Cin, have_h0, ksize):
    """Steps T-1 .. 0 of BPTT in one cooperative launch: dgrad conv of dz_t with the gate gradients of step
    t-1 in its epilogue (see include/b200_convlstm.h).  dz_all[T-1] and dc_buf[(T-1) & 1] must be filled."""
    T, B, H, W, C4 = dz_all.shape
    Ch = C4 // 4
    fl = 2.0 * T * B * H * W * ksize * ksize * C4 * (Cin + Ch)
    _lib.call("b200_convlstm_seq_bwd_tc", _p(dz_all), _p(wd), _p(gates), _p(c_all), _p(dh_seq), _p(dc_buf),
              _p(dx_seq), _p(dh0), Cin, Ch, T, B, H, W, int(have_h0), ksize, _st(),
              tag=f"Ch{Ch} {H}x{W} T{T}", work=(fl, None))


def lstm_cell_fwd_unfused(x_t, h_prev, c_prev, wp, bias, c_next, h_next, gates, ksize, zbuf):
    """Generic path: CUDA-core gate conv into fp32 pre-activations, then the gate-math kernel."""
    B, H, W, Cin = x_t.shape
    Ch = c_next.shape[-1]
    if h_prev is None:
        # zero initial state (unet.py:23-25): only the x columns of the packed weights contribute
        raise RuntimeError("lstm_cell_fwd_unfused needs an explicit h_prev")
    _lib.call("b200_conv_simt_fwd", _p(x_t), Cin, _p(h_prev), Ch, B, H, W, _p(wp), _p(bias), 4 * Ch, ksize,
              _p(zbuf), 4 * Ch, 4 * Ch, None, 0, _f32(x_t), 1, 0, _st())
    _lib.call("b200_lstm_gates_fwd", _p(zbuf), _p(c_prev), _p(gates), _p(c_next), _p(h_next), B * H * W, Ch,
              _f32(x_t), _st())


def lstm_gates_bwd(gates, c_prev, c_next, dh_a, dh_b, dc_next, dz, dc_prev):
    B, H, W, Ch = c_next.shape
    es = gates.element_size()
    nb = B * H * W * Ch * (4 * es + 8 + es * (1 + (dh_b is not None)) + 4 * (dc_next is not None) + 4 * es + 4)
    _lib.call("b200_lstm_gates_bwd", _p(gates), _p(c_prev), _p(c_next), _p(dh_a), _p(dh_b), _p(dc_next), _p(dz),
              _p(dc_prev), B * H * W, Ch, _f32(gates), _st(), tag=f"Ch{Ch} {H}x{W}", work=(None, nb))
