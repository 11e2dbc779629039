"""B200-native drop-in for `train/unet.py` of dordanino12/unet-convlstm.

Same class names, constructor arguments, tensor layouts (NCHW fp32 at the module boundary) and
state_dict keys as the reference, so main.py / train/overfit_check.py / train/get_metrics.py import
and drive it unchanged.  Every forward/backward runs hand-written sm_100a CUDA kernels through the
C ABI of include/b200_convlstm.h (unet_convlstm_b200/): there is no PyTorch-op, cuDNN or CPU fallback
-- a CPU tensor or a missing library raises.

Parameters live in the same leaf modules the reference uses (nn.Conv2d / nn.BatchNorm2d /
nn.ConvTranspose2d), which keeps the key names, shapes, default initialisation and the order in which
the RNG is consumed identical; those leaves are parameter holders only, their forward is never called.

Internally activations are channels-last sequence tensors [T, B, H, W, C]; the encoder and decoder
run on all T frames at once while BatchNorm keeps the reference's per-timestep statistics
(the reference calls each block once per frame: unet.py:179-182, :196-202).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn
from torch.utils.data import Dataset

from unet_convlstm_b200 import functional as Fn
from unet_convlstm_b200 import ops


def _require_cuda(t: torch.Tensor, who: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{who}: input is on {t.device}; the B200 kernels have no CPU fallback")


def _to_nhwc(x: torch.Tensor, pad_to=None) -> torch.Tensor:
    """[B,C,H,W] (any float dtype) -> [1,B,H,W,C] in the activation dtype."""
    return Fn.permute_cast(x, (0, 2, 3, 1), ops.act_dtype(), pad_to).unsqueeze(0)


def _to_nchw(y: torch.Tensor) -> torch.Tensor:
    """[1,B,H,W,C] -> [B,C,H,W] fp32."""
    return Fn.permute_cast(y[0], (0, 3, 1, 2), torch.float32)


def _in_pad(c: int) -> int | None:
    """bf16 mode: the first conv's few input channels are zero-padded to one tensor-core K chunk."""
    if ops.get_precision() == "bf16":
        return 16 if c < 16 else None
    if ops.get_precision() == "tf32":
        return 8 if c < 8 else None      # one tf32 K block (32 bytes)
    return None


# -----------------------------------------------------------------------------------------------
# ConvLSTM (reference unet.py:14-60)
# -----------------------------------------------------------------------------------------------
class ConvLSTMCell(nn.Module):
    def __init__(self, input_dim, hidden_dim, kernel_size=3, bias=True):
        super().__init__()
        self.hidden_dim = hidden_dim
        self.conv = nn.Conv2d(input_dim + hidden_dim, 4 * hidden_dim, kernel_size, padding=kernel_size // 2, bias=bias)
        self._cache = Fn.WeightCache()

    def _seq(self, x_seq, h0, c0):
        """x_seq [T,B,H,W,Cin]; h0 (act dtype) / c0 (fp32) [B,H,W,Ch] or None -> (h_seq, c_T)."""
        return Fn.ConvLSTMSeq.apply(x_seq, h0, c0, self.conv.weight, self.conv.bias, self._cache)

    def forward(self, x, state=None):
        _require_cuda(x, "ConvLSTMCell")
        xs = _to_nhwc(x)
        h0 = c0 = None
        if state is not None:
            h0 = Fn.permute_cast(state[0], (0, 2, 3, 1), ops.act_dtype())
            c0 = Fn.permute_cast(state[1], (0, 2, 3, 1), torch.float32)
        h_seq, c_T = self._seq(xs, h0, c0)
        h = _to_nchw(h_seq)
        c = Fn.permute_cast(c_T, (0, 3, 1, 2), torch.float32)
        return h, (h, c)


class ConvLSTM(nn.Module):
    def __init__(self, input_dim, hidden_dim, num_layers=1, kernel_size=3):
        super().__init__()
        self.layers = nn.ModuleList(
            ConvLSTMCell(input_dim if l == 0 else hidden_dim, hidden_dim, kernel_size) for l in range(num_layers))

    def _seq(self, x_seq, state):
        """Layer-major like the reference (unet.py:52-57).  state: list of (h0, c0) NHWC or None."""
        out = x_seq
        finals = []
        for li, layer in enumerate(self.layers):
            h0, c0 = (None, None) if state is None or state[li] is None else state[li]
            out, c_T = layer._seq(out, h0, c0)
            finals.append((out[-1], c_T))
        return out, finals

    def forward(self, x_seq, state=None):
        T = len(x_seq)
        _require_cuda(x_seq[0], "ConvLSTM")
        x = torch.stack(list(x_seq), dim=0)  # [T,B,C,H,W]
        xs = Fn.permute_cast(x, (0, 1, 3, 4, 2), ops.act_dtype())
        st = None
        if state is not None:
            st = [None if s is None or s[0] is None else
                  (Fn.permute_cast(s[0], (0, 2, 3, 1), ops.act_dtype()), Fn.permute_cast(s[1], (0, 2, 3, 1), torch.float32))
                  for s in state]
        out, finals = self._seq(xs, st)
        out_nchw = Fn.permute_cast(out, (0, 1, 4, 2, 3), torch.float32)
        new_states = [(Fn.permute_cast(h, (0, 3, 1, 2), torch.float32), Fn.permute_cast(c, (0, 3, 1, 2), torch.float32))
                      for h, c in finals]
        # unbind, not T x select: the backward of unbind stacks the T frame gradients in one pass, T selects would
        # each materialise a full-size zero tensor and autograd would add the T of them
        return list(out_nchw.unbind(0)), new_states


# -----------------------------------------------------------------------------------------------
# UNet blocks (reference unet.py:66-107)
# -----------------------------------------------------------------------------------------------
class DoubleConv(nn.Module):
    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.net = nn.Sequential(
            nn.Conv2d(in_ch, out_ch, 3, padding=1), nn.BatchNorm2d(out_ch), nn.ReLU(inplace=True),
            nn.Conv2d(out_ch, out_ch, 3, padding=1), nn.BatchNorm2d(out_ch), nn.ReLU(inplace=True))
        self._caches = (Fn.WeightCache(), Fn.WeightCache())

    def _half(self, i, x0, x1, pool=False, outc=None):
        """One conv + BatchNorm + ReLU.  pool: returns (y, maxpool2x2(y)) -- the skip tensor and the input of the next
        Down stage -- from one normalise pass when the fused kernels apply, from a separate max-pool otherwise.
        outc (the nn.Conv2d of OutConv): returns outc(y) as fp32 [T,B,H,W,out] -- from the normalise pass itself when
        there is one output channel (y is then never written), from the separate 1x1 kernels otherwise."""
        conv, bn = self.net[3 * i], self.net[3 * i + 1]
        T = x0.shape[0]
        training = self.training or not bn.track_running_stats
        if not training and not torch.is_grad_enabled() and ops.conv_affine_relu_ok(x0, x1, conv.out_channels):
            # inference (model.eval() under torch.no_grad()): BatchNorm folded into the conv epilogue -- one kernel
            # per conv instead of conv + finalize + normalise/ReLU pass (SURVEY.md section 8 f3)
            K = x0.shape[-1] + (0 if x1 is None else x1.shape[-1])
            self._caches[i].begin_forward(False)
            wp = self._caches[i].get(("fwd", x0.dtype, K), (conv.weight,),
                                     lambda: ops.pack_conv_weight(conv.weight, x0.dtype, K))
            scale, shift = self._caches[i].get(
                ("bn_eval",), (bn.weight, bn.bias, bn.running_mean, bn.running_var, conv.bias),
                lambda: ops.bn_eval_scale_shift(bn.weight.detach(), bn.bias.detach(), bn.running_mean, bn.running_var,
                                                bn.eps, conv.bias))
            y = ops.conv_affine_relu(Fn._c(x0), None if x1 is None else Fn._c(x1), wp, scale, shift,
                                     conv.kernel_size[0])
            if outc is not None:
                return Fn.OutConv1x1.apply(y, outc.weight, outc.bias)
            return Fn.PoolFork.apply(y) if pool else y
        # momentum=None is torch's cumulative moving average (factor 1 / num_batches_tracked): encoded for the finalize
        # kernel as -(n0 + 1), n0 = the count before this call (one BatchNorm call per timestep, so step t uses n0 + t + 1)
        if bn.momentum is not None:
            momentum = float(bn.momentum)
        else:
            momentum = -(float(bn.num_batches_tracked) + 1.0) if bn.track_running_stats else 0.0
        fuse_pool = pool and ops.bn_pool_ok(x0)
        fuse_out = outc is not None and ops.bn_outconv_ok(conv.out_channels, x0.dtype, outc.out_channels)
        y = Fn.ConvBnRelu.apply(x0, x1, conv.weight, conv.bias, bn.weight, bn.bias, bn.running_mean, bn.running_var,
                                training, bn.eps, momentum, self._caches[i], fuse_pool,
                                outc.weight if fuse_out else None, outc.bias if fuse_out else None)
        if training and bn.track_running_stats:
            bn.num_batches_tracked += T  # one BatchNorm call per timestep in the reference
        if outc is not None and not fuse_out:
            return Fn.OutConv1x1.apply(y, outc.weight, outc.bias)
        return Fn.PoolFork.apply(y) if (pool and not fuse_pool) else y

    def _seq(self, x0, x1=None, pool=False, outc=None):
        return self._half(1, self._half(0, x0, x1), None, pool, outc)

    def forward(self, x):
        _require_cuda(x, "DoubleConv")
        return _to_nchw(self._seq(_to_nhwc(x, _in_pad(x.shape[1]))))


class Down(nn.Module):
    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.net = nn.Sequential(nn.MaxPool2d(2), DoubleConv(in_ch, out_ch))

    def _seq(self, x):
        return self.net[1]._seq(Fn.MaxPool2.apply(x))

    def _seq_pooled(self, pooled, pool=False):
        """The DoubleConv of this stage on an input the previous stage already pooled (DoubleConv._seq(pool=True))."""
        return self.net[1]._seq(pooled, None, pool)

    def forward(self, x):
        _require_cuda(x, "Down")
        return _to_nchw(self._seq(_to_nhwc(x)))


class Up(nn.Module):
    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.up = nn.ConvTranspose2d(in_ch, in_ch // 2, 2, stride=2)
        self.conv = DoubleConv(in_ch, out_ch)
        self._cache = Fn.WeightCache()

    def _seq(self, x1, x2, outc=None):
        u = Fn.ConvT2x2.apply(x1, self.up.weight, self.up.bias, x2.shape[2], x2.shape[3], self._cache)
        return self.conv._seq(x2, u, False, outc)  # cat([skip, upsampled]) is virtual: two sources of one K loop

    def forward(self, x1, x2):
        _require_cuda(x1, "Up")
        return _to_nchw(self._seq(_to_nhwc(x1), _to_nhwc(x2)))


class OutConv(nn.Module):
    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.conv = nn.Conv2d(in_ch, out_ch, 1)

    def _seq(self, x):
        return Fn.OutConv1x1.apply(x, self.conv.weight, self.conv.bias)

    def forward(self, x):
        _require_cuda(x, "OutConv")
        return _to_nchw(self._seq(_to_nhwc(x)))


class SpatialAttention(nn.Module):
    """Optional bottleneck attention (reference unet.py:113-125): x * sigmoid(conv_k([mean_c x ; amax_c x])), on the
    kernels of csrc/attention.cu (kernel_size 1, 3, 5 or 7; any other size raises at the first call)."""

    def __init__(self, kernel_size=7):
        super().__init__()
        self.conv = nn.Conv2d(2, 1, kernel_size, padding=kernel_size // 2, bias=False)
        self.sigmoid = nn.Sigmoid()

    def _seq(self, x):
        """x [T,B,H,W,C] channels-last in the activation dtype -> the same shape and dtype."""
        return Fn.SpatialAttention.apply(x, self.conv.weight)

    def forward(self, x):
        _require_cuda(x, "SpatialAttention")
        return _to_nchw(self._seq(_to_nhwc(x)))


# -----------------------------------------------------------------------------------------------
# Temporal UNet (reference unet.py:131-204)
# -----------------------------------------------------------------------------------------------
class TemporalUNetDualView(nn.Module):
    def __init__(self, in_channels_per_sat=1, out_channels=1, base_ch=32, lstm_layers=1, use_skip_lstm=False,
                 use_attention=False):
        super().__init__()
        b = base_ch
        self.inc = DoubleConv(in_channels_per_sat * 2, b)
        self.down1 = Down(b, b * 2)
        self.down2 = Down(b * 2, b * 4)
        self.down3 = Down(b * 4, b * 8)
        self.bottleneck = Down(b * 8, b * 16)
        self.use_attention = use_attention
        if use_attention:
            self.attention = SpatialAttention()
        self.temporal = ConvLSTM(b * 16, b * 16, num_layers=lstm_layers)
        self.use_skip_lstm = use_skip_lstm
        if use_skip_lstm:
            self.lstm_skip3 = ConvLSTM(b * 8, b * 8)
            self.lstm_skip2 = ConvLSTM(b * 4, b * 4)
        self.up3 = Up(b * 16, b * 8)
        self.up2 = Up(b * 8, b * 4)
        self.up1 = Up(b * 4, b * 2)
        self.up0 = Up(b * 2, b)
        self.outc = OutConv(b, out_channels)

    def _encode(self, x):
        # every encoder output feeds a skip connection and the max-pool of the next stage: the stage that produces it
        # also pools it (one pass; the two gradients meet inside its BatchNorm backward)
        x0, p0 = self.inc._seq(x, None, True)
        x1, p1 = self.down1._seq_pooled(p0, True)
        x2, p2 = self.down2._seq_pooled(p1, True)
        x3, p3 = self.down3._seq_pooled(p2, True)
        xb = self.bottleneck._seq_pooled(p3)
        if self.use_attention:
            xb = self.attention._seq(xb)
        return xb, (x3, x2, x1, x0)

    def encode_once(self, x_t):
        """Reference-compatible single-frame encoder (unet.py:161-172): NCHW in, NCHW out."""
        _require_cuda(x_t, "TemporalUNetDualView.encode_once")
        xb, skips = self._encode(_to_nhwc(x_t, _in_pad(x_t.shape[1])))
        return _to_nchw(xb), tuple(_to_nchw(s) for s in skips)

    def _core(self, x, st, skip_st=None):
        """x [T,B,H,W,C] channels-last in the activation dtype -> (y fp32 [T,B,H,W,out], final (h, c) of every temporal
        layer, final (h, c) of lstm_skip3 and lstm_skip2).  st: initial NHWC state per temporal layer (or None);
        skip_st: the skip cells' initial states [(h, c) of lstm_skip3, (h, c) of lstm_skip2], None = zero (forward)."""
        xb, (x3, x2, x1, x0) = self._encode(x)
        hb, finals = self.temporal._seq(xb, st)
        skip_finals = []
        if self.use_skip_lstm:
            # forward: the skip LSTMs always start from a zero state and their final state is dropped (unet.py:190-191);
            # streaming inference (FrameStream) carries it from frame to frame
            x3, f3 = self.lstm_skip3._seq(x3, None if skip_st is None else [skip_st[0]])
            x2, f2 = self.lstm_skip2._seq(x2, None if skip_st is None else [skip_st[1]])
            skip_finals = f3 + f2

        d3 = self.up3._seq(hb, x3)
        d2 = self.up2._seq(d3, x2)
        d1 = self.up1._seq(d2, x1)
        # the last DoubleConv and the 1x1 output convolution: fp32 [T,B,H,W,out]; with one output channel the normalise
        # pass of the DoubleConv produces it directly (the 64-channel full-resolution activation is never written)
        y = self.up0._seq(d1, x0, self.outc.conv)
        return y, finals, skip_finals

    def forward(self, x_seq, state=None):
        _require_cuda(x_seq, "TemporalUNetDualView")
        B, T, C, H, W = x_seq.shape
        act = ops.act_dtype()
        # [B,T,C,H,W] fp32 -> [T,B,H,W,C] channels-last (input channels zero-padded in bf16 mode)
        x = Fn.permute_cast(x_seq, (1, 0, 3, 4, 2), act, _in_pad(C))
        y, finals, _ = self._core(x, None if state is None else _state_to_nhwc(state, act))

        # list of T frames as views of one buffer.  unbind, not T x select: the backward of unbind stacks the T frame
        # gradients in one pass; T selects each materialise a full-size zero tensor that autograd then adds up
        # (59 element-wise launches over the whole output map per step at T = 20)
        if y.shape[-1] == 1:
            out_seq = list(y.view(T, B, 1, H, W).unbind(0))  # C == 1: NHWC and NCHW coincide
        else:
            out_seq = list(Fn.permute_cast(y, (0, 1, 4, 2, 3), torch.float32).unbind(0))
        return out_seq, _state_to_nchw(finals)

    def stream(self, state=None):
        """Streaming inference, one frame at a time with every ConvLSTM state carried (unet_convlstm_b200/stream.py):
        for an eval-mode model under no_grad, [s.step(x[:, t]) for t in range(T)] and s.state equal model(x, state)."""
        from unet_convlstm_b200.stream import FrameStream
        return FrameStream(self, state)


def _state_to_nhwc(state, act):
    """forward's `state` ([(h, c)] NCHW per temporal layer, entries may be None) -> NHWC (h: act dtype, c: fp32)."""
    return [None if s is None or s[0] is None else
            (Fn.permute_cast(s[0], (0, 2, 3, 1), act), Fn.permute_cast(s[1], (0, 2, 3, 1), torch.float32))
            for s in state]


def _state_to_nchw(finals):
    """[(h, c)] NHWC -> the [(h, c)] NCHW fp32 state forward returns."""
    return [(Fn.permute_cast(h, (0, 3, 1, 2), torch.float32), Fn.permute_cast(c, (0, 3, 1, 2), torch.float32))
            for h, c in finals]


# -----------------------------------------------------------------------------------------------
# Dataset (host-side data preparation; reference unet.py:208-327).  Not a kernel: kept because the
# reference's scripts import it from this module.
# -----------------------------------------------------------------------------------------------
class NPZSequenceDataset(Dataset):
    """NPZ with X [N,T,2,H,W] radiances and Y [N,T,1,H,W] velocities.  Items are
    (x / max(x_max, 1), y mapped through clip -> asinh|signed_log -> affine to [-1,1], cloud mask of raw x)."""

    def __init__(self, npz_path, lower_percentile=0.00001, upper_percentile=99.99999, clip_outliers=True,
                 min_y=-7.5987958908081055, max_y=8.784920692443848, y_transform='asinh', y_transform_scale=None,
                 y_transform_percentile=99):
        data = np.load(npz_path)
        self.X = data["X"].astype(np.float32)
        self.Y = data["Y"].astype(np.float32)
        self.N, self.T, _, self.H, self.W = self.X.shape
        self.x_max = np.max(self.X)
        self.norm_const = max(self.x_max, 1.0)
        explicit = (min_y is not None) and (max_y is not None)
        if explicit:
            self.min_vel, self.max_vel = float(min_y), float(max_y)
        else:
            self.min_vel = np.percentile(self.Y, lower_percentile)
            self.max_vel = np.percentile(self.Y, upper_percentile)
        self.clip_outliers = clip_outliers
        self.y_transform = y_transform
        if y_transform_scale is not None:
            self.y_scale = float(y_transform_scale)
        elif y_transform_percentile is not None:
            self.y_scale = float(np.percentile(np.abs(self.Y), y_transform_percentile))
        else:
            self.y_scale = 1.0
        if explicit:
            self.trans_min, self.trans_max = self._transform(self.min_vel), self._transform(self.max_vel)
        else:
            yt = self._transform(self.Y)
            self.trans_min, self.trans_max = np.percentile(yt, lower_percentile), np.percentile(yt, upper_percentile)
        if self.trans_max == self.trans_min:
            self.trans_max = self.trans_min + 1.0
            print("[WARN] Transformed Y max equals min; adjusted to avoid division by zero.")
        print(f"[INFO] Dataset Loaded. X Range: [0.0, {self.x_max:.2f}]")
        print(f"[INFO] Y Normalization ({'explicit' if explicit else 'percentile'}); transform={self.y_transform} "
              f"scale={self.y_scale:.3f} -> trans_range: [{self.trans_min:.3f}, {self.trans_max:.3f}]")

    def _transform(self, arr):
        if self.y_transform == 'asinh':
            return np.arcsinh(arr / self.y_scale)
        if self.y_transform == 'signed_log':
            return np.sign(arr) * np.log1p(np.abs(arr) / self.y_scale)
        return arr

    def __len__(self):
        return self.N

    def __getitem__(self, idx):
        x = torch.from_numpy(self.X[idx])
        mask = (x[:, 0:1] > 1.1).float()  # on raw radiances, before normalisation
        x = x / self.norm_const
        y = self.Y[idx]
        if self.clip_outliers:
            y = np.clip(y, self.min_vel, self.max_vel)
        y = 2 * (self._transform(y) - self.trans_min) / (self.trans_max - self.trans_min) - 1.0
        return x, torch.from_numpy(y.astype(np.float32)), mask

    def denormalize(self, y_norm):
        is_torch = isinstance(y_norm, torch.Tensor)
        if is_torch:
            y_norm = y_norm.cpu().numpy()
        yt = (y_norm + 1.0) / 2.0 * (self.trans_max - self.trans_min) + self.trans_min
        if self.y_transform == 'asinh':
            y = np.sinh(yt) * self.y_scale
        elif self.y_transform == 'signed_log':
            y = np.sign(yt) * (np.expm1(np.abs(yt)) * self.y_scale)
        else:
            y = yt
        return torch.from_numpy(y) if is_torch else y
