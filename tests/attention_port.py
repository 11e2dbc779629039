"""fp64 CPU reference of TemporalUNetDualView(use_attention=True) for tests/test_attention.py and
tests/test_gpu_attention.py.

oracle/torch_port.py restates the reference's forward for use_attention=False.  temporal_unet below is the same forward
built from that port's block functions, with the reference's SpatialAttention (unet.py:113-125) applied to the
bottleneck output of every frame before the temporal ConvLSTM (unet.py:169-170) when p holds attention.conv.weight.
Without that key it computes exactly what oracle.torch_port.temporal_unet computes (tests/test_attention.py checks
both)."""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import torch_port as TP


class RefSpatialAttention(nn.Module):
    """The reference's module (unet.py:113-125), NCHW: the specification of the kernels."""

    def __init__(self, kernel_size=7):
        super().__init__()
        self.conv = nn.Conv2d(2, 1, kernel_size, padding=kernel_size // 2, bias=False)
        self.sigmoid = nn.Sigmoid()

    def forward(self, x):
        pooled = torch.cat([x.mean(dim=1, keepdim=True), x.amax(dim=1, keepdim=True)], dim=1)
        return x * self.sigmoid(self.conv(pooled))


def port_attention(w, x):
    """SpatialAttention.forward as a function of its weight w [1, 2, k, k]; x NCHW."""
    pooled = torch.cat([x.mean(dim=1, keepdim=True), x.amax(dim=1, keepdim=True)], dim=1)
    return x * torch.sigmoid(F.conv2d(pooled, w, padding=w.shape[-1] // 2))


def temporal_unet(p, x_seq, state=None, training=True, track=True, attention=None):
    """TemporalUNetDualView.forward (unet.py:174-204) on the blocks of oracle/torch_port.py, with the bottleneck attention
    when p holds attention.conv.weight.  attention: a callable NCHW -> NCHW used instead of port_attention (a check
    against another statement of the module).  Returns (list of T tensors [B,out,H,W], new_state)."""
    T = x_seq.shape[1]
    use_skip = "lstm_skip3.layers.0.conv.weight" in p
    if attention is None and "attention.conv.weight" in p:
        w = p["attention.conv.weight"]
        attention = lambda x: port_attention(w, x)  # noqa: E731
    bott, skips = [], []
    for t in range(T):
        x0 = TP.double_conv(p, "inc.net", x_seq[:, t], training, track)
        x1 = TP.down(p, "down1", x0, training, track)
        x2 = TP.down(p, "down2", x1, training, track)
        x3 = TP.down(p, "down3", x2, training, track)
        xb = TP.down(p, "bottleneck", x3, training, track)
        bott.append(xb if attention is None else attention(xb))
        skips.append([x3, x2, x1, x0])
    hb, new_state = TP.convlstm(p, "temporal", bott, state)
    if use_skip:
        s3, _ = TP.convlstm(p, "lstm_skip3", [s[0] for s in skips])
        s2, _ = TP.convlstm(p, "lstm_skip2", [s[1] for s in skips])
        for t in range(T):
            skips[t][0], skips[t][1] = s3[t], s2[t]
    out = []
    for t in range(T):
        x3, x2, x1, x0 = skips[t]
        d = TP.up(p, "up3", hb[t], x3, training, track)
        d = TP.up(p, "up2", d, x2, training, track)
        d = TP.up(p, "up1", d, x1, training, track)
        d = TP.up(p, "up0", d, x0, training, track)
        out.append(F.conv2d(d, p["outc.conv.weight"], p["outc.conv.bias"]))
    return out, new_state
