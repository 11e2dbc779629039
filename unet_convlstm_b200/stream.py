"""Streaming inference of TemporalUNetDualView: frames arrive one at a time, every ConvLSTM state is carried.

`model(x[:, t:t+1], state)` carries only the temporal cell's (h, c): the skip cells lstm_skip3 / lstm_skip2 restart
from zero on every call (the reference's forward, unet.py:190-191), so calling it frame by frame does not compute what
`model(x)` computes.  The only exact online method was to re-run the whole prefix for every new frame, O(T^2).
FrameStream carries the state of every ConvLSTM layer in buffers it owns, so frame t costs one frame:

    s = model.stream()                    # model.eval(); optional state seeds the temporal layers, as forward's
    ys = [s.step(x[:, t]) for t in range(T)]
    # ys[t] == model(x)[0][t] and s.state == model(x)[1]

Per frame it runs the model's own stage functions at T = 1 (TemporalUNetDualView._core).  Frame 0 of a sequence runs
eagerly (a zero initial state skips the h half of the first gate convolution, as step 0 of the full sequence does);
frame 1 runs eagerly on the stream the capture will use, which packs the weights, encodes the TMA tensor maps and
sizes the split-K workspace there; from frame 2 on every frame is one replay of a CUDA graph with a private memory
pool, which ends by copying the frame's new h / c over the carried ones.  Inside the stream, bf16 single-frame
convolutions with few M tiles run split over K (ops.split_k_routing, b200_splitk_splits).
"""
from __future__ import annotations

import torch

from . import functional as Fn
from . import ops


class FrameStream:
    """Frame-by-frame inference of an eval-mode TemporalUNetDualView (see the module docstring).

    step(x_t): x_t [B, C_in, H, W] -> [B, out_channels, H, W] fp32.  state: the temporal layers' [(h, c), ...] NCHW fp32,
    the format forward returns and accepts.  reset(state=None) starts a new sequence.  The model is bound at the first
    frame after a reset: a parameter or buffer changed after that (in-place op, load_state_dict, optimizer step) makes
    step() raise until reset() is called."""

    def __init__(self, model, state=None):
        self.model = model
        self._cs = None       # the capture stream (created at the first CUDA warm-up frame)
        self._sig = None      # (shape, dtype, device, precision mode) of the first frame
        self._bound = None    # parameter / buffer versions and optimizer generation at the first frame
        self._drop_graph()
        self.reset(state)

    def _drop_graph(self):
        self._carry = None    # NHWC (h, c) of every ConvLSTM layer: the temporal layers, then lstm_skip3, lstm_skip2
        self._graph = None
        self._x = None        # static input of the graph
        self._y = None        # static output of the graph

    def reset(self, state=None):
        """Starts a new sequence; `state` seeds the temporal layers (the skip cells start from zero, as in forward).
        A sequence whose first frame has the shape, dtype and device of the previous one, under unchanged weights and
        precision mode, keeps the captured graph: its frames from the second on are replays."""
        self._state0 = None if state is None else list(state)
        self._frames = 0

    @property
    def state(self):
        if self._frames == 0:
            return self._state0
        from train.unet import _state_to_nchw
        return _state_to_nchw(self._carry[:len(self.model.temporal.layers)])

    def _stamp(self):
        m = self.model
        return Fn.WeightCache._stamp(list(m.parameters()) + list(m.buffers()), Fn._OPT_GENERATION[0])

    def step(self, x_t: torch.Tensor) -> torch.Tensor:
        from train.unet import _require_cuda
        m = self.model
        if m.training:
            raise RuntimeError("FrameStream.step: the model is in training mode; streaming inference needs model.eval() "
                               "(per-frame batch statistics and running-statistics updates are not supported)")
        _require_cuda(x_t, "FrameStream.step")
        if x_t.dim() != 4:
            raise RuntimeError(f"FrameStream.step: expected one frame [B, C, H, W], got shape {tuple(x_t.shape)}")
        sig = (tuple(x_t.shape), x_t.dtype, x_t.device, ops.get_precision())
        if self._frames == 0:
            stamp = self._stamp()
            if (sig, stamp) != (self._sig, self._bound):   # a new binding: buffers and graph are rebuilt
                self._sig, self._bound = sig, stamp
                self._drop_graph()
        elif sig != self._sig:
            raise RuntimeError(f"FrameStream.step: frame (shape, dtype, device, precision) {sig} differs from the first "
                               f"frame of this sequence {self._sig}; call reset() to start a new sequence")
        elif self._stamp() != self._bound:
            raise RuntimeError("FrameStream.step: a parameter or buffer of the model changed since this stream bound it "
                               "at its first frame; call reset()")
        with torch.no_grad(), ops.split_k_routing():
            if self._frames == 0:
                y = self._first(x_t)
            elif self._graph is None and (self._frames == 1 or not x_t.is_cuda):
                y = self._eager(x_t)
            else:
                y = self._replay(x_t)
        self._frames += 1
        return y

    # ---------------------------------------------------------------------------------------------------------------
    def _run(self, x, st, skip_st):
        """One frame through the model's stages at T = 1: ([B, out, H, W] fp32, final NHWC (h, c) of every layer)."""
        from train.unet import _in_pad
        B, C, H, W = x.shape
        xs = Fn.permute_cast(x.unsqueeze(1), (1, 0, 3, 4, 2), ops.act_dtype(), _in_pad(C))
        y, finals, skip_finals = self.model._core(xs, st, skip_st)
        out = y.view(B, 1, H, W) if y.shape[-1] == 1 else Fn.permute_cast(y[0], (0, 3, 1, 2), torch.float32)
        return out, list(finals) + list(skip_finals)

    def _step_carried(self, x):
        """A frame from the carried states; the new states are copied over them."""
        L = len(self.model.temporal.layers)
        out, new = self._run(x, self._carry[:L], self._carry[L:] or None)
        for (h, c), (nh, nc) in zip(self._carry, new):
            ops.copy_(h, nh)
            ops.copy_(c, nc)
        return out

    def _first(self, x_t):
        """Frame 0, eager: the given initial state of the temporal layers (or zero), zero skip-cell states."""
        from train.unet import _state_to_nhwc
        st = None if self._state0 is None else _state_to_nhwc(self._state0, ops.act_dtype())
        out, new = self._run(x_t, st, None)
        if self._carry is None:
            self._carry = [(torch.empty(nh.shape, device=nh.device, dtype=nh.dtype),
                            torch.empty(nc.shape, device=nc.device, dtype=nc.dtype)) for nh, nc in new]
        for (h, c), (nh, nc) in zip(self._carry, new):
            ops.copy_(h, nh)
            ops.copy_(c, nc)
        return out

    def _eager(self, x_t):
        """Frame 1 (the warm-up of the capture): eager, on the capture stream.  Without a device (host dry runs with the
        device checks stubbed) every frame after the first takes this path."""
        if not x_t.is_cuda:
            return self._step_carried(x_t)
        self._x = torch.empty_like(x_t)
        ops.copy_(self._x, x_t)
        cur = torch.cuda.current_stream(x_t.device)
        if self._cs is None or self._cs.device != x_t.device:
            self._cs = torch.cuda.Stream(device=x_t.device)
        self._cs.wait_stream(cur)
        with torch.cuda.stream(self._cs):
            out = self._step_carried(self._x)
        cur.wait_stream(self._cs)
        out.record_stream(cur)
        return out

    def _replay(self, x_t):
        ops.copy_(self._x, x_t)
        if self._graph is None:
            # splitk_workspace cannot grow during the capture: frame 1 ran the same shapes on this stream already
            self._graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph, stream=self._cs):
                self._y = self._step_carried(self._x)
        self._graph.replay()
        out = torch.empty(self._y.shape, device=self._y.device, dtype=self._y.dtype)
        ops.copy_(out, self._y)
        return out
