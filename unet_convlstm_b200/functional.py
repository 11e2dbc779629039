"""Autograd functions of the hot path on NHWC sequence tensors [T, B, H, W, C].

Each Function's forward/backward is a short sequence of launches of our CUDA kernels (ops.py);
the backward formulas are the hand-derived autograd of the reference modules in train/unet.py
(dordanino12/unet-convlstm), cited per class.
"""
from __future__ import annotations

import weakref

import torch

from . import ops


# Every torch.optim.Optimizer.step() -- including the FUSED implementations (`torch._fused_adamw_` ...), which update
# parameters WITHOUT touching their version counters -- bumps this generation through a global post-step hook.
_OPT_GENERATION = [0]


def _bump_generation(*_a, **_k):
    _OPT_GENERATION[0] += 1


from torch.optim.optimizer import register_optimizer_step_post_hook as _reg_step_hook  # noqa: E402

_reg_step_hook(_bump_generation)


_CACHES = weakref.WeakSet()   # every WeightCache alive (pack_refresh_plan)


def pack_refresh_plan(updated):
    """For an optimizer about to update the parameters `updated` ({data_ptr: tensor}): the packed copies it can emit
    itself.  Returns (packs, redo, entries): packs = {data_ptr: [geometry of ops._pack, ...]} for b200_adamw_pack,
    redo = closures to run after the update (small derived tensors: the gate-interleaved bias), entries = the cache
    entries all of whose recipes are covered -- pass them to pack_refresh_commit() after the update.  Only entries that
    are valid right now and derive from nothing but the parameters in `updated` qualify; everything else is left to the
    version / generation check of WeightCache.get()."""
    packs, redo, entries = {}, [], []
    for cache in list(_CACHES):
        for ent in cache._d.values():
            ver, _, recipes, params = ent
            if not recipes or ver != WeightCache._stamp(params, _OPT_GENERATION[0]):
                continue
            ok = all((r[0] == "pack" and _same(updated.get(r[1].data_ptr()), r[1])) or
                     (r[0] == "redo" and all(_same(updated.get(q.data_ptr()), q) for q in r[1])) for r in recipes)
            if not ok:
                continue
            for r in recipes:
                if r[0] == "pack":
                    packs.setdefault(r[1].data_ptr(), []).append(r[2])
                else:
                    redo.append(r[2])
            entries.append(ent)
    return packs, redo, entries


def _same(p, w):
    return p is not None and p.numel() == w.numel() and p.dtype == w.dtype


def pack_refresh_commit(entries):
    """The packed values of `entries` now hold the updated parameters: stamp them with the parameter versions as they
    are now and with the optimizer generation the post-step hook (_bump_generation) is about to set."""
    for ent in entries:
        ent[0] = WeightCache._stamp(ent[3], _OPT_GENERATION[0] + 1)


class WeightCache:
    """Packed (GEMM-layout, activation-dtype) copies of a module's parameters, rebuilt when the parameter changes.
    Two signals: the tensor version (in-place torch ops, load_state_dict, this package's optimizer) and the optimizer
    generation above (any torch optimizer step).  Round 1 instead emptied the cache at the first forward after a
    backward; a no-grad forward between backward and optimizer.step() consumed that flag and the next training
    forward used stale packed weights (ADVICE r01) -- the generation counter has no such window, and an evaluation
    loop after training keeps its packed weights."""

    def __init__(self):
        self._d = {}          # key -> [version stamp, value, recipes (ops._PACK_RECORDER), params]
        self._open = 0        # forward passes (with a graph) whose backward has not run yet
        self._shared = False  # the parameters were used more than once in the graph(s) still open
        _CACHES.add(self)

    def begin_forward(self, differentiated: bool) -> bool:
        """Call at the top of every forward pass, BEFORE the first get().  Returns `differentiated`."""
        if differentiated:
            self._open += 1
            if self._open > 1:
                self._shared = True
        return differentiated

    def note_backward(self) -> bool:
        """True if this backward is the ONLY gradient contribution the parameters receive in this pass (autograd sums
        several contributions on the current stream, which rules out producing one of them on the background
        stream, ops.background)."""
        single = not self._shared
        self._open = max(0, self._open - 1)
        if self._open == 0:
            self._shared = False
        return single

    @staticmethod
    def _stamp(params, generation):
        return (generation,) + tuple((p.data_ptr(), p._version) for p in params if p is not None)

    def get(self, key, params, builder):
        ver = self._stamp(params, _OPT_GENERATION[0])
        hit = self._d.get(key)
        if hit is not None and hit[0] == ver:
            return hit[1]
        recipes = []
        prev, ops._PACK_RECORDER = ops._PACK_RECORDER, recipes
        try:
            val = builder()
        finally:
            ops._PACK_RECORDER = prev
        self._d[key] = [ver, val, recipes, tuple(params)]
        return val

    def clear(self):
        self._d.clear()


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


def _count_use(ctx, cache) -> bool:
    """Top of a Function.forward: drops packed weights a finished backward (hence possibly an optimizer step) has
    outdated, and registers the pass if it will be differentiated (see WeightCache.note_backward)."""
    return cache.begin_forward(any(ctx.needs_input_grad))


# ------------------------------------------------------------------------------------------------
# layout changes at the module boundary (reference tensors are NCHW fp32)
# ------------------------------------------------------------------------------------------------
class PermuteCast(torch.autograd.Function):
    """y = x.permute(perm) as a contiguous tensor of `dtype`, last dim zero-padded to `pad_to`."""

    @staticmethod
    def forward(ctx, x, perm, dtype, pad_to):
        xv = x.permute(*perm)
        C = xv.shape[-1]
        Cp = C if pad_to is None else max(C, pad_to)
        shape = tuple(xv.shape[:-1]) + (Cp,)
        y = (torch.zeros if Cp != C else torch.empty)(shape, device=x.device, dtype=dtype)
        ops.copy_(y[..., :C], xv)
        ctx.perm, ctx.C, ctx.xdtype, ctx.xshape = perm, C, x.dtype, x.shape
        return y

    @staticmethod
    def backward(ctx, dy):
        inv = [0] * len(ctx.perm)
        for i, p in enumerate(ctx.perm):
            inv[p] = i
        dx = torch.empty(ctx.xshape, device=dy.device, dtype=ctx.xdtype)
        ops.copy_(dx, dy[..., :ctx.C].permute(*inv))
        return dx, None, None, None


def permute_cast(x, perm, dtype, pad_to=None):
    return PermuteCast.apply(x, tuple(perm), dtype, pad_to)


# ------------------------------------------------------------------------------------------------
# conv3x3 + BatchNorm + ReLU (one half of DoubleConv, unet.py:66-75)
# ------------------------------------------------------------------------------------------------
class ConvBnRelu(torch.autograd.Function):
    """y = relu(bn(conv3x3([x0 ; x1]) + bias)).  The channel concat of Up (unet.py:98) is virtual:
    the GEMM K loop reads x0 then x1.  BatchNorm statistics are per timestep (unet.py:179-182).

    pool=True returns (y, maxpool2x2(y)) -- an encoder output that feeds a skip connection and the MaxPool2d of the
    next Down stage (unet.py:81, 179-182 -> 196-202): the normalise/ReLU pass writes the pooled tensor too, and in
    backward the sum of the skip gradient and the routed pool gradient is formed inside the BatchNorm-backward
    passes instead of by a max-pool backward kernel (ops.bn_relu_fwd / bn_relu_bwd)."""

    @staticmethod
    def forward(ctx, x0, x1, weight, bias, gamma, beta, rm, rv, training, eps, momentum, cache, pool=False,
                out_w=None, out_b=None):
        """out_w [1, N, 1, 1] / out_b [1] (OutConv, unet.py:101-107, one output channel): returns
        outconv(relu(bn(conv))) as fp32 [T,B,H,W,1] from the normalise pass; the activation is not materialised."""
        ctx.counted = _count_use(ctx, cache)
        ctx.set_materialize_grads(False)   # an unused output (skip or pooled) arrives as None, not as a zero tensor
        x0 = _c(x0)
        x1 = None if x1 is None else _c(x1)
        dt = x0.dtype
        T, B, H, W, C0 = x0.shape
        C1 = 0 if x1 is None else x1.shape[-1]
        N, K = weight.shape[0], weight.shape[1]
        ks = weight.shape[2]
        if K > C0 + C1 or (x1 is not None and K != C0 + C1):
            raise ValueError(f"conv weight expects {K} input channels, got {C0}+{C1}")
        z = torch.empty((T, B, H, W, N), device=x0.device, dtype=dt)
        wp = cache.get(("fwd", dt, C0 + C1), (weight,), lambda: ops.pack_conv_weight(weight, dt, C0 + C1))
        # The BatchNorm sums CAN come out of the conv epilogue (b200_conv_bnstats_tc_fwd), but measured on
        # B200 the cross-lane column reduction makes the epilogue of the narrow layers longer than their
        # main loop (K64->N64 @64x64: +1.05 ms per call against 0.65 ms for the separate HBM-bound
        # b200_bn_stats pass, profiles/r01_fused_bn_stats_measured.txt), so it is opt-in.
        ws = torch.empty((2, T, N), device=x0.device, dtype=torch.float64) if (training and ops.FUSE_BN_STATS) else None
        fused = ops.conv_fwd(x0, x1, wp, bias.detach() if bias is not None else None, ks, z, bn_ws=ws)
        outconv = None
        if out_w is not None:
            outconv = (out_w.detach().reshape(-1), None if out_b is None else out_b.detach())
        y, stats = ops.bn_relu_fwd(z, gamma.detach(), beta.detach(), rm, rv, training, eps, momentum,
                                   ws=ws if fused else None, pool=pool, outconv=outconv)
        ctx.save_for_backward(x0, x1, z, weight, gamma, *stats[:4], out_w)
        ctx.tstride = stats[4]
        ctx.training, ctx.cache, ctx.has_bias = training, cache, bias is not None
        ctx.has_out_b = out_b is not None
        return y

    @staticmethod
    def backward(ctx, dy, dpool=None):
        x0, x1, z, weight, gamma, mean, rstd, scale, shift, out_w = ctx.saved_tensors
        single = ctx.cache.note_backward() if ctx.counted else True
        dt = z.dtype

        def as_act(g):
            if g is None:
                return None
            g = _c(g)
            return g if g.dtype == dt else g.to(dt)

        d_out_w = d_out_b = None
        if out_w is not None:
            if dy is None:
                return (None,) * 15
            dy = _c(dy).float()                 # gradient of the 1x1 convolution's output, fp32 [T,B,H,W,1]
        else:
            dy, dpool = as_act(dy), as_act(dpool)
            if dy is None and dpool is None:
                return (None,) * 15
        T, B, H, W, N = z.shape
        C0 = x0.shape[-1]
        C1 = 0 if x1 is None else x1.shape[-1]
        K, ks = weight.shape[1], weight.shape[2]
        # the conv-bias gradient comes out of the BatchNorm sums in closed form (zero in training mode)
        if out_w is not None:
            dz, dgamma, dbeta, dbias, dwo = ops.bn_relu_bwd(z, dy, (mean, rstd, scale, shift, ctx.tstride), ctx.training,
                                                            ctx.has_bias, outconv_w=out_w.detach().reshape(-1))
            d_out_w = dwo.view_as(out_w)
            if ctx.has_out_b:
                d_out_b = ops.colsum(dy.numel(), dy, 1)
        else:
            dz, dgamma, dbeta, dbias = ops.bn_relu_bwd(z, dy, (mean, rstd, scale, shift, ctx.tstride), ctx.training,
                                                       ctx.has_bias, dpool=dpool)
        # weight gradient, batched over all T*B images
        def wgrad():
            dwp = torch.zeros((ks * ks, N, C0 + C1), device=z.device, dtype=torch.float32)
            ops.conv_wgrad(dz, x0, ks, dwp, 0)
            if x1 is not None:
                ops.conv_wgrad(dz, x1, ks, dwp, C0)
            return ops.unpack_conv_wgrad(dwp, K)

        def dgrad():
            # data gradient, split over the two sources of the virtual concat
            wd = ctx.cache.get(("dgrad", dt, C0 + C1), (weight,),
                               lambda: _dgrad_pack_padded(weight, dt, C0 + C1))
            d0 = torch.empty_like(x0)
            d1 = torch.empty_like(x1) if x1 is not None else None
            ops.conv_fwd(dz, None, wd, None, ks, d0, d1)
            return d0, d1

        dx0 = dx1 = None
        need0, need1 = ctx.needs_input_grad[0], (x1 is not None and ctx.needs_input_grad[1])
        bg = ops.background(weight, dz, x0, x1, allow=single and ctx.needs_input_grad[2])
        if bg.active and (need0 or need1):
            dx0, dx1 = dgrad()     # the critical path first: the background wgrad takes the SMs the dgrad frees
        dweight = None
        if ctx.needs_input_grad[2]:          # frozen weights (fine-tuning a decoder): no weight-gradient GEMM
            with bg:
                dweight = wgrad()
                bg.keep(dweight)
        if not bg.active and (need0 or need1):
            dx0, dx1 = dgrad()
        return dx0, dx1, dweight, dbias, dgamma, dbeta, None, None, None, None, None, None, None, d_out_w, d_out_b


def _dgrad_pack_padded(weight, dt, Kp):
    """Data-gradient weights [taps, Kp, N]; rows >= K (zero-padded input channels) stay zero."""
    return ops.pack_conv_weight_dgrad(weight, dt, Kp)


# ------------------------------------------------------------------------------------------------
# 2x2 max-pool (Down, unet.py:78-84)
# ------------------------------------------------------------------------------------------------
class MaxPool2(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x = _c(x)
        y = ops.maxpool2_fwd(x)
        ctx.save_for_backward(x)
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        return ops.maxpool2_bwd(x, _c(dy).to(x.dtype))


class PoolFork(torch.autograd.Function):
    """(skip, pooled) = (x, maxpool2(x)) for an encoder output that feeds both the next Down stage and a skip
    connection (unet.py:179-182 -> :196-202).  Autograd would sum the two gradients of x with an extra element-wise
    pass (2 reads + 1 write of the largest activation tensors); here the max-pool backward ADDS its routed gradient
    into the skip gradient in place (1 extra read)."""

    @staticmethod
    def forward(ctx, x):
        x = _c(x)
        y = ops.maxpool2_fwd(x)
        ctx.save_for_backward(x)
        return x.view_as(x), y

    @staticmethod
    def backward(ctx, g_skip, g_pool):
        (x,) = ctx.saved_tensors
        if g_pool is None:
            return g_skip
        g_pool = _c(g_pool).to(x.dtype)
        if g_skip is None:
            return ops.maxpool2_bwd(x, g_pool)
        if g_skip.dtype != x.dtype or not g_skip.is_contiguous():
            g_skip = g_skip.to(x.dtype).contiguous()
        return ops.maxpool2_bwd(x, g_pool, accumulate_into=g_skip)


# ------------------------------------------------------------------------------------------------
# ConvTranspose2d(k=2, stride=2) + F.pad to the skip size (Up, unet.py:90-97)
# ------------------------------------------------------------------------------------------------
class ConvT2x2(torch.autograd.Function):
    """A GEMM [P, Cin] x [Cin, 4*Cout] followed by a pixel shuffle (each input pixel produces a 2x2
    output patch, no overlap)."""

    @staticmethod
    def forward(ctx, x, weight, bias, Hd, Wd, cache):
        ctx.counted = _count_use(ctx, cache)
        x = _c(x)
        dt = x.dtype
        T, B, H, W, Cin = x.shape
        Cout = weight.shape[1]
        wf, _ = cache.get(("convT", dt), (weight,), lambda: ops.pack_convT_weight(weight, dt))
        y = ops.convT2x2_fwd(x, wf, bias.detach() if bias is not None else None, Cout, Hd, Wd)
        ctx.save_for_backward(x, weight)
        ctx.cache, ctx.has_bias, ctx.bias = cache, bias is not None, bias
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        single = ctx.cache.note_backward() if ctx.counted else True
        dt = x.dtype
        T, B, H, W, Cin = x.shape
        Cout = weight.shape[1]
        du = ops.unshuffle2x2(_c(dy).to(dt), H, W)  # [T,B,H,W,4*Cout]
        dx = None
        if ctx.needs_input_grad[0]:
            _, wb = ctx.cache.get(("convT", dt), (weight,), lambda: ops.pack_convT_weight(weight, dt))
            dx = torch.empty_like(x)
            ops.conv_fwd(du, None, wb, None, 1, dx)
        with ops.background((weight, ctx.bias), du, x, allow=single) as bg:
            dbias = ops.colsum(T * B * H * W * 4, du, Cout) if ctx.has_bias else None
            dwp = torch.zeros((1, 4 * Cout, Cin), device=x.device, dtype=torch.float32)
            ops.conv_wgrad(du, x, 1, dwp, 0)
            dweight = torch.empty_like(weight)
            ops.copy_(dweight.view(Cin, Cout, 4), dwp.view(4, Cout, Cin).permute(2, 1, 0))
            bg.keep(dweight, dbias)
        return dx, dweight, dbias, None, None, None


# ------------------------------------------------------------------------------------------------
# 1x1 output convolution (OutConv, unet.py:101-107), fp32 output
# ------------------------------------------------------------------------------------------------
class OutConv1x1(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias):
        x = _c(x)
        w2 = weight.detach().reshape(weight.shape[0], weight.shape[1])
        y = ops.outconv_fwd(x, w2, bias.detach() if bias is not None else None)
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        w2 = weight.detach().reshape(weight.shape[0], weight.shape[1])
        dx, dw, db = ops.outconv_bwd(x, w2, _c(dy).float(), ctx.needs_input_grad[0])
        return dx, dw.view_as(weight), (db if ctx.has_bias else None)


# ------------------------------------------------------------------------------------------------
# ConvLSTM layer over a whole sequence (ConvLSTMCell + the t-loop of ConvLSTM, unet.py:14-60)
# ------------------------------------------------------------------------------------------------
class ConvLSTMSeq(torch.autograd.Function):
    """h_seq, c_T = ConvLSTM layer(x_seq, h0, c0).

    Forward, per timestep: one fused kernel -- implicit-GEMM gate conv over the virtual concat
    [x_t ; h_{t-1}] on tcgen05 with the sigmoid/tanh gate math and the c/h update in the epilogue --
    or, in the fp32 check mode / for shapes the tensor-core path cannot tile, a CUDA-core conv plus
    the gate-math kernel.  h_t (activation dtype), c_t (fp32) and the activated gates are kept for BPTT.
    Backward: for t = T-1..0 the gate-gradient kernel and the data-gradient conv ([dx_t ; dh_{t-1}]);
    the weight gradient is ONE reduction over all T*B*H*W pixels after the sweep."""

    @staticmethod
    def forward(ctx, x_seq, h0, c0, weight, bias, cache):
        ctx.counted = _count_use(ctx, cache)
        x_seq = _c(x_seq)
        dt = x_seq.dtype
        T, B, H, W, Cin = x_seq.shape
        Ch = weight.shape[0] // 4
        ks = weight.shape[2]
        dev = x_seq.device
        if weight.shape[1] != Cin + Ch:
            raise ValueError(f"ConvLSTM weight expects {weight.shape[1]} input channels, got {Cin}+{Ch}")
        fused = ops.lstm_tc_ok(x_seq[0], Ch)
        h_all = torch.empty((T + 1, B, H, W, Ch), device=dev, dtype=dt)
        c_all = torch.empty((T + 1, B, H, W, Ch), device=dev, dtype=torch.float32)
        # gate recompute (ops.GATE_RECOMPUTE): the activated gates are not kept for backward
        recompute = bool(fused and dt == torch.bfloat16 and ops.GATE_RECOMPUTE and any(ctx.needs_input_grad))
        gates = None if recompute else torch.empty((T, B, H, W, 4 * Ch), device=dev, dtype=dt)
        have_h0 = h0 is not None
        if have_h0:
            ops.copy_(h_all[0], h0.detach())
            ops.copy_(c_all[0], c0.detach())
        elif not fused or recompute:
            h_all[0].zero_()      # the recompute pass reads slot 0 as h_{-1} = 0 / c_{-1} = 0
            c_all[0].zero_()
        if fused:
            wp, bp = cache.get(("lstm", dt), (weight, bias), lambda: ops.pack_lstm_weight(weight, bias, dt))
            if ops.PERSISTENT_LSTM and dt == torch.bfloat16:   # (the tf32 mode launches the fused cell per step)
                ops.lstm_seq_fwd_fused(x_seq, h_all, c_all, wp, bp, gates, have_h0, ks)
            else:
                for t in range(T):
                    first_zero = (t == 0 and not have_h0)
                    ops.lstm_cell_fwd_fused(x_seq[t], None if first_zero else h_all[t],
                                            None if first_zero else c_all[t], wp, bp, c_all[t + 1], h_all[t + 1],
                                            None if gates is None else gates[t], ks)
        else:
            wp = cache.get(("fwd", dt, Cin + Ch), (weight,), lambda: ops.pack_conv_weight(weight, dt))
            zbuf = torch.empty((B, H, W, 4 * Ch), device=dev, dtype=torch.float32)
            bd = bias.detach() if bias is not None else None
            for t in range(T):
                first_zero = (t == 0 and not have_h0)
                ops.lstm_cell_fwd_unfused(x_seq[t], h_all[t], None if first_zero else c_all[t], wp, bd,
                                          c_all[t + 1], h_all[t + 1], gates[t], ks, zbuf)
        ctx.save_for_backward(x_seq, weight)
        ctx.h_all, ctx.c_all, ctx.gates = h_all, c_all, gates
        ctx.have_h0, ctx.cache, ctx.has_bias, ctx.bias = have_h0, cache, bias is not None, bias
        h_seq = h_all[1:]
        c_T = c_all[T]
        ctx.mark_non_differentiable()
        return h_seq, c_T

    @staticmethod
    def backward(ctx, dh_seq, dc_T):
        x_seq, weight = ctx.saved_tensors
        h_all, c_all, gates = ctx.h_all, ctx.c_all, ctx.gates
        dt = x_seq.dtype
        T, B, H, W, Cin = x_seq.shape
        Ch = weight.shape[0] // 4
        ks = weight.shape[2]
        dev = x_seq.device
        dh_seq = None if dh_seq is None else _c(dh_seq).to(dt)
        dc_next = None if dc_T is None else _c(dc_T).float()
        wd = ctx.cache.get(("dgrad", dt, Cin + Ch), (weight,), lambda: ops.pack_conv_weight_dgrad(weight, dt))
        dz_all = torch.empty((T, B, H, W, 4 * Ch), device=dev, dtype=dt)
        if gates is None:
            # gate recompute: all T steps in one launch, into the buffer the gate-gradient kernel overwrites with dz
            # (element for element in place: every thread reads its four gates before it writes its four dz)
            wp, bp = ctx.cache.get(("lstm", dt), (weight, ctx.bias), lambda: ops.pack_lstm_weight(weight, ctx.bias, dt))
            ops.lstm_gates_recompute(x_seq, h_all, c_all, wp, bp, dz_all, ks)
            gates = dz_all
        need_dx = ctx.needs_input_grad[0]
        dx_seq = torch.empty_like(x_seq) if need_dx else None
        if ops.lstm_seq_bwd_ok(x_seq, Ch):
            # fused timestep-persistent BPTT: the gate gradients of the last step, then ONE cooperative
            # launch for t = T-1 .. 0 (dgrad conv of dz_t with the gate gradients of step t-1 in its epilogue)
            dc_buf = torch.empty((2, B, H, W, Ch), device=dev, dtype=torch.float32)
            want_dh0 = ctx.have_h0 and ctx.needs_input_grad[1]
            dh0 = torch.empty((B, H, W, Ch), device=dev, dtype=dt) if want_dh0 else None
            ops.lstm_gates_bwd(gates[T - 1], c_all[T - 1], c_all[T], None if dh_seq is None else dh_seq[T - 1], None,
                               dc_next, dz_all[T - 1], dc_buf[(T - 1) & 1])
            ops.lstm_seq_bwd_fused(dz_all, wd, gates, c_all, dh_seq, dc_buf, dx_seq, dh0, Cin, ctx.have_h0, ks)
            dc0 = dc_buf[0] if (ctx.have_h0 and ctx.needs_input_grad[2]) else None
            return ConvLSTMSeq._finish_backward(ctx, x_seq, weight, h_all, dz_all, dx_seq, dh0, dc0)
        dx_scratch = None if need_dx else torch.empty_like(x_seq[0])
        dh_rec = [torch.empty((B, H, W, Ch), device=dev, dtype=dt) for _ in range(2)]
        dc_buf = [torch.empty((B, H, W, Ch), device=dev, dtype=torch.float32) for _ in range(2)]
        dh_b = None
        # Weight gradient in chunks of timesteps on the background stream WHILE the sweep continues: the HBM-bound
        # gate-gradient kernel of every step leaves the tensor pipes idle, and the chunk already swept fills them.
        single = ctx.cache.note_backward() if ctx.counted else True
        chunk = ops.LSTM_WGRAD_CHUNK
        chunked = None
        if chunk > 0 and T > chunk and ops.background((weight, ctx.bias), allow=single).active:
            chunked = {"dwp": torch.zeros((ks * ks, 4 * Ch, Cin + Ch), device=dev, dtype=torch.float32), "hi": T}
        for t in reversed(range(T)):
            zero_prev = (t == 0 and not ctx.have_h0)
            ops.lstm_gates_bwd(gates[t], None if zero_prev else c_all[t], c_all[t + 1],
                               None if dh_seq is None else dh_seq[t], dh_b, dc_next, dz_all[t], dc_buf[t & 1])
            dc_next = dc_buf[t & 1]
            need_dh_prev = t > 0 or (ctx.have_h0 and (ctx.needs_input_grad[1]))
            if need_dh_prev:
                dxt = dx_seq[t] if need_dx else dx_scratch
                ops.conv_fwd(dz_all[t].unsqueeze(0), None, wd, None, ks, dxt.unsqueeze(0), dh_rec[t & 1].unsqueeze(0))
                dh_b = dh_rec[t & 1]
            elif need_dx:
                # only the x columns of the data gradient are needed at t = 0 with a zero initial state
                ops.conv_fwd(dz_all[t].unsqueeze(0), None, wd[:, :Cin, :].contiguous(), None, ks,
                             dx_seq[t].unsqueeze(0))
            if chunked is not None and t > 0 and (T - t) % chunk == 0:
                with ops.background((weight, ctx.bias), dz_all, x_seq, h_all, chunked["dwp"], allow=single):
                    ConvLSTMSeq._wgrad_range(ctx, x_seq, h_all, dz_all, chunked["dwp"], t, chunked["hi"], Cin, ks)
                chunked["hi"] = t
        dh0 = dc0 = None
        if ctx.have_h0:
            if ctx.needs_input_grad[1]:
                dh0 = dh_b
            if ctx.needs_input_grad[2]:
                dc0 = dc_next
        return ConvLSTMSeq._finish_backward(ctx, x_seq, weight, h_all, dz_all, dx_seq, dh0, dc0, single, chunked)

    @staticmethod
    def _wgrad_range(ctx, x_seq, h_all, dz_all, dwp, lo, hi, Cin, ks):
        """dwp += the weight gradient of timesteps [lo, hi): the x columns from x_t, the h columns from h_{t-1} =
        h_all[t] (h_{-1} = 0 contributes nothing when the initial state is zero)."""
        ops.conv_wgrad(dz_all[lo:hi], x_seq[lo:hi], ks, dwp, 0)
        lo_h = lo if ctx.have_h0 else max(lo, 1)
        if hi > lo_h:
            ops.conv_wgrad(dz_all[lo_h:hi], h_all[lo_h:hi], ks, dwp, Cin)

    @staticmethod
    def _finish_backward(ctx, x_seq, weight, h_all, dz_all, dx_seq, dh0, dc0, single=None, chunked=None):
        """Weight / bias gradients: one reduction over the whole sequence (K = T*B*H*W), or what is left of it when
        the sweep already queued chunks."""
        T, B, H, W, Cin = x_seq.shape
        Ch = weight.shape[0] // 4
        ks = weight.shape[2]
        if single is None:
            single = ctx.cache.note_backward() if ctx.counted else True
        bg = ops.background((weight, ctx.bias), dz_all, x_seq, h_all, None if chunked is None else chunked["dwp"],
                            allow=single)
        if chunked is not None and not bg.active:
            ops.background_join()  # chunks are in flight on the background stream; the rest runs in line
        with bg:
            if chunked is not None:
                dwp, hi = chunked["dwp"], chunked["hi"]
            else:
                dwp, hi = torch.zeros((ks * ks, 4 * Ch, Cin + Ch), device=x_seq.device, dtype=torch.float32), T
            ConvLSTMSeq._wgrad_range(ctx, x_seq, h_all, dz_all, dwp, 0, hi, Cin, ks)
            dweight = ops.unpack_conv_wgrad(dwp, Cin + Ch)
            dbias = ops.colsum(T * B * H * W, dz_all, 4 * Ch) if ctx.has_bias else None
            bg.keep(dweight, dbias)
        ctx.h_all = ctx.c_all = ctx.gates = None
        return dx_seq, dh0, dc0, dweight, dbias, None


# ------------------------------------------------------------------------------------------------
# SpatialAttention (unet.py:113-125), the optional bottleneck attention of TemporalUNetDualView
# ------------------------------------------------------------------------------------------------
class SpatialAttention(torch.autograd.Function):
    """y = x * a, a = sigmoid(conv_k([mean_c x ; amax_c x])) per image of x [T,B,H,W,C] (weight: the nn.Conv2d weight
    [1, 2, k, k], read by the kernels as it is: no packed copy).  The pooled map and a (fp32, one or two values per
    pixel) are kept for backward with x; the gradient of the max goes to every tied maximum in equal parts, as
    torch.amax's does."""

    @staticmethod
    def forward(ctx, x, weight):
        x = _c(x)
        w = _c(weight.detach())
        y, pooled, a = ops.spatial_attention_fwd(x, w)
        ctx.save_for_backward(x, weight, pooled, a)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight, pooled, a = ctx.saved_tensors
        dy = _c(dy)
        dx, dw = ops.spatial_attention_bwd(x, dy if dy.dtype == x.dtype else dy.to(x.dtype), _c(weight.detach()), pooled,
                                           a, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        return dx, dw
