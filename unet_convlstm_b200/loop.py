"""The host side of the reference's training / evaluation loops (SURVEY.md section 8 f2).

`train_one_epoch` and `evaluate` have the signatures and return values of the reference's functions of the same
names (main.py:77-145, :150-204): `(avg_loss, avg_mae, avg_rmse, avg_me)` over one pass of the loader.  What
differs is where the work happens:

  * the reference copies y, y_pred and the mask to the host EVERY step, de-normalises them in NumPy and
    `list.extend`s three Python lists with one float per valid pixel (main.py:110-133); here one kernel per step
    (`b200_denorm_metrics_accum`) de-normalises on the device and adds to four fp64 accumulators;
  * `loss.item()` (main.py:108) synchronises the host with the device every step; here the running loss is a
    device scalar and the host reads five numbers once per epoch;
  * batches that arrive as host tensors are copied by a side stream from pinned memory one step ahead
    (`DevicePrefetcher`) instead of synchronously on the compute stream (main.py:89).

CUDA only: there is no CPU fallback.
"""
from __future__ import annotations

import math

import torch

from . import _lib
from .data import DeviceLoader, DevicePrefetcher, DeviceSequenceData
from .loss import compute_loss
from .optim import AdamW
from .ops import _p, _st

_TRANSFORMS = {None: 0, "none": 0, "asinh": 1, "signed_log": 2}


class RunningMetrics:
    """MAE / RMSE / ME of the de-normalised prediction over the valid pixels, accumulated on the device.

    dataset_obj: anything with the normalisation attributes of the reference's NPZSequenceDataset
    (`trans_min`, `trans_max`, `y_scale`, `y_transform`; unet.py:233-262)."""

    def __init__(self, dataset_obj, device):
        tr = getattr(dataset_obj, "y_transform", None)
        if tr not in _TRANSFORMS:
            tr = None  # the reference's denormalize treats any other value as the identity (unet.py:322-323)
        self.transform = _TRANSFORMS[tr]
        self.trans_min = float(dataset_obj.trans_min)
        self.trans_max = float(dataset_obj.trans_max)
        self.y_scale = float(getattr(dataset_obj, "y_scale", 1.0))
        self.acc = torch.zeros(4, device=device, dtype=torch.float64)

    def reset(self):
        self.acc.zero_()

    def update(self, y_pred, y, mask=None, use_mask=True):
        for t, name in ((y_pred, "y_pred"), (y, "y"), (mask, "mask")):
            if t is not None and not t.is_cuda:
                raise RuntimeError(f"RunningMetrics.update: {name} is on {t.device}; there is no CPU fallback")
        if y_pred.shape != y.shape or (mask is not None and use_mask and mask.shape != y.shape):
            raise ValueError("RunningMetrics.update: shapes differ")
        yp = y_pred.detach().float().contiguous()
        yt = y.detach().float().contiguous()
        mk = mask.detach().float().contiguous() if (use_mask and mask is not None) else None
        _lib.call("b200_denorm_metrics_accum", _p(yp), _p(yt), _p(mk), yp.numel(), self.transform, self.trans_min,
                  self.trans_max, self.y_scale, _p(self.acc), _st())

    def compute(self):
        """(mae, rmse, me); all zero when no pixel was valid (main.py:137-143).  One device->host read."""
        s_abs, s_sq, s_err, cnt = self.acc.tolist()
        if cnt <= 0:
            return 0.0, 0.0, 0.0
        return s_abs / cnt, math.sqrt(s_sq / cnt), s_err / cnt


def _device_batches(loader, device):
    """Yields (x, y, mask) on `device`; host batches are copied one step ahead on a side stream."""
    pf = None
    it = iter(loader)

    def prep(batch):
        nonlocal pf
        if all(t.is_cuda for t in batch):
            return batch, False
        if pf is None:
            pf = DevicePrefetcher(device)
        pf.start(*[t if t.is_pinned() else t.pin_memory() for t in batch])
        return None, True

    try:
        cur, staged = prep(next(it))
    except StopIteration:
        return
    while True:
        if staged:
            cur = pf.get()
        try:
            nxt = next(it)
        except StopIteration:
            yield cur
            return
        nxt_dev, nxt_staged = prep(nxt)
        yield cur
        cur, staged = nxt_dev, nxt_staged


def make_loaders(dataset, batch_size, seed=42, train_fraction=0.8, rank=None, world=None, device=None):
    """The data pipeline of main.py:241-246 for one rank of a data-parallel job: the same 80/20 random split on every
    rank (seeded -- main.py splits unseeded, a single process does not care), then a per-rank DistributedSampler over
    the training part (shuffled, re-seeded per epoch by `loader.sampler.set_epoch(e)`) and over the validation part
    (in order).  `batch_size` is per rank.  With world == 1 this is exactly main.py's pair of DataLoaders.

    device: None returns those host DataLoaders.  A CUDA device uploads the dataset once (data.DeviceSequenceData) and
    returns a pair of data.DeviceLoader with the same split, samplers and seeds: the same batches in the same order,
    each built on the device by one kernel launch instead of NPZSequenceDataset.__getitem__ on the host."""
    import torch.distributed as dist
    from torch.utils.data import DataLoader, DistributedSampler, RandomSampler, SequentialSampler, random_split
    if world is None:
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    if rank is None:
        rank = dist.get_rank() if world > 1 else 0
    n_train = int(train_fraction * len(dataset))
    gen = torch.Generator().manual_seed(seed)
    train_ds, val_ds = random_split(dataset, [n_train, len(dataset) - n_train], generator=gen)
    if world == 1:
        g2 = torch.Generator().manual_seed(seed)
        if device is None:
            return (DataLoader(train_ds, batch_size=batch_size, shuffle=True, pin_memory=True, generator=g2),
                    DataLoader(val_ds, batch_size=batch_size, shuffle=False, pin_memory=True))
        ts, vs, tgen = RandomSampler(train_ds, generator=g2), SequentialSampler(val_ds), g2
    else:
        ts = DistributedSampler(train_ds, num_replicas=world, rank=rank, shuffle=True, seed=seed, drop_last=False)
        vs = DistributedSampler(val_ds, num_replicas=world, rank=rank, shuffle=False, drop_last=False)
        if device is None:
            return (DataLoader(train_ds, batch_size=batch_size, sampler=ts, pin_memory=True),
                    DataLoader(val_ds, batch_size=batch_size, sampler=vs, pin_memory=True))
        tgen = None
    data = DeviceSequenceData(dataset, device)
    # DataLoader(shuffle=True, generator=g2) draws its base seed from g2; the other loaders draw it from torch's
    # default generator, and so do these
    return (DeviceLoader(data, ts, batch_size, rows=train_ds.indices, generator=tgen),
            DeviceLoader(data, vs, batch_size, rows=val_ds.indices))


def _stack(output):
    return torch.stack(output, dim=1) if isinstance(output, (list, tuple)) else output


def train_one_epoch(model, loader, optimizer, device, dataset_obj, use_mask=True, max_norm=1.0, after_backward=None):
    """One epoch of main.py:77-145: forward, compute_loss, backward, clip_grad_norm_(max_norm), optimizer step, and
    the running loss / MAE / RMSE / ME.  `after_backward`: optional callable run between backward and the clip
    (the data-parallel gradient reducer's `finish`)."""
    from . import ops
    ops.enable_background_wgrad()  # gradients are read after backward() (clip + optimizer below, or the GradReducer)
    model.train()
    device = torch.device(device)
    metrics = RunningMetrics(dataset_obj, device)
    total = torch.zeros((), device=device, dtype=torch.float64)
    n = 0
    for x, y, mask in _device_batches(loader, device):
        optimizer.zero_grad(set_to_none=True)
        output, _ = model(x)
        y_pred = _stack(output)
        loss = compute_loss(y_pred, y, mask, use_mask)
        loss.backward()
        if after_backward is not None:
            after_backward()
        if isinstance(optimizer, AdamW):
            optimizer.step(clip_max_norm=max_norm)   # norm + clip + update: two passes, nothing read back
        else:
            torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm)
            optimizer.step()
        total += loss.detach().double() * x.size(0)
        n += x.size(0)
        metrics.update(y_pred, y, mask, use_mask)
    if n == 0:
        raise ZeroDivisionError("train_one_epoch: empty loader")  # the reference divides by n = 0 (main.py:136)
    return (float(total) / n, *metrics.compute())


@torch.no_grad()
def evaluate(model, loader, device, dataset_obj, use_mask=True):
    """main.py:150-204: eval-mode forward, loss in the normalised space, metrics in physical units."""
    model.eval()
    device = torch.device(device)
    metrics = RunningMetrics(dataset_obj, device)
    total = torch.zeros((), device=device, dtype=torch.float64)
    n = 0
    for x, y, mask in _device_batches(loader, device):
        output, _ = model(x)
        y_pred = _stack(output)
        total += compute_loss(y_pred, y, mask, use_mask).double() * x.size(0)
        n += x.size(0)
        metrics.update(y_pred, y, mask, use_mask)
    if n == 0:
        raise ZeroDivisionError("evaluate: empty loader")
    return (float(total) / n, *metrics.compute())
