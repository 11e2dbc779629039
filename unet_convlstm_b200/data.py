"""Host -> device input pipeline of the training loop (SURVEY.md section 8 f2): the reference copies
every batch synchronously on the compute stream (main.py:87-91, `x = x.to(device)`); here the copy of
batch i+1 runs on a side stream from pinned host memory while batch i computes."""
from __future__ import annotations

import numpy as np
import torch


class DevicePrefetcher:
    """Double-buffered asynchronous host->device copies.

        pf = DevicePrefetcher(device)
        pf.start(x_host, y_host)            # pinned host tensors
        for ...:
            x, y = pf.get()                 # device tensors of the batch started last
            pf.start(next_x_host, next_y_host)
            step(x, y)
    """

    def __init__(self, device):
        self.device = torch.device(device)
        self.stream = torch.cuda.Stream(self.device)
        self._pending = None

    def start(self, *host_tensors):
        for t in host_tensors:
            if not t.is_pinned():
                raise RuntimeError("DevicePrefetcher: host tensors must be in pinned memory (tensor.pin_memory())")
        with torch.cuda.stream(self.stream):
            dev = [t.to(self.device, non_blocking=True) for t in host_tensors]
            ev = torch.cuda.Event()
            ev.record(self.stream)
        self._pending = (dev, ev)

    def get(self):
        if self._pending is None:
            raise RuntimeError("DevicePrefetcher.get() without a started copy")
        dev, ev = self._pending
        self._pending = None
        cur = torch.cuda.current_stream(self.device)
        cur.wait_event(ev)
        for t in dev:
            t.record_stream(cur)  # the caching allocator must not recycle the buffer while `cur` uses it
        return dev


# -----------------------------------------------------------------------------------------------------------------------
# The whole dataset in device memory: NPZSequenceDataset.__getitem__ (train/unet.py:393-401) + default_collate as one
# kernel launch per batch (b200_sequence_batch), fed by index lists drawn exactly like the host DataLoader's.
# -----------------------------------------------------------------------------------------------------------------------
_UPLOAD_CHUNK_BYTES = 256 << 20


def _free_device_bytes(device) -> int:
    """Bytes a new allocation on `device` can use: free device memory plus what torch's caching allocator holds unused."""
    free, _ = torch.cuda.mem_get_info(device)
    return int(free) + int(torch.cuda.memory_reserved(device) - torch.cuda.memory_allocated(device))


def _upload(arr, device):
    """fp32 NumPy array -> a new device tensor, copied in slices of the leading dimension (plain synchronous copies)."""
    out = torch.empty(arr.shape, dtype=torch.float32, device=device)
    step = max(1, _UPLOAD_CHUNK_BYTES // max(1, arr[:1].nbytes))
    for i in range(0, arr.shape[0], step):
        out[i:i + step].copy_(torch.from_numpy(np.ascontiguousarray(arr[i:i + step])))
    return out


def _numpy_dtypes(ds, transform):
    """(dtype of the clip, of the transform, of the affine map) in which NumPy 2 evaluates __getitem__'s y for these
    constants (NEP 50: Python floats are weak, np.float64 scalars promote the fp32 item to float64)."""
    f32 = np.dtype(np.float32)
    wdt = np.result_type(np.empty(0, f32), ds.min_vel, ds.max_vel) if ds.clip_outliers else f32
    tdt = np.result_type(np.empty(0, wdt), ds.y_scale) if transform else wdt
    adt = np.result_type(np.empty(0, tdt), ds.trans_min, ds.trans_max - ds.trans_min)
    for d in (wdt, tdt, adt):
        if d not in (np.float32, np.float64):
            raise TypeError(f"DeviceSequenceData: the dataset's constants make NumPy compute in {d}; only float32 and "
                            "float64 are reproduced")
    return wdt, tdt, adt


class DeviceSequenceData:
    """An NPZSequenceDataset's raw X / Y uploaded once to `device`; `batch(indices)` returns what
    default_collate([dataset[i] for i in indices]) returns, as device tensors, from one kernel launch.

    `dataset`: an NPZSequenceDataset, or anything with its attributes X, Y (fp32 [N,T,Cx,H,W] / [N,T,1,H,W]),
    norm_const, min_vel, max_vel, clip_outliers, y_transform, y_scale, trans_min, trans_max.  The constants are the
    dataset's own (its __init__ computed the percentile statistics on the host); they are read here, not recomputed.
    x and mask are bit-identical to the host item; y is bit-identical for the identity transform, and for asinh /
    signed_log within the ulps by which CUDA's asinhf / log1pf (asinh / log1p) differ from the host's.

    Indices are range-checked on the host before they are copied to the device (a CUDA tensor of indices is checked
    with one device-to-host read), so the kernel never sees an out-of-range row."""

    def __init__(self, dataset, device):
        from .loop import _TRANSFORMS
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError(f"DeviceSequenceData: device {device} is not a CUDA device (there is no CPU fallback)")
        X, Y = dataset.X, dataset.Y
        if X.dtype != np.float32 or Y.dtype != np.float32:
            raise TypeError(f"DeviceSequenceData: X and Y must be float32 arrays, got {X.dtype} / {Y.dtype}")
        if X.ndim != 5 or Y.ndim != 5 or Y.shape[2] != 1 or X.shape[:2] != Y.shape[:2] or X.shape[3:] != Y.shape[3:]:
            raise ValueError(f"DeviceSequenceData: expected X [N,T,Cx,H,W] and Y [N,T,1,H,W], got {X.shape} / {Y.shape}")
        need = X.nbytes + Y.nbytes
        free = _free_device_bytes(device)
        if need > free:
            raise RuntimeError(f"DeviceSequenceData: the dataset needs {need} bytes of device memory and {device} has "
                               f"{free} bytes free; use the host loaders (loop.make_loaders without device)")
        self.N, self.T, self.Cx, self.H, self.W = X.shape
        tr = getattr(dataset, "y_transform", None)
        self.transform = _TRANSFORMS[tr if tr in _TRANSFORMS else None]  # any other value: identity, like _transform
        wdt, tdt, adt = _numpy_dtypes(dataset, self.transform)
        # the clip bounds rounded to the clip's dtype: the kernel's fp64 path then also reproduces an fp32 clip followed
        # by an fp64 transform (Python-float bounds with a np.float64 y_scale), since fp32 values are exact in fp64
        lo, hi = (float(np.asarray(dataset.min_vel, wdt)), float(np.asarray(dataset.max_vel, wdt))) \
            if dataset.clip_outliers else (0.0, 0.0)
        self.norm_const = float(dataset.norm_const)
        self.clip = int(bool(dataset.clip_outliers))
        self.min_vel, self.max_vel = lo, hi
        self.y_scale = float(dataset.y_scale)
        self.trans_min = float(dataset.trans_min)
        self.trans_range = float(dataset.trans_max - dataset.trans_min)  # as __getitem__ computes it, then widened
        self.fp64_transform = int(tdt == np.float64)
        self.fp64_affine = int(adt == np.float64)
        self.X = _upload(X, device)
        self.Y = _upload(Y, device)
        self.device = self.X.device

    def __len__(self):
        return self.N

    def device_indices(self, indices):
        """`indices` (list, NumPy array, CPU or CUDA tensor) -> int64 [B] on the device, checked against [0, N)."""
        if torch.is_tensor(indices) and indices.is_cuda:
            idx = indices.reshape(-1).to(self.device, torch.int64)
            if idx.numel() and bool(((idx < 0) | (idx >= self.N)).any()):
                raise IndexError(f"DeviceSequenceData: an index is outside [0, {self.N})")
        else:
            idx = torch.as_tensor(indices, dtype=torch.int64).reshape(-1)
            if idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= self.N):
                raise IndexError(f"DeviceSequenceData: index {int(idx.min()) if int(idx.min()) < 0 else int(idx.max())} "
                                 f"is outside [0, {self.N})")
            if self.X.is_cuda:
                idx = idx.pin_memory().to(self.device, non_blocking=True)
        if idx.numel() == 0:
            raise ValueError("DeviceSequenceData: empty batch")
        return idx

    def batch(self, indices):
        """(x, y, mask) fp32 [B,T,Cx,H,W] / [B,T,1,H,W] / [B,T,1,H,W] on the device for the dataset rows `indices`: new
        tensors from the caching allocator, written by one launch on the current stream of the dataset's device (which
        need not be the current device)."""
        return self._batch(self.device_indices(indices))

    def _batch(self, idx):
        """batch() of int64 device indices that device_indices() has already checked."""
        from . import _lib
        from .ops import _st
        B = idx.numel()
        x = torch.empty((B, self.T, self.Cx, self.H, self.W), dtype=torch.float32, device=self.device)
        y = torch.empty((B, self.T, 1, self.H, self.W), dtype=torch.float32, device=self.device)
        mask = torch.empty_like(y)
        # the launch goes to the current device and its current stream: make that the dataset's device (get_device()
        # is -1, a no-op, only for arrays left on the host)
        with torch.cuda.device(self.X.get_device()):
            _lib.call("b200_sequence_batch", self.X, self.Y, self.N, self.T, self.Cx, self.H, self.W, idx, B,
                      self.norm_const, self.clip, self.min_vel, self.max_vel, self.transform, self.y_scale,
                      self.trans_min, self.trans_range, self.fp64_transform, self.fp64_affine, x, y, mask, _st())
        return x, y, mask


class DeviceLoader:
    """Batches of a DeviceSequenceData in the order a torch.utils.data.DataLoader with the same sampler, batch_size,
    drop_last and generator yields them, epoch after epoch.

    `sampler`: a RandomSampler (with its generator), a SequentialSampler or a DistributedSampler over positions
    0..len(rows)-1; `rows`: the dataset row of each position (a random_split Subset's `indices`; None = identity).
    `generator`: the DataLoader's own generator (None = torch's default one).  Like DataLoader, every iteration first
    draws one int64 from it (the DataLoader's base seed) and only then lets the sampler draw, so both the order and the
    state of the generators stay in step with the host loader.  Each epoch's index list is copied to the device once."""

    def __init__(self, data, sampler, batch_size, drop_last=False, rows=None, generator=None):
        if batch_size < 1:
            raise ValueError("DeviceLoader: batch_size must be >= 1")
        self.data = data
        self.sampler = sampler
        self.batch_size = int(batch_size)
        self.drop_last = bool(drop_last)
        self.rows = torch.arange(len(data)) if rows is None else torch.as_tensor(rows, dtype=torch.int64)
        self.generator = generator

    def __len__(self):
        n = len(self.sampler)
        return n // self.batch_size if self.drop_last else -(-n // self.batch_size)

    def epoch_indices(self):
        """The dataset rows of one epoch, in order (advances the generators exactly like iterating a DataLoader)."""
        torch.empty((), dtype=torch.int64).random_(generator=self.generator)  # DataLoader's _base_seed
        pos = torch.as_tensor(list(iter(self.sampler)), dtype=torch.int64)
        if self.drop_last:
            pos = pos[:len(self) * self.batch_size]
        return self.rows[pos]

    def __iter__(self):
        rows = self.epoch_indices()
        if rows.numel() == 0:
            return
        dev = self.data.device_indices(rows)
        for s in range(0, rows.numel(), self.batch_size):
            yield self.data._batch(dev[s:s + self.batch_size])
