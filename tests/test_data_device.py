"""The device-resident dataset (unet_convlstm_b200/data.py: DeviceSequenceData, DeviceLoader) without a GPU: the batch
order of the device loaders against torch's DataLoader, a dry run of the b200_sequence_batch call against its prototype
in include/b200_convlstm.h, the dtypes the kernel is told to compute in, and the refusals."""
import ctypes
import types

import numpy as np
import pytest
import torch


class _Rows(torch.utils.data.Dataset):
    """Item i is the dataset row i itself: a DataLoader over it yields the rows of each batch."""

    def __init__(self, n):
        self.n = n

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        return torch.tensor(i)


class _RowsOnDevice:
    """Stands in for DeviceSequenceData: a batch is its (checked) row indices."""

    def __init__(self, dataset, device):
        self.n = len(dataset)

    def __len__(self):
        return self.n

    def device_indices(self, rows):
        return torch.as_tensor(rows, dtype=torch.int64)

    def _batch(self, idx):
        return idx


def _host_and_device(monkeypatch, n, batch_size, rank, world):
    from unet_convlstm_b200 import loop
    monkeypatch.setattr(loop, "DeviceSequenceData", _RowsOnDevice)
    ds = _Rows(n)
    return (loop.make_loaders(ds, batch_size, rank=rank, world=world),
            loop.make_loaders(ds, batch_size, rank=rank, world=world, device="cuda"))


def _epochs(loader, epochs, set_epoch):
    out = []
    for e in range(epochs):
        if set_epoch:
            loader.sampler.set_epoch(e)
        out.append([b.tolist() for b in loader])
    return out


@pytest.mark.filterwarnings("ignore:.*pin_memory")
def test_order_matches_dataloader_world1(monkeypatch):
    """make_loaders(device=...) at world 1: the shuffled training loader and the validation loader yield the rows of
    the host DataLoaders, batch for batch, over 3 epochs (23 items: 18 / 5, batch 4, partial last batches), and leave
    torch's default generator in the same state."""
    torch.manual_seed(0)
    (htr, hva), (dtr, dva) = _host_and_device(monkeypatch, 23, 4, 0, 1)
    torch.manual_seed(7)
    host = [_epochs(htr, 1, False) + _epochs(hva, 1, False) for _ in range(3)]
    host_rng = torch.get_rng_state()
    torch.manual_seed(7)
    dev = [_epochs(dtr, 1, False) + _epochs(dva, 1, False) for _ in range(3)]
    assert dev == host
    assert torch.equal(torch.get_rng_state(), host_rng)
    assert [len(b) for b in host[0][0]] == [4, 4, 4, 4, 2] and [len(b) for b in host[0][1]] == [4, 1]
    assert host[0][0] != host[1][0] != host[2][0]                  # reshuffled every epoch
    assert len(dtr) == len(htr) == 5 and len(dva) == len(hva) == 2


@pytest.mark.filterwarnings("ignore:.*pin_memory")
@pytest.mark.parametrize("rank", range(4))
def test_order_matches_dataloader_world4(monkeypatch, rank):
    """At world 4 every rank's DistributedSampler pair, re-seeded with set_epoch, yields the host loaders' rows."""
    (htr, hva), (dtr, dva) = _host_and_device(monkeypatch, 41, 3, rank, 4)
    assert _epochs(dtr, 3, True) == _epochs(htr, 3, True)
    assert _epochs(dva, 3, True) == _epochs(hva, 3, True)
    assert [len(b) for b in _epochs(dtr, 1, True)[0]] == [3, 3, 2]  # 32 training items: 8 per rank
    assert dtr.sampler is not htr.sampler and len(dtr) == len(htr)


def test_random_sampler_draws_after_the_base_seed():
    """DataLoader draws its base seed from the generator before the RandomSampler's permutation: for seed 42 and
    10 items the batches are [6,5,4,0], [8,9,2,1], [3,7], not the permutation the sampler would draw alone."""
    from torch.utils.data import DataLoader, RandomSampler
    from unet_convlstm_b200.data import DeviceLoader
    g = torch.Generator().manual_seed(42)
    host = [b.tolist() for b in DataLoader(_Rows(10), batch_size=4, shuffle=True, generator=g)]
    assert host == [[6, 5, 4, 0], [8, 9, 2, 1], [3, 7]]
    g = torch.Generator().manual_seed(42)
    dev = DeviceLoader(_RowsOnDevice(_Rows(10), None), RandomSampler(_Rows(10), generator=g), 4, generator=g)
    assert [b.tolist() for b in dev] == host
    g = torch.Generator().manual_seed(42)
    assert list(RandomSampler(_Rows(10), generator=g))[:4] != host[0]
    g = torch.Generator().manual_seed(42)
    dev = DeviceLoader(_RowsOnDevice(_Rows(10), None), RandomSampler(_Rows(10), generator=g), 4, drop_last=True,
                       generator=g)
    assert [b.tolist() for b in dev] == host[:2] and len(dev) == 2


def _dataset(tmp_path, **kw):
    from train.unet import NPZSequenceDataset
    rng = np.random.default_rng(3)
    X = (rng.random((5, 3, 2, 8, 12)) * 3).astype(np.float32)
    Y = (rng.standard_normal((5, 3, 1, 8, 12)) * 4).astype(np.float32)
    np.savez(tmp_path / "d.npz", X=X, Y=Y)
    return NPZSequenceDataset(str(tmp_path / "d.npz"), **kw)


@pytest.fixture
def dry(monkeypatch):
    """DeviceSequenceData with the arrays left on the host and every C-ABI call checked against the header, not run."""
    from unet_convlstm_b200 import _lib, data, ops
    protos = _lib.parse_header()
    calls = []

    def fake_call(name, *args, tag="", work=None):
        assert name in protos, f"{name} is not declared in include/b200_convlstm.h"
        _, argtypes = protos[name]
        assert len(args) == len(argtypes), (name, len(args), len(argtypes))
        for i, (a, t) in enumerate(zip(args, argtypes)):
            if t is ctypes.c_void_p:
                assert a is None or hasattr(a, "data_ptr") or isinstance(a, int), (name, i, type(a))
            elif t in (ctypes.c_int, ctypes.c_longlong):
                assert isinstance(a, int) and not isinstance(a, bool), (name, i, type(a), a)
            else:
                assert isinstance(a, float), (name, i, type(a))
        calls.append((name, args))

    monkeypatch.setattr(_lib, "call", fake_call)
    monkeypatch.setattr(ops, "_st", lambda: 0)
    monkeypatch.setattr(data, "_free_device_bytes", lambda device: 1 << 40)
    monkeypatch.setattr(data, "_upload", lambda arr, device: torch.from_numpy(np.ascontiguousarray(arr)))
    return calls


def test_dry_run_matches_the_header(dry, tmp_path):
    from unet_convlstm_b200.data import DeviceSequenceData
    ds = _dataset(tmp_path)
    d = DeviceSequenceData(ds, "cuda")
    x, y, mask = d.batch([4, 0, 4])
    assert x.shape == (3, 3, 2, 8, 12) and y.shape == mask.shape == (3, 3, 1, 8, 12)
    assert all(t.dtype == torch.float32 and t.is_contiguous() for t in (x, y, mask))
    (name, args), = dry
    assert name == "b200_sequence_batch"
    assert args[7].dtype == torch.int64 and args[7].tolist() == [4, 0, 4] and args[8] == 3
    assert args[2:7] == (5, 3, 2, 8, 12)
    assert args[19] is x and args[20] is y and args[21] is mask


def _flags(d):
    return d.clip, d.transform, d.fp64_transform, d.fp64_affine


def test_numpy_dtypes_are_followed(dry, tmp_path):
    """The precision flags follow the types of the dataset's constants as NumPy 2 promotes them in __getitem__."""
    from unet_convlstm_b200.data import DeviceSequenceData
    # explicit constants: Python-float bounds (fp32 clip and transform), np.float64 trans_min (fp64 affine map)
    assert _flags(DeviceSequenceData(_dataset(tmp_path), "cuda")) == (1, 1, 0, 1)
    assert _flags(DeviceSequenceData(_dataset(tmp_path, y_transform="signed_log"), "cuda")) == (1, 2, 0, 1)
    # identity: trans_min is the Python float min_y itself, so the affine map stays fp32
    assert _flags(DeviceSequenceData(_dataset(tmp_path, y_transform=None), "cuda")) == (1, 0, 0, 0)
    assert _flags(DeviceSequenceData(_dataset(tmp_path, y_transform="other"), "cuda")) == (1, 0, 0, 0)
    # percentile constants of fp32 data are np.float32: everything fp32
    pct = _dataset(tmp_path, min_y=None, max_y=None, lower_percentile=1, upper_percentile=99)
    assert _flags(DeviceSequenceData(pct, "cuda")) == (1, 1, 0, 0)
    pct.clip_outliers = False
    assert _flags(DeviceSequenceData(pct, "cuda")) == (0, 1, 0, 0)
    # np.float64 clip bounds promote the item to float64 before the transform
    ds = _dataset(tmp_path)
    ds.min_vel, ds.max_vel = np.float64(-3.5), np.float64(3.25)
    d = DeviceSequenceData(ds, "cuda")
    assert _flags(d) == (1, 1, 1, 1) and (d.min_vel, d.max_vel) == (-3.5, 3.25)
    # Python-float bounds reach the kernel rounded to fp32, as NumPy rounds them for the fp32 clip
    ds = _dataset(tmp_path, min_y=-0.1, max_y=0.3)
    d = DeviceSequenceData(ds, "cuda")
    assert d.min_vel == float(np.float32(-0.1)) and d.max_vel == float(np.float32(0.3))
    assert d.trans_range == float(ds.trans_max - ds.trans_min)


def test_refusals(dry, tmp_path, monkeypatch):
    from unet_convlstm_b200 import data
    from unet_convlstm_b200.data import DeviceSequenceData
    ds = _dataset(tmp_path)
    with pytest.raises(RuntimeError, match="not a CUDA device"):
        DeviceSequenceData(ds, "cpu")
    need = ds.X.nbytes + ds.Y.nbytes
    monkeypatch.setattr(data, "_free_device_bytes", lambda device: need - 1)
    with pytest.raises(RuntimeError, match=f"needs {need} bytes of device memory and cuda has {need - 1} bytes free"):
        DeviceSequenceData(ds, "cuda")
    monkeypatch.setattr(data, "_free_device_bytes", lambda device: need)
    d = DeviceSequenceData(ds, "cuda")
    for bad in ([0, 5], [-1], torch.tensor([2, 7]), np.array([5])):
        with pytest.raises(IndexError, match=r"outside \[0, 5\)"):
            d.batch(bad)
    with pytest.raises(ValueError, match="empty batch"):
        d.batch([])
    assert not dry                                                   # nothing reached the kernel
    bad = types.SimpleNamespace(**{k: getattr(ds, k) for k in ("norm_const", "min_vel", "max_vel", "clip_outliers",
                                                               "y_transform", "y_scale", "trans_min", "trans_max")})
    bad.X, bad.Y = ds.X.astype(np.float64), ds.Y
    with pytest.raises(TypeError, match="float32"):
        DeviceSequenceData(bad, "cuda")
    bad.X, bad.Y = ds.X, ds.Y[:, :, :, :4]
    with pytest.raises(ValueError, match="expected X"):
        DeviceSequenceData(bad, "cuda")
