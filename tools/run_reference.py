"""Runs the reference's own scripts UNCHANGED on top of this repository's `train/unet.py` (or, with --impl reference,
on top of the reference's own `train/unet.py`, for the A/B).

    python tools/run_reference.py overfit     [--impl b200|reference] [--precision bf16|fp32] [--iters 300] [--out curve.json]
    python tools/run_reference.py main        [--impl ...] [--epochs 1] [--batch-size 8]
    python tools/run_reference.py get_metrics [--impl ...] --checkpoint models/..._best_skip.pt

The scripts (reference main.py:211-325, train/overfit_check.py:36-139, train/get_metrics.py:66-173) are executed from
their own source files, in the checkout of the reference project that B200_REFERENCE_DIR names (this repository does
not ship them).  What this launcher supplies is ENVIRONMENT only (SURVEY.md section 8b "hazards"):

  1. sys.path: the repository root first, so `from train.unet import ...` resolves to the B200 implementation while
     `train.resnet18` / `train.overfit_check` / `train.get_metrics` (the namespace package `train` has no __init__.py)
     still resolve to the reference's files; with --impl reference the reference root goes first instead.
  2. a stub `segmentation_models_pytorch` (absent here, needs a download) for the `import` in train/resnet18.py:5,
     and a stub `matplotlib` (absent) whose savefig() writes placeholder files, for train/get_metrics.py.
  3. `ReduceLROnPlateau(verbose=True)` (main.py:278-280) raises TypeError on torch >= 2.7: the keyword is dropped.
  4. `torch.load` defaults to weights_only=True since torch 2.6, which rejects the numpy index array the reference's
     checkpoints hold (overfit_check.py:126-130): the launcher passes weights_only=False for these trusted files.
  5. the scripts' in-file CONSTANTS (USE_PRETRAINED, NPZ_PATH, EPOCHS, ... -- the reference has no flags, one edits the
     file: main.py:213-228, overfit_check.py:26-31, get_metrics.py:42-61) are overridden by value, either as module
     attributes after import (overfit_check) or, for the flat `__main__` scripts, by rewriting ONLY the right-hand
     side of those assignments in the parsed AST before execution.  No statement of the scripts' logic is touched.
  6. a synthetic NPZ with the reference's keys X [N,T,2,H,W] / Y [N,T,1,H,W] (unet.py:212-215) at the configured path.
"""
from __future__ import annotations

import argparse
import ast
import builtins
import contextlib
import io
import json
import os
import re
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def find_reference() -> str | None:
    """The absolute path of the reference checkout named by B200_REFERENCE_DIR, or None when it is unset or holds no
    train/unet.py."""
    cand = os.environ.get("B200_REFERENCE_DIR")
    if cand and os.path.exists(os.path.join(cand, "train", "unet.py")):
        return os.path.abspath(cand)
    return None


def reference_root() -> str:
    """The directory holding the reference's scripts (find_reference); raises when there is none."""
    ref = find_reference()
    if ref is None:
        raise RuntimeError("reference sources not found: set B200_REFERENCE_DIR to a checkout of the reference project "
                           "(dordanino12/unet-convlstm)")
    return ref


# ------------------------------------------------------------------------------------------------
# environment shims
# ------------------------------------------------------------------------------------------------
class _Stub:
    """Accepts any attribute access, call, item access and `a, b = stub` unpacking."""

    def __init__(self, name="stub"):
        self.__dict__["_name"] = name

    def __getattr__(self, k):
        if k.startswith("__") and k.endswith("__"):
            raise AttributeError(k)
        return _Stub(f"{self._name}.{k}")

    def __setattr__(self, k, v):
        pass

    def __call__(self, *a, **kw):
        return _Stub(self._name + "()")

    def __getitem__(self, k):
        return _Stub(self._name + "[]")

    def __setitem__(self, k, v):
        pass

    def __iter__(self):
        return iter((_Stub(self._name + "[0]"), _Stub(self._name + "[1]")))


def _savefig(path, *a, **kw):
    path = str(path)
    os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
    if path.lower().endswith((".png", ".jpg", ".jpeg")):
        from PIL import Image
        Image.new("RGB", (16, 16), "white").save(path)
    else:
        with open(path, "wb") as f:
            f.write(b"%placeholder written by tools/run_reference.py (matplotlib is not installed)\n")


def install_stubs():
    import torch
    if "segmentation_models_pytorch" not in sys.modules:
        try:
            import segmentation_models_pytorch  # noqa: F401
        except ImportError:
            smp = types.ModuleType("segmentation_models_pytorch")

            def _unet(*a, **kw):
                raise RuntimeError("segmentation_models_pytorch is not installed (no network): PretrainedTemporalUNet "
                                   "cannot be built; run with USE_PRETRAINED=False")
            smp.Unet = _unet
            sys.modules["segmentation_models_pytorch"] = smp
    try:
        import matplotlib  # noqa: F401
    except ImportError:
        mpl = types.ModuleType("matplotlib")
        mpl.rcParams = {}
        mpl.use = lambda *a, **kw: None
        plt = types.ModuleType("matplotlib.pyplot")
        stub = _Stub("plt")
        plt.__getattr__ = lambda k: getattr(stub, k)
        plt.savefig = _savefig
        mpl.pyplot = plt
        sys.modules["matplotlib"] = mpl
        sys.modules["matplotlib.pyplot"] = plt
    # (3) verbose= keyword of ReduceLROnPlateau
    sched = torch.optim.lr_scheduler
    if not getattr(sched.ReduceLROnPlateau, "_b200_shim", False):
        base = sched.ReduceLROnPlateau

        class ReduceLROnPlateau(base):
            _b200_shim = True

            def __init__(self, *a, verbose=None, **kw):
                super().__init__(*a, **kw)
        sched.ReduceLROnPlateau = ReduceLROnPlateau
    # (4) weights_only default of torch.load
    if not getattr(torch.load, "_b200_shim", False):
        orig = torch.load

        def load(*a, **kw):
            kw.setdefault("weights_only", False)
            return orig(*a, **kw)
        load._b200_shim = True
        torch.load = load


def set_paths(impl: str):
    ref = reference_root()
    for p in (ROOT, ref):
        while p in sys.path:
            sys.path.remove(p)
    order = [ROOT, ref] if impl == "b200" else [ref, ROOT]
    sys.path[:0] = order
    for k in [k for k in sys.modules if k == "train" or k.startswith("train.")]:
        del sys.modules[k]
    return ref


def run_flat_script(path: str, overrides: dict, run_name="__main__"):
    """Executes a flat script with the right-hand sides of `NAME = <literal>` assignments replaced (hazard 5)."""
    src = open(path).read()
    tree = ast.parse(src, filename=path)
    seen = set()

    class Rewrite(ast.NodeTransformer):
        def visit_Assign(self, node):
            if len(node.targets) == 1 and isinstance(node.targets[0], ast.Name) and node.targets[0].id in overrides:
                seen.add(node.targets[0].id)
                node.value = ast.copy_location(ast.Constant(overrides[node.targets[0].id]), node.value)
            return node
    tree = ast.fix_missing_locations(Rewrite().visit(tree))
    missing = set(overrides) - seen
    if missing:
        raise RuntimeError(f"{path}: constants {sorted(missing)} not found")
    g = {"__name__": run_name, "__file__": path, "__builtins__": builtins}
    exec(compile(tree, path, "exec"), g)
    return g


def write_synthetic_npz(path: str, N=24, T=8, S=64, seed=0):
    """Cloud-shaped synthetic data with the reference's NPZ keys (unet.py:212-215): X non-negative radiance with
    values above the cloud-mask threshold 1.1 (unet.py:279), Y a smooth velocity field in m/s."""
    import numpy as np
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:S, 0:S].astype(np.float32)
    X = np.zeros((N, T, 2, S, S), np.float32)
    Y = np.zeros((N, T, 1, S, S), np.float32)
    for n in range(N):
        cx, cy = rng.uniform(S * 0.2, S * 0.8, 2)
        vx, vy = rng.uniform(-2.5, 2.5, 2)
        sg = rng.uniform(S * 0.12, S * 0.25)
        amp = rng.uniform(15, 43)
        for t in range(T):
            blob = amp * np.exp(-(((xx - cx - vx * t) ** 2 + (yy - cy - vy * t) ** 2) / (2 * sg * sg)))
            X[n, t, 0] = blob
            X[n, t, 1] = np.roll(blob, 2, axis=1) * 0.9
            Y[n, t, 0] = (blob > 1.1) * (vx * 2.0 + 0.5 * np.sin(xx / 7.0))
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    np.savez(path, X=X, Y=Y)
    return path


def _seed(seed):
    import numpy as np
    import torch
    np.random.seed(seed)
    torch.manual_seed(seed)


def _work_dir():
    """Scratch directory for the synthetic NPZ and the checkpoints the scripts save (0.5 GB each at base_ch 64):
    outside the repository, so they neither enter a snapshot nor gpurun_out/."""
    import tempfile
    d = os.environ.get("B200_WORK_DIR") or os.path.join(tempfile.gettempdir(), "b200_run_reference")
    os.makedirs(d, exist_ok=True)
    return d


class _Tee(io.TextIOBase):
    def __init__(self, real):
        self.real, self.buf = real, io.StringIO()

    def write(self, s):
        self.real.write(s)
        self.buf.write(s)
        return len(s)

    def flush(self):
        self.real.flush()


# ------------------------------------------------------------------------------------------------
# the three scripts
# ------------------------------------------------------------------------------------------------
def run_overfit(args):
    """train/overfit_check.py: run_overfit_test_and_save() as shipped, bounded to --iters iterations."""
    set_paths(args.impl)
    install_stubs()
    npz = args.npz or write_synthetic_npz(os.path.join(_work_dir(), "overfit.npz"), T=args.seq_len, S=args.size)
    _seed(args.seed)
    import importlib
    oc = importlib.import_module("train.overfit_check")
    oc.USE_PRETRAINED = False          # overfit_check.py:26 (the committed default needs the smp download)
    oc.npz_path = npz                  # overfit_check.py:29-31
    oc.current_dir = _work_dir()       # where the script saves its checkpoint (overfit_check.py:121,135)
    iters = args.iters
    oc.range = lambda n: builtins.range(min(n, iters + 1))  # `for i in range(3001)` (overfit_check.py:91)
    _seed(args.seed)                   # the script seeds nothing itself (np.random.choice at :43)
    tee = _Tee(sys.stdout)
    with contextlib.redirect_stdout(tee):
        oc.run_overfit_test_and_save()
    curve = {int(m.group(1)): float(m.group(2)) for m in re.finditer(r"Iter (\d+) \| Loss: ([0-9.eE+-]+)", tee.buf.getvalue())}
    import train.unet as tu
    res = {"impl": args.impl, "precision": args.precision, "unet_module": tu.__file__, "curve": curve}
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f)
    print(json.dumps(res))
    return res


def run_main(args):
    """main.py as `__main__` (data split, model, AdamW, ReduceLROnPlateau, epochs of train_one_epoch + evaluate,
    best-checkpoint save)."""
    ref = set_paths(args.impl)
    install_stubs()
    wd = _work_dir()
    npz = args.npz or write_synthetic_npz(os.path.join(wd, "main.npz"), N=args.num_seq, T=args.seq_len, S=args.size)
    _seed(args.seed)
    cwd = os.getcwd()
    os.chdir(wd)                       # main.py saves to ./models (main.py:284-285)
    try:
        g = run_flat_script(os.path.join(ref, "main.py"),
                            {"USE_PRETRAINED": False, "NPZ_PATH": npz, "EPOCHS": args.epochs, "BATCH_SIZE": args.batch_size})
    finally:
        os.chdir(cwd)
    ck = os.path.join(wd, "models", "custom_unet_64ch_best_skip.pt")
    print(json.dumps({"impl": args.impl, "best_val_loss": g.get("best_val_loss"), "checkpoint": ck if os.path.exists(ck) else None}))
    return g


def run_get_metrics(args):
    """train/get_metrics.py as `__main__`: checkpoint -> model from its config -> per-sequence inference -> metrics."""
    ref = set_paths(args.impl)
    install_stubs()
    wd = _work_dir()
    npz = args.npz or os.path.join(wd, "main.npz")
    if not os.path.exists(npz):
        write_synthetic_npz(npz, N=args.num_seq, T=args.seq_len, S=args.size)
    ck = args.checkpoint or os.path.join(wd, "models", "custom_unet_64ch_best_skip.pt")
    _seed(args.seed)
    tee = _Tee(sys.stdout)
    with contextlib.redirect_stdout(tee):
        run_flat_script(os.path.join(ref, "train", "get_metrics.py"),
                        {"NPZ_PATH": npz, "CHECKPOINT_PATH": ck, "save_path": os.path.join(wd, "plots", "evaluation_comprehensive.pdf"),
                         "output_dir": os.path.join(wd, "plots") + os.sep})
    txt = tee.buf.getvalue()
    m = {k: float(v) for k, v in re.findall(r"Global (MAE|RMSE|Mean Error \(Bias\)|Error Std):\s+([0-9.eE+-]+)", txt)}
    print(json.dumps({"impl": args.impl, "metrics": m}))
    return m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("script", choices=["overfit", "main", "get_metrics"])
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "tf32", "fp32"])
    ap.add_argument("--iters", type=int, default=300)
    ap.add_argument("--epochs", type=int, default=1)
    ap.add_argument("--batch-size", type=int, default=8)
    ap.add_argument("--num-seq", type=int, default=24)
    ap.add_argument("--seq-len", type=int, default=8)
    ap.add_argument("--size", type=int, default=64)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--npz", default="")
    ap.add_argument("--checkpoint", default="")
    ap.add_argument("--out", default="")
    ap.add_argument("--tf32", type=int, default=1, help="--impl reference on a GPU: cuDNN TF32 convolutions (torch's default) on/off")
    args = ap.parse_args()
    import torch
    if args.impl == "b200":
        sys.path.insert(0, ROOT)
        import unet_convlstm_b200 as pkg
        pkg.set_precision(args.precision)
    else:
        torch.backends.cudnn.allow_tf32 = bool(args.tf32)
        torch.backends.cuda.matmul.allow_tf32 = bool(args.tf32)
    {"overfit": run_overfit, "main": run_main, "get_metrics": run_get_metrics}[args.script](args)


if __name__ == "__main__":
    main()
