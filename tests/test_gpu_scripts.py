"""The reference's scripts, UNCHANGED, on top of this repository's train/unet.py (VERDICT r01 item 4, north_star "so
main.py, train/overfit_check.py and train/get_metrics.py run unchanged ... the overfit_check loss curve matches within
tolerance").  tools/run_reference.py executes the scripts from their own source files and only supplies environment:
import path order, stubs for the absent smp / matplotlib, the torch-2.11 keyword shims, constant overrides, a synthetic
NPZ.  The scripts are the reference project's, which this repository does not ship: these tests run when
B200_REFERENCE_DIR names a checkout of it and are skipped otherwise.

The A/B partner (--impl reference) is the reference's own train/unet.py through stock PyTorch on the same GPU
(cuDNN, TF32 off): same script, same seeds, same NPZ.
"""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOOL = os.path.join(ROOT, "tools", "run_reference.py")
sys.path.insert(0, os.path.dirname(TOOL))
try:
    import run_reference as RR
finally:
    sys.path.pop(0)
REF = RR.find_reference()

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(REF is None, reason="needs the reference project's scripts: set B200_REFERENCE_DIR")]


def _run(*args, timeout=1500):
    r = subprocess.run([sys.executable, TOOL, *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1]), r.stdout


@pytest.fixture(scope="module")
def reference_curve():
    res, _ = _run("overfit", "--impl", "reference", "--iters", "300", "--tf32", "0")
    assert res["unet_module"] == os.path.join(REF, "train", "unet.py")
    return {int(k): v for k, v in res["curve"].items()}


SUCCESS = 5e-4   # the script's own convergence criterion (overfit_check.py:116)


@pytest.mark.parametrize("precision,tol0", [("fp32", 1e-4), ("bf16", 2e-2)])
def test_overfit_check_loss_curve_matches_reference(reference_curve, precision, tol0):
    """overfit_check.run_overfit_test_and_save (overfit_check.py:36-139): masked-MSE loss printed every 100 iterations
    of AdamW on 16 sequences, base_ch 64 + skip ConvLSTMs, until the script's own success criterion (loss < 5e-4) stops
    it.  Iteration 0 is a pure forward pass and must agree to the mode's tolerance.  Iteration 100 must agree within
    a factor of two (the trajectories are chaotic: fp32 atomics in the split-K weight gradients already make two runs
    of the same build differ by 10-20 % there).  Beyond that the trajectory is chaotic in the reference itself -- measured on B200 (profiles/
    r02_overfit_curves.txt): reference fp32 0.000631 / 0.001037 / 0.000121 at 100 / 200 / 300, reference with cuDNN
    TF32 0.000534 / 0.000200 (stops at 200) -- so later points are not compared one by one: the run must reach the script's [SUCCESS] branch (loss < 5e-4)
    within 500 iterations (measured: at iteration 200 in both modes)."""
    res, out = _run("overfit", "--impl", "b200", "--precision", precision, "--iters", "500")
    assert res["unet_module"] == os.path.join(ROOT, "train", "unet.py")
    curve = {int(k): v for k, v in res["curve"].items()}
    assert abs(curve[0] - reference_curve[0]) <= tol0 * reference_curve[0], (curve, reference_curve)
    assert 0.5 * reference_curve[100] <= curve[100] <= 2.0 * reference_curve[100], (curve, reference_curve)
    # the script's own success criterion, reached like the reference reaches it (iteration 200-300 there)
    assert "[SUCCESS]" in out and min(curve.values()) < SUCCESS and max(curve) <= 500, curve


def test_main_and_get_metrics_run_unchanged():
    """main.py (__main__: split, AdamW, ReduceLROnPlateau(verbose=True), train_one_epoch, evaluate, best-checkpoint
    save) for two epochs on the B200 implementation, then train/get_metrics.py on the checkpoint it saved -- once with
    this implementation and once with the reference's own model class loading the SAME checkpoint (state_dict keys
    and tensor layouts interchange): the evaluation metrics agree."""
    res, out = _run("main", "--impl", "b200", "--epochs", "2", "--batch-size", "8", "--num-seq", "24")
    assert res["checkpoint"] and os.path.exists(res["checkpoint"]), out[-2000:]
    assert "Epoch 2/2" in out and "New best model" in out
    ours, _ = _run("get_metrics", "--impl", "b200", "--checkpoint", res["checkpoint"])
    ref, _ = _run("get_metrics", "--impl", "reference", "--checkpoint", res["checkpoint"])
    for k in ("MAE", "RMSE"):
        assert abs(ours["metrics"][k] - ref["metrics"][k]) <= 3e-2 * ref["metrics"][k] + 1e-3, (ours, ref)
