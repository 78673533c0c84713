"""LatentBrownianBridgeModel drop-in (SURVEY section 8 row a23) against the UNMODIFIED reference class:
same config (Template-LBBDM-f4.yaml shrunk), same seeded weights -> state_dict names, get_parameters, encode,
sample, training loss, apply contracts.  The reference's results are stored by tests/golden/make_golden.py in
reference_contracts.npz.  CPU: the bridge kernels and the VQGAN engine run on the oracle-backed emulation backend
(tests only)."""
import os

import numpy as np
import pytest
import torch

import conftest
from _emu_backend import EmuBackend
from _recipe import lbbdm_small_config, lbbdm_state_dict, rel_dev, synth_images

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("condition_key", ["nocond", "SpatialRescaler"])
def test_latent_model_matches_reference(condition_key, monkeypatch):
    from bbdm_b200.bridge import BridgeOps
    from bbdm_b200.cond import SpatialRescaler
    from bbdm_b200.vqgan_engine import VQGANEngine
    monkeypatch.setattr(BridgeOps, "backend_factory", staticmethod(lambda: EmuBackend()))
    monkeypatch.setattr(SpatialRescaler, "backend_factory", staticmethod(lambda: EmuBackend()))
    import model.BrownianBridge.LatentBrownianBridgeModel as mine_mod
    assert mine_mod.__file__.startswith(conftest.REPO)
    # CPU tensors take the kernel path too, through the emulated backend
    monkeypatch.setattr(mine_mod.LatentBrownianBridgeModel, "_native", lambda self, fn, x, *a: fn(x, *a))
    g = {k: v[()] if v.ndim == 0 else v for k, v in
         np.load(os.path.join(GOLD, "reference_contracts.npz")).items() if k.startswith(condition_key + "_")}

    torch.manual_seed(0)
    mine = mine_mod.LatentBrownianBridgeModel(lbbdm_small_config(condition_key)).eval()
    mine.__dict__["_vq_eng"] = VQGANEngine(mine.vqgan, backend=EmuBackend())
    sd = lbbdm_state_dict(mine.state_dict())
    assert sorted(sd) == g[f"{condition_key}_keys"].tolist()      # identical key set (checkpoint format)
    mine.load_state_dict(sd)
    assert all(not p.requires_grad for p in mine.vqgan.parameters())
    assert sum(p.numel() for p in mine.get_parameters()) == g[f"{condition_key}_n_params"]

    x = synth_images((2, 3, 32, 32), 1)
    xc = synth_images((2, 3, 32, 32), 2)
    assert rel_dev(mine.encode(xc, cond=True), torch.from_numpy(g[f"{condition_key}_encode"])) < 1e-4
    torch.manual_seed(5)
    got = mine.sample(xc, clip_denoised=False)
    want = torch.from_numpy(g[f"{condition_key}_sample"])
    assert got.shape == want.shape == (2, 3, 32, 32)
    # the decoder quantises to the nearest codebook entry: an exact match of the decoded image means the
    # latents agreed closely enough to select the same codes everywhere
    assert rel_dev(got, want) < 1e-3
    lw = float(g[f"{condition_key}_loss"])
    torch.manual_seed(9)
    lg, log = mine(x, xc)
    assert abs(lw - float(lg)) < 1e-5 * abs(lw)
    assert lg.requires_grad and "x0_recon" in log
    imgs, one = mine.sample(xc, clip_denoised=False, sample_mid_step=True)
    assert len(imgs) == len(mine.steps) + 1 and len(one) == len(mine.steps) and imgs[0].device.type == "cpu"
    assert mine.apply(lambda m: None) is mine and mine.get_ema_net() is mine
