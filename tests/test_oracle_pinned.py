"""Pin the oracle against the committed fixtures the unmodified reference generated (tests/golden/make_golden.py)."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from _recipe import GOLDEN_THREADS, UNET_CONFIGS, fill_state_dict, rel_dev, synth_images
from oracle import bbdm_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")
TAGS = {  # tag -> (unet config name, bridge kwargs used by make_golden.py)
    "tiny_pixel": ("tiny_pixel", {}),
    "tiny_latent": ("tiny_latent", dict(objective="noise", loss_type="l2")),
    "tiny_variant": ("tiny_variant", dict(objective="ysubx", eta=0.5)),
    "mid_pixel": ("mid_pixel", {}),
    "cfg1": ("cfg1", dict(sample_step=100)),
    "lbbdm_f4": ("lbbdm_f4", {}),        # BASELINE configs[2] UNet (latent 64x64x3, nocond)
    "lbbdm_f8": ("lbbdm_f8", {}),        # configs[3] UNet (64x64x4)
    "lbbdm_f16": ("lbbdm_f16", {}),      # configs[4] UNet (64x64x16, 6 attention blocks)
}


@pytest.fixture(autouse=True)
def _golden_thread_count():
    """The oracle's fp32 CPU convolutions sum in an order that depends on torch's thread count, which other tests in
    the session may change.  make_golden.py runs with GOLDEN_THREADS; at that count the oracle reproduces the
    fixtures bit for bit, and the 2e-6 tolerances below hold at any other count only by luck."""
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def oracle_state(unet_name, seed=1234):
    """UNet parameter shapes come from the PRODUCT module (independent of the reference),
    values from the seeded recipe."""
    from bbdm_b200.unet import UNetModel
    net = UNetModel(**UNET_CONFIGS[unet_name])
    shapes = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    return fill_state_dict(shapes, seed=seed)


def load(tag):
    p = os.path.join(GOLD, tag + ".npz")
    if not os.path.exists(p):
        pytest.skip(f"{tag}.npz not generated")
    return {k: torch.from_numpy(v) if v.ndim else v for k, v in np.load(p).items()}


def test_schedule_kats():
    kats = json.load(open(os.path.join(GOLD, "schedule_kats.json")))
    cases = {
        "linear_200": dict(),
        "linear_100": dict(sample_step=100),
        "linear_noskip": dict(skip_sample=False),
        "sin_200": dict(mt_type="sin"),
        "linear_maxvar2_50": dict(max_var=2.0, sample_step=50),
    }
    for name, kw in cases.items():
        bufs, steps = O.make_schedule(**kw)
        k = kats[name]
        s = steps.numpy().astype("<i8")
        assert hashlib.sha256(s.tobytes()).hexdigest() == k["steps_sha256"], name
        assert s[:8].tolist() == k["steps_head"] and s[-8:].tolist() == k["steps_tail"]
        for b, v in bufs.items():
            assert hashlib.sha256(v.numpy().astype("<f4").tobytes()).hexdigest() == k[b + "_sha256"], (name, b)
            assert [float.hex(float(v[i])) for i in k["idx"]] == k[b]
    # the survey's literal KAT (SURVEY.md section 8c)
    assert kats["linear_200"]["steps_sha256"] == \
        "ae04a57e690feed9e30cef016f2d727b7aea84906c016904c1561c9c20b1d896"
    _, steps = O.make_schedule()
    assert steps[:5].tolist() == [999, 993, 988, 983, 978] and steps[-5:].tolist() == [15, 10, 5, 1, 0]


@pytest.mark.parametrize("tag", ["tiny_pixel", "tiny_latent", "tiny_variant", "mid_pixel"])
def test_oracle_matches_reference_fixture(tag):
    unet_name, bkw = TAGS[tag]
    g = load(tag)
    cfg = O.unet_cfg(**UNET_CONFIGS[unet_name])
    sd = oracle_state(unet_name)
    objective = bkw.get("objective", "grad")
    eta = bkw.get("eta", 1.0)
    bufs, steps = O.make_schedule(sample_step=bkw.get("sample_step", 200))
    x, y, t = g["x"], g["y"], g["t"]
    ctx = None if cfg.condition_key == "nocond" else y

    out = O.unet_forward(sd, cfg, x, t, ctx)
    assert rel_dev(out, g["unet_out"]) < 2e-6

    xt, obj = O.q_sample(bufs, x, y, t, g["q_noise"], objective)
    assert torch.equal(xt, g["q_xt"]) and torch.equal(obj, g["q_obj"])
    loss, x0r = O.p_losses(sd, cfg, bufs, x, y, ctx, t, g["q_noise"], objective,
                           bkw.get("loss_type", "l1"), prefix="")
    assert abs(float(loss) - float(g["loss"])) <= 2e-6 * abs(float(g["loss"]))
    assert rel_dev(x0r, g["x0_recon"]) < 2e-6

    for i in g["ps_ids"].tolist():
        for clip, key in ((False, f"ps{i}_out"), (True, f"ps{i}_out_clip")):
            o, x0 = O.p_sample(sd, cfg, bufs, steps, i, g[f"ps{i}_xt"], y, ctx, g[f"ps{i}_noise"],
                               objective, eta, clip, prefix="")
            assert rel_dev(o, g[key]) < 2e-6, (i, clip)
        # elementwise part alone is bit-exact given the reference's own eps
        eps = g[f"ps{i}_xt"] - g[f"ps{i}_x0"] if objective == "grad" else None
        if eps is not None:
            o2, x02 = O.p_sample_update(bufs, steps, i, g[f"ps{i}_xt"], y, eps, g[f"ps{i}_noise"],
                                        objective, eta, False)
            assert rel_dev(o2, g[f"ps{i}_out"]) < 1e-6

    # 8-step loop with the reference's own noise sequence
    bufs8, steps8 = O.make_schedule(sample_step=8)
    assert steps8.tolist() == g["loop8_steps"].tolist()
    img = y
    for i in range(len(steps8)):
        nz = g["loop8_noise"][i] if i < len(steps8) - 1 else torch.zeros_like(y)
        img, _ = O.p_sample(sd, cfg, bufs8, steps8, i, img, y, ctx, nz, objective, eta, True, prefix="")
    assert rel_dev(img, g["loop8_out"]) < 1e-5


def test_oracle_spatial_transformer_matches_reference_fixture():
    """SpatialTransformer / cross-attention UNet (use_spatial_transformer, context_dim 3): the oracle's restatement of
    base/modules/attention.py against the fixture of the unmodified reference."""
    g = load("tiny_st")
    cfg = O.unet_cfg(**UNET_CONFIGS["tiny_st"])
    sd = oracle_state("tiny_st")
    bufs, steps = O.make_schedule()
    x, y, t = g["x"], g["y"], g["t"]
    assert rel_dev(O.unet_forward(sd, cfg, x, t, y), g["unet_out"]) < 2e-6
    for i in g["ps_ids"].tolist():
        o, _ = O.p_sample(sd, cfg, bufs, steps, i, g[f"ps{i}_xt"], y, y, g[f"ps{i}_noise"], prefix="")
        assert rel_dev(o, g[f"ps{i}_out"]) < 2e-6


@pytest.mark.parametrize("tag", ["cfg1", "lbbdm_f4", "lbbdm_f8", "lbbdm_f16"])
def test_oracle_matches_full_size_fixture(tag):
    """Full-size template UNets (237-258 M parameters): BASELINE configs[0] and the UNets of configs[2..4]."""
    g = load(tag)
    cfg = O.unet_cfg(**UNET_CONFIGS[tag])
    sd = oracle_state(tag)
    n = sum(v.numel() for v in sd.values())
    assert n == {"cfg1": 237_094_787}.get(tag, n) and 237e6 < n < 259e6      # 237.09 M / 258.1 M (SURVEY section 6)
    ctx = None if cfg.condition_key == "nocond" else g["y"]
    out = O.unet_forward(sd, cfg, g["x"], g["t"], ctx)
    assert rel_dev(out, g["unet_out"]) < 2e-6


def test_oracle_matches_cfg2_full_size_fixture():
    """BASELINE configs[1] at full size (256x256, B = 1): the oracle's UNet forward against the fixture the
    unmodified reference produced (one forward, ~20 s on 8 cores)."""
    g = load("cfg2_b1")
    cfg = O.unet_cfg(**UNET_CONFIGS["cfg2"])
    sd = oracle_state("cfg2")
    x = synth_images((1, 3, 256, 256), seed=11)
    y = synth_images((1, 3, 256, 256), seed=12)
    out = O.unet_forward(sd, cfg, x, g["t"], y)
    assert rel_dev(out, g["unet_out"]) < 2e-6


def test_oracle_matches_live_reference():
    """Fresh inputs (not in the other fixtures) through the unmodified reference's full sampling loop, stored by
    make_golden.py in reference_contracts.npz."""
    g = np.load(os.path.join(GOLD, "reference_contracts.npz"))
    for unet_name, bkw in (("tiny_pixel", dict(sample_step=20)),
                           ("tiny_latent", dict(objective="noise", skip_sample=False,
                                                num_timesteps=30))):
        sd = oracle_state(unet_name, seed=99)
        cfg = O.unet_cfg(**UNET_CONFIGS[unet_name])
        u = UNET_CONFIGS[unet_name]
        y = synth_images((2, u["out_channels"], 16, 16), seed=3)
        bufs, steps = O.make_schedule(num_timesteps=bkw.get("num_timesteps", 1000),
                                      skip_sample=bkw.get("skip_sample", True),
                                      sample_step=bkw.get("sample_step", 200))
        assert steps.tolist() == g[f"{unet_name}_steps"].tolist()
        torch.manual_seed(7)
        got = O.p_sample_loop(sd, cfg, bufs, steps, y, None, bkw.get("objective", "grad"), 1.0,
                              False, prefix="")
        assert rel_dev(got, torch.from_numpy(g[f"{unet_name}_sample"])) < 2e-5
