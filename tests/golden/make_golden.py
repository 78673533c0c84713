#!/usr/bin/env python
"""Generate the committed golden fixtures by running the UNMODIFIED reference.

Needs an upstream BBDM checkout, named by BBDM_REFERENCE:

    BBDM_REFERENCE=<checkout> python tests/golden/make_golden.py            # small fixtures (seconds)
    BBDM_REFERENCE=<checkout> python tests/golden/make_golden.py --cfg1     # + full-size cfg1 fixture (~1 min CPU)

Writes ``tests/golden/*.npz`` / ``*.json``.  Weights are never stored: they are
regenerated from names+shapes by tests/_recipe.fill_state_dict (same code both sides).
Everything the reference computes here is CPU fp32 (true fp32, no TF32).
"""
import argparse
import hashlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import conftest  # noqa: E402
from _recipe import GOLDEN_THREADS, UNET_CONFIGS, bb_namespace, fill_state_dict, synth_images  # noqa: E402

torch.set_grad_enabled(False)


def build_ref(unet_name, **bb_kw):
    ref = conftest.load_reference_module("ref_bbdm", "model/BrownianBridge/BrownianBridgeModel.py")
    net = ref.BrownianBridgeModel(bb_namespace(UNET_CONFIGS[unet_name], **bb_kw)).eval()
    shapes = {k: tuple(v.shape) for k, v in net.denoise_fn.state_dict().items()}
    sd = fill_state_dict(shapes, seed=1234)
    net.denoise_fn.load_state_dict(sd, strict=True)
    return net


def schedule_kats():
    out = {}
    for name, kw in {
        "linear_200": dict(),
        "linear_100": dict(sample_step=100),
        "linear_noskip": dict(skip_sample=False),
        "sin_200": dict(mt_type="sin"),
        "linear_maxvar2_50": dict(max_var=2.0, sample_step=50),
    }.items():
        net = build_ref("tiny_latent", **kw)
        steps = net.steps.numpy().astype("<i8")
        ent = {"steps_sha256": hashlib.sha256(steps.tobytes()).hexdigest(),
               "steps_len": int(len(steps)),
               "steps_head": steps[:8].tolist(), "steps_tail": steps[-8:].tolist()}
        idx = [0, 1, 2, 499, 500, 997, 998, 999]
        ent["idx"] = idx
        for b in ("m_t", "m_tminus", "variance_t", "variance_tminus", "variance_t_tminus",
                  "posterior_variance_t"):
            v = getattr(net, b)
            ent[b] = [float.hex(float(v[i])) for i in idx]          # exact fp32 values
            ent[b + "_sha256"] = hashlib.sha256(v.numpy().astype("<f4").tobytes()).hexdigest()
        out[name] = ent
    with open(os.path.join(HERE, "schedule_kats.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("schedule_kats.json", {k: v["steps_sha256"][:12] for k, v in out.items()})


def unet_and_psample(unet_name, B, tag, bb_kw=None, step_ids=(3, -1), with_loop=True):
    """UNet forward, p_sample (mid + final), q_sample/p_losses, short loop -> npz."""
    bb_kw = dict(bb_kw or {})
    net = build_ref(unet_name, **bb_kw)
    u = UNET_CONFIGS[unet_name]
    cx = u["out_channels"]
    S = u["image_size"]
    x = synth_images((B, cx, S, S), seed=11)
    y = synth_images((B, cx, S, S), seed=12)
    ctx = None if u["condition_key"] == "nocond" else y
    data = {"x": x.numpy(), "y": y.numpy()}

    # --- UNet forward at a few timesteps (per-sample t, like training) ---
    t = torch.tensor([(17 + 311 * i) % 1000 for i in range(B)], dtype=torch.long)
    data["t"] = t.numpy()
    data["unet_out"] = net.denoise_fn(x, timesteps=t, context=ctx).numpy()

    # --- q_sample + p_losses with supplied noise ---
    g = torch.Generator().manual_seed(77)
    noise = torch.randn(x.shape, generator=g)
    data["q_noise"] = noise.numpy()
    x_t, obj = net.q_sample(x, y, t, noise)
    data["q_xt"], data["q_obj"] = x_t.numpy(), obj.numpy()
    loss, log = net.p_losses(x, y, ctx, t, noise)
    data["loss"] = np.float32(loss.item())
    data["x0_recon"] = log["x0_recon"].numpy()

    # --- single p_sample steps (mid-trajectory and final) ---
    nsteps = len(net.steps)
    for si in step_ids:
        i = si % nsteps
        xt = synth_images((B, cx, S, S), seed=100 + i)
        torch.manual_seed(5000 + i)
        out, x0r = net.p_sample(xt, y, ctx, i, clip_denoised=False)
        torch.manual_seed(5000 + i)
        nz = torch.randn_like(xt)          # the noise the reference drew (UNet draws none)
        data[f"ps{i}_xt"], data[f"ps{i}_noise"] = xt.numpy(), nz.numpy()
        data[f"ps{i}_out"], data[f"ps{i}_x0"] = out.numpy(), x0r.numpy()
        torch.manual_seed(5000 + i)
        outc, _ = net.p_sample(xt, y, ctx, i, clip_denoised=True)
        data[f"ps{i}_out_clip"] = outc.numpy()
    data["ps_ids"] = np.array([si % nsteps for si in step_ids])

    # --- short full loop with a private small schedule ---
    if with_loop:
        kw = dict(bb_kw)
        kw.update(sample_step=8)
        net8 = build_ref(unet_name, **kw)
        torch.manual_seed(4242)
        img = net8.sample(y, clip_denoised=True)
        torch.manual_seed(4242)
        noises = [torch.randn_like(y) for _ in range(len(net8.steps) - 1)]
        data["loop8_out"] = img.numpy()
        data["loop8_noise"] = torch.stack(noises).numpy()
        data["loop8_steps"] = net8.steps.numpy()
    path = os.path.join(HERE, f"{tag}.npz")
    np.savez_compressed(path, **data)
    print(tag, {k: getattr(v, "shape", v) for k, v in data.items() if k in ("unet_out", "loss")},
          f"{os.path.getsize(path) / 1e3:.0f} kB")


def mid_pixel_gradients():
    """Training step of the UNMODIFIED reference on mid_pixel (the fixture's x, y, t, q_noise): loss and the gradients
    of a spread of parameters (stem, a ResBlock's convs / norms / FiLM linear, attention qkv + proj, time MLP, head) ->
    mid_pixel_grads.npz.  Checked on the GPU against the native training path (tests/test_gpu_training.py)."""
    torch.set_grad_enabled(True)
    net = build_ref("mid_pixel").train()
    g = np.load(os.path.join(HERE, "mid_pixel.npz"))
    x, y, t, nz = (torch.from_numpy(g[k]) for k in ("x", "y", "t", "q_noise"))
    loss, _ = net.p_losses(x, y, y, t, nz)
    loss.backward()
    names = [n for n, _ in net.denoise_fn.named_parameters()]
    pick = [n for n in names if n.startswith(("time_embed.0", "input_blocks.0.0", "input_blocks.1.0.", "input_blocks.3.0.",
                                               "middle_block.1.", "output_blocks.2.0.in_layers.2", "output_blocks.5.0.skip",
                                               "out.0", "out.2"))]
    data = {"loss": np.float32(loss.item())}
    params = dict(net.denoise_fn.named_parameters())
    for n in pick:
        data["grad:" + n] = params[n].grad.detach().numpy()
    path = os.path.join(HERE, "mid_pixel_grads.npz")
    np.savez_compressed(path, **data)
    torch.set_grad_enabled(False)
    print("mid_pixel_grads", len(pick), "tensors", f"{os.path.getsize(path) / 1e3:.0f} kB")


def cfg2_full_size(B=1):
    """BASELINE configs[1] at FULL size (256x256 pixel BBDM, 200-step schedule): UNet forward, one mid-trajectory
    and the final p_sample of the unmodified reference.  Inputs are regenerated by the tests from the same seeds
    (synth_images / manual_seed), only the noise the reference drew and its outputs are stored (~5 MB)."""
    net = build_ref("cfg2")
    S, cx = 256, 3
    x = synth_images((B, cx, S, S), seed=11)
    y = synth_images((B, cx, S, S), seed=12)
    t = torch.tensor([(517 + 311 * i) % 1000 for i in range(B)], dtype=torch.long)
    data = {"t": t.numpy(), "unet_out": net.denoise_fn(x, timesteps=t, context=y).numpy()}
    nsteps = len(net.steps)
    ids = [100, nsteps - 1]
    for i in ids:
        xt = synth_images((B, cx, S, S), seed=100 + i)
        torch.manual_seed(5000 + i)
        out, x0r = net.p_sample(xt, y, y, i, clip_denoised=False)
        torch.manual_seed(5000 + i)
        nz = torch.randn_like(xt)
        data[f"ps{i}_noise"] = nz.numpy()
        data[f"ps{i}_out"], data[f"ps{i}_x0"] = out.numpy(), x0r.numpy()
    data["ps_ids"] = np.array(ids)
    path = os.path.join(HERE, "cfg2_b1.npz")
    np.savez_compressed(path, **data)
    print("cfg2_b1", f"{os.path.getsize(path) / 1e6:.1f} MB")


def reference_contracts():
    """Everything the CPU tests compare against that needs the reference's own Python modules or config files:

    - the ``model`` section of the three LBBDM templates and the state_dict names / shapes of the reference
      VQModel built from each (the checkpoint format ``bbdm_b200.vqgan.VQModel`` must load) -> lbbdm_templates.json
    - the reference's full sampling loop on fresh inputs (tests/test_oracle_pinned.py)
    - the reference LatentBrownianBridgeModel on the shrunken f4 template with seeded weights
      (tests/test_latent_model_host.py): state_dict names, parameter count, encode, sample, training loss
    -> reference_contracts.npz"""
    import yaml
    from _recipe import lbbdm_small_config, lbbdm_state_dict
    conftest.install_reference_shims()
    from utils import dict2namespace
    from model.VQGAN.vqgan import VQModel as RefVQ
    templates = {}
    for name in ("Template-LBBDM-f4.yaml", "Template-LBBDM-f8.yaml", "Template-LBBDM-f16.yaml"):
        with open(os.path.join(conftest.REF, "configs", name)) as f:
            model = yaml.load(f, Loader=yaml.FullLoader)["model"]
        params = dict(model["VQGAN"]["params"], ckpt_path=None)
        with torch.device("meta"):
            vq = RefVQ(**vars(dict2namespace({"p": params}).p))
        templates[name] = {"model": model, "vqgan_state_dict": {k: list(v.shape) for k, v in vq.state_dict().items()}}
    with open(os.path.join(HERE, "lbbdm_templates.json"), "w") as f:
        json.dump(templates, f, indent=1)

    data = {}
    for unet_name, bkw in (("tiny_pixel", dict(sample_step=20)),
                           ("tiny_latent", dict(objective="noise", skip_sample=False, num_timesteps=30))):
        net = build_ref(unet_name, **bkw)
        shapes = {k: tuple(v.shape) for k, v in net.denoise_fn.state_dict().items()}
        net.denoise_fn.load_state_dict(fill_state_dict(shapes, seed=99))
        y = synth_images((2, UNET_CONFIGS[unet_name]["out_channels"], 16, 16), seed=3)
        torch.manual_seed(7)
        data[f"{unet_name}_steps"] = net.steps.numpy()
        data[f"{unet_name}_sample"] = net.sample(y, clip_denoised=False).numpy()

    # a PURE reference pair: load the reference latent module while the dotted base-module name points at the
    # reference's own BrownianBridgeModel, then restore the overlay
    name = "model.BrownianBridge.BrownianBridgeModel"
    overlay = sys.modules.get(name)
    sys.modules[name] = conftest.load_reference_module("ref_bbdm", "model/BrownianBridge/BrownianBridgeModel.py")
    try:
        ref_mod = conftest.load_reference_module("ref_lbbdm", "model/BrownianBridge/LatentBrownianBridgeModel.py")
    finally:
        sys.modules.pop(name)
        if overlay is not None:
            sys.modules[name] = overlay
    for ck in ("nocond", "SpatialRescaler"):
        torch.manual_seed(0)
        ref = ref_mod.LatentBrownianBridgeModel(lbbdm_small_config(ck)).eval()
        sd = lbbdm_state_dict(ref.state_dict())
        ref.load_state_dict(sd)
        x = synth_images((2, 3, 32, 32), 1)
        xc = synth_images((2, 3, 32, 32), 2)
        data[f"{ck}_keys"] = np.array(sorted(sd))
        data[f"{ck}_n_params"] = np.int64(sum(p.numel() for p in ref.get_parameters()))
        data[f"{ck}_encode"] = ref.encode(xc, cond=True).numpy()
        torch.manual_seed(5)
        data[f"{ck}_sample"] = ref.sample(xc, clip_denoised=False).numpy()
        torch.manual_seed(9)
        data[f"{ck}_loss"] = np.float64(ref(x, xc)[0].item())
    path = os.path.join(HERE, "reference_contracts.npz")
    np.savez_compressed(path, **data)
    print("reference_contracts", f"{os.path.getsize(path) / 1e3:.0f} kB")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--cfg1", action="store_true")
    ap.add_argument("--contracts-only", action="store_true", help="only the reference model / config contracts")
    ap.add_argument("--cfg2-only", action="store_true", help="only the full-size 256x256 fixture (~2 min CPU)")
    ap.add_argument("--st-only", action="store_true", help="only the SpatialTransformer fixture")
    ap.add_argument("--grads-only", action="store_true", help="only the mid_pixel gradient fixture")
    a = ap.parse_args()
    torch.set_num_threads(GOLDEN_THREADS)
    if a.contracts_only:
        reference_contracts()
        sys.exit(0)
    if a.cfg2_only:
        cfg2_full_size()
        sys.exit(0)
    if a.grads_only:
        mid_pixel_gradients()
        sys.exit(0)
    if a.st_only:
        unet_and_psample("tiny_st", 2, "tiny_st", with_loop=False)
        sys.exit(0)
    schedule_kats()
    unet_and_psample("tiny_pixel", 2, "tiny_pixel")
    unet_and_psample("tiny_latent", 3, "tiny_latent", bb_kw=dict(objective="noise", loss_type="l2"))
    unet_and_psample("tiny_variant", 2, "tiny_variant", bb_kw=dict(objective="ysubx", eta=0.5))
    unet_and_psample("mid_pixel", 2, "mid_pixel")
    unet_and_psample("tiny_st", 2, "tiny_st", with_loop=False)          # SpatialTransformer / cross-attention UNet
    mid_pixel_gradients()
    reference_contracts()
    if a.cfg1:
        unet_and_psample("cfg1", 4, "cfg1", bb_kw=dict(sample_step=100), with_loop=False)
        # BASELINE configs[2..4] UNet shapes at a reduced batch (full channel widths / resolutions)
        for name in ("lbbdm_f4", "lbbdm_f8", "lbbdm_f16"):
            unet_and_psample(name, 2, name, with_loop=False)
