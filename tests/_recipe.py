"""Shared test helpers: seeded weight recipe, synthetic inputs, config builders.

Golden fixtures never store weights (237 M parameters would not fit in git): both
``tests/golden/make_golden.py`` (which runs the unmodified reference) and the tests
fill a ``state_dict`` from names + shapes with :func:`fill_state_dict`, so the same
weights are reproduced anywhere without the reference being present.
"""
from __future__ import annotations

import argparse
import zlib

import torch

# ---- UNet configurations used by fixtures and tests -------------------------------------
# "tiny*" shrink the template UNet (model_channels 128 -> 32) so CPU oracles finish in
# well under a second; "cfg1" is BASELINE.json configs[0] (Template-BBDM.yaml, 64x64, B=4).
UNET_CONFIGS = {
    # concat-conditioned pixel model, attention at ds=2,4 (input/output blocks) + middle
    "tiny_pixel": dict(image_size=16, in_channels=6, model_channels=32, out_channels=3,
                       num_res_blocks=2, attention_resolutions=(2, 4), channel_mult=(1, 4, 8),
                       conv_resample=True, dims=2, num_heads=8, num_head_channels=32,
                       use_scale_shift_norm=True, resblock_updown=True,
                       use_spatial_transformer=False, context_dim=None,
                       condition_key="SpatialRescaler"),
    # unconditioned latent model, template attention_resolutions (never match -> middle only)
    "tiny_latent": dict(image_size=16, in_channels=4, model_channels=32, out_channels=4,
                        num_res_blocks=2, attention_resolutions=(32, 16, 8), channel_mult=(1, 4, 8),
                        conv_resample=True, dims=2, num_heads=8, num_head_channels=32,
                        use_scale_shift_norm=True, resblock_updown=True,
                        use_spatial_transformer=False, context_dim=None, condition_key="nocond"),
    # tensor-core-aligned small model (all conv channel counts multiples of 64, head dim 64)
    "mid_pixel": dict(image_size=32, in_channels=6, model_channels=64, out_channels=3,
                      num_res_blocks=1, attention_resolutions=(4,), channel_mult=(1, 2, 4),
                      conv_resample=True, dims=2, num_heads=8, num_head_channels=64,
                      use_scale_shift_norm=True, resblock_updown=True,
                      use_spatial_transformer=False, context_dim=None,
                      condition_key="SpatialRescaler"),
    # non-template switches: no scale-shift norm, conv up/downsample, new attention order
    "tiny_variant": dict(image_size=16, in_channels=3, model_channels=32, out_channels=3,
                         num_res_blocks=1, attention_resolutions=(2,), channel_mult=(1, 2),
                         conv_resample=True, dims=2, num_heads=4, num_head_channels=-1,
                         use_scale_shift_norm=False, resblock_updown=False,
                         use_new_attention_order=True, use_spatial_transformer=False,
                         context_dim=None, condition_key="nocond"),
    # cross-attention conditioning: SpatialTransformer blocks instead of AttentionBlocks (SURVEY 8(f) rank 4); the
    # transformers attend to the same 3-channel conditioning image that is concatenated to the input
    "tiny_st": dict(image_size=16, in_channels=6, model_channels=32, out_channels=3,
                    num_res_blocks=1, attention_resolutions=(2, 4), channel_mult=(1, 4, 8),
                    conv_resample=True, dims=2, num_heads=8, num_head_channels=32,
                    use_scale_shift_norm=True, resblock_updown=True,
                    use_spatial_transformer=True, transformer_depth=1, context_dim=3,
                    condition_key="SpatialRescaler"),
    # BASELINE configs[2..4] UNets (LBBDM-f4 / f8-variant / f16-variant, SURVEY section 8 cfg3-cfg5):
    # 64x64 latents, condition_key nocond; f16 has attention at ds=4 (6 AttentionBlocks, T=256)
    "lbbdm_f4": dict(image_size=64, in_channels=3, model_channels=128, out_channels=3, num_res_blocks=2,
                     attention_resolutions=(32, 16, 8), channel_mult=(1, 4, 8), conv_resample=True, dims=2,
                     num_heads=8, num_head_channels=64, use_scale_shift_norm=True, resblock_updown=True,
                     use_spatial_transformer=False, context_dim=None, condition_key="nocond"),
    "lbbdm_f8": dict(image_size=64, in_channels=4, model_channels=128, out_channels=4, num_res_blocks=2,
                     attention_resolutions=(32, 16, 8), channel_mult=(1, 4, 8), conv_resample=True, dims=2,
                     num_heads=8, num_head_channels=64, use_scale_shift_norm=True, resblock_updown=True,
                     use_spatial_transformer=False, context_dim=None, condition_key="nocond"),
    "lbbdm_f16": dict(image_size=64, in_channels=16, model_channels=128, out_channels=16, num_res_blocks=2,
                      attention_resolutions=(16, 8, 4), channel_mult=(1, 4, 8), conv_resample=True, dims=2,
                      num_heads=8, num_head_channels=64, use_scale_shift_norm=True, resblock_updown=True,
                      use_spatial_transformer=False, context_dim=None, condition_key="nocond"),
    # BASELINE configs[1]: the pixel template at UNet image_size 256 (T = 4096 attention in the middle block)
    "cfg2": dict(image_size=256, in_channels=6, model_channels=128, out_channels=3,
                 num_res_blocks=2, attention_resolutions=(32, 16, 8), channel_mult=(1, 4, 8),
                 conv_resample=True, dims=2, num_heads=8, num_head_channels=64,
                 use_scale_shift_norm=True, resblock_updown=True,
                 use_spatial_transformer=False, context_dim=None,
                 condition_key="SpatialRescaler"),
    "cfg1": dict(image_size=64, in_channels=6, model_channels=128, out_channels=3,
                 num_res_blocks=2, attention_resolutions=(32, 16, 8), channel_mult=(1, 4, 8),
                 conv_resample=True, dims=2, num_heads=8, num_head_channels=64,
                 use_scale_shift_norm=True, resblock_updown=True,
                 use_spatial_transformer=False, context_dim=None,
                 condition_key="SpatialRescaler"),
}


# torch CPU threads the fixtures are generated and checked with (fp32 summation order depends on it)
GOLDEN_THREADS = 8


def bb_namespace(unet: dict, *, num_timesteps=1000, mt_type="linear", objective="grad",
                 loss_type="l1", skip_sample=True, sample_type="linear", sample_step=200,
                 eta=1.0, max_var=1.0):
    """``config.model`` Namespace tree as utils.dict2namespace builds it from Template-BBDM.yaml."""
    ns = argparse.Namespace
    params = ns(mt_type=mt_type, objective=objective, loss_type=loss_type, skip_sample=skip_sample,
                sample_type=sample_type, sample_step=sample_step, num_timesteps=num_timesteps,
                eta=eta, max_var=max_var, UNetParams=ns(**unet))
    return ns(model_name="BrownianBridge", model_type="BBDM", latent_before_quant_conv=False,
              normalize_latent=False, only_load_latent_mean_std=False,
              BB=ns(params=params))


def fill_state_dict(shapes: dict, seed: int = 1234, dtype=torch.float32):
    """Deterministic weights from (name -> shape).

    >=2-D weights ~ N(0, 0.02) (what runners/utils.py:35-45 ``weights_init`` gives every
    Conv2d/Linear; also used for the Conv1d qkv / proj_out so attention is live, SURVEY Q3);
    1-D ``.weight`` (GroupNorm gamma) ~ 1 + 0.1 N(0,1); biases ~ 0.02 N(0,1).
    Schedule buffers (non-parameter float buffers of the bridge model) are left untouched by
    passing only UNet entries in ``shapes``.
    """
    out = {}
    for name in sorted(shapes):
        shape = tuple(shapes[name])
        g = torch.Generator().manual_seed((zlib.crc32(name.encode()) + seed) & 0x7FFFFFFF)
        r = torch.randn(shape, generator=g, dtype=torch.float32)
        if name.endswith(".weight") and len(shape) >= 2:
            v = 0.02 * r
        elif name.endswith(".weight"):
            v = 1.0 + 0.1 * r
        else:
            v = 0.02 * r
        out[name] = v.to(dtype)
    return out


def synth_images(shape, seed, device="cpu"):
    """clamp(N(0, 0.5), -1, 1) fp32 NCHW -- the synthetic paired images of BASELINE.md section 3."""
    g = torch.Generator().manual_seed(seed)
    return (0.5 * torch.randn(shape, generator=g)).clamp_(-1, 1).to(device)


def rel_dev(a: torch.Tensor, b: torch.Tensor) -> float:
    """max|a-b| / max|b| -- the deviation metric of SURVEY section 7 H1 / BASELINE north_star."""
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


# ---- VQGAN ends (SURVEY 8(f) rank 1): shrunken ddconfigs of Template-LBBDM-f*.yaml ---------------------------
VQGAN_CONFIGS = {
    # tensor-core paths: fused nin_shortcut, GEMM-composed AttnBlock (C=128, T=256), fused upsample conv, padded head
    "vq_tc": dict(embed_dim=3, n_embed=128,
                  ddconfig=dict(double_z=False, z_channels=3, resolution=32, in_channels=3, out_ch=3, ch=64,
                                ch_mult=(1, 2), num_res_blocks=1, attn_resolutions=[], dropout=0.0)),
    # CUDA-core conv paths (C=32), flash AttnBlocks (C=64) inside a level, separate shortcut conv, z_channels 4
    "vq_small": dict(embed_dim=4, n_embed=64,
                     ddconfig=dict(double_z=False, z_channels=4, resolution=32, in_channels=3, out_ch=3, ch=32,
                                   ch_mult=(1, 2), num_res_blocks=1, attn_resolutions=[16], dropout=0.0)),
}


def vqgan_namespace(cfg: dict):
    return dict(embed_dim=cfg["embed_dim"], n_embed=cfg["n_embed"], ckpt_path=None,
                ddconfig=argparse.Namespace(**cfg["ddconfig"]),
                lossconfig=argparse.Namespace(target="torch.nn.Identity"))


def vqgan_state_dict(shapes: dict, seed: int = 4321):
    """fill_state_dict + a codebook of O(1) entries (0.5 N(0,1), like a trained one) so that the nearest-code
    search is well conditioned (the ctor's uniform(+-1/n_e) init puts every code within fp32 noise of the others)."""
    sd = fill_state_dict(shapes, seed)
    sd["quantize.embedding.weight"] = sd["quantize.embedding.weight"] * 25.0
    return sd


# ---- LatentBrownianBridgeModel on the reference's f4 template, shrunk for a CPU test -----------------------------
def to_namespace(d):
    """Nested dicts -> nested argparse.Namespace, as the reference's config loader builds ``config.model``."""
    return argparse.Namespace(**{k: to_namespace(v) if isinstance(v, dict) else v for k, v in d.items()})


def lbbdm_small_config(condition_key: str):
    """``config.model`` of Template-LBBDM-f4.yaml (committed in tests/golden/lbbdm_templates.json) with a 32x32
    image -> 8x8x3 latent VQGAN, a two-level UNet and a 4-step schedule."""
    import copy
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "lbbdm_templates.json")) as f:
        m = copy.deepcopy(json.load(f)["Template-LBBDM-f4.yaml"]["model"])
    m["VQGAN"]["params"]["ckpt_path"] = None
    m["VQGAN"]["params"]["ddconfig"].update(resolution=32, ch=32, ch_mult=(1, 2, 2))
    m["VQGAN"]["params"]["n_embed"] = 64
    m["BB"]["params"]["UNetParams"].update(image_size=8, model_channels=32, num_head_channels=32, channel_mult=(1, 2),
                                           condition_key=condition_key, in_channels=6 if condition_key != "nocond" else 3)
    m["BB"]["params"]["sample_step"] = 4
    m["CondStageParams"].update(n_stages=2, in_channels=3, out_channels=3)
    return to_namespace(m)


def lbbdm_state_dict(sd: dict):
    """Seeded values for every parameter of a LatentBrownianBridgeModel state_dict (UNet, VQGAN, cond stage); the
    bridge's schedule buffers keep the values given."""
    out = dict(sd)
    for prefix, fill in (("denoise_fn.", lambda s: fill_state_dict(s, seed=7)), ("vqgan.", vqgan_state_dict),
                         ("cond_stage_model.", lambda s: fill_state_dict(s, seed=11))):
        shapes = {k[len(prefix):]: tuple(v.shape) for k, v in sd.items() if k.startswith(prefix)}
        out.update({prefix + k: v for k, v in fill(shapes).items()})
    return out
