#!/usr/bin/env python
"""bench.py -- denoising-steps/sec of the BBDM hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config cfg2] [--dump-outputs DIR]

One "step" = one p_sample at the configured batch: UNet forward + fused Brownian-bridge update
(+ the Gaussian draw), i.e. one iteration of the reference's p_sample_loop
(model/BrownianBridge/BrownianBridgeModel.py:171-221).  Workload at N=1: BASELINE configs[1],
pixel-space BBDM 256x256 RGB, batch 16, 200-step skip schedule, random-init weights, synthetic
paired images.  N>1: one process per GPU (torchrun), every rank samples its own batch of 16
(the test set shards with no collective, SURVEY section 8e) => weak scaling, value = sum over ranks.

Prints ONE JSON line (see the task contract): value (HBM-resident inputs), e2e (host buffers,
H2D + D2H inside the timed region), roofline (tcgen05 conv kernel family), cpu_baseline
(oracle port on the host cores, bounded sample), clocks, gpu_launches.

--dump-outputs DIR writes what the last timed step returned (rank 0) as DIR/<name>.npy, float32, so that two builds
can be compared output for output: inputs, weights and noise are seeded, identical from run to run for the same
arguments.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from

import numpy as np  # noqa: E402
import torch  # noqa: E402

CONFIGS = {
    # name: (UNet kwargs, batch, image size, sample_step, description)
    "cfg2": dict(unet=dict(image_size=256, in_channels=6, model_channels=128, out_channels=3, num_res_blocks=2,
                           attention_resolutions=(32, 16, 8), channel_mult=(1, 4, 8), conv_resample=True, dims=2,
                           num_heads=8, num_head_channels=64, use_scale_shift_norm=True, resblock_updown=True,
                           use_spatial_transformer=False, context_dim=None, condition_key="SpatialRescaler"),
                 batch=16, size=256, channels=3, sample_step=200,
                 name="pixel-BBDM 256x256 RGB, batch 16, 200-step skip sampling (BASELINE configs[1])",
                 flops_per_step=64.46e12),
    "cfg1": dict(unet=dict(image_size=64, in_channels=6, model_channels=128, out_channels=3, num_res_blocks=2,
                           attention_resolutions=(32, 16, 8), channel_mult=(1, 4, 8), conv_resample=True, dims=2,
                           num_heads=8, num_head_channels=64, use_scale_shift_norm=True, resblock_updown=True,
                           use_spatial_transformer=False, context_dim=None, condition_key="SpatialRescaler"),
                 batch=4, size=64, channels=3, sample_step=100,
                 name="pixel-BBDM 64x64 RGB, batch 4, 100 steps (BASELINE configs[0])",
                 flops_per_step=0.991e12),
    # BASELINE configs[2..4]: the latent UNets (the step metric is the UNet's p_sample; the VQGAN ends run once per
    # sampled batch and are timed separately, tools/bench_vqgan.py).  These are parity-test cases; bench lines for
    # them are informational.
    "cfg3": dict(unet=dict(image_size=64, in_channels=3, model_channels=128, out_channels=3, num_res_blocks=2,
                           attention_resolutions=(32, 16, 8), channel_mult=(1, 4, 8), conv_resample=True, dims=2,
                           num_heads=8, num_head_channels=64, use_scale_shift_norm=True, resblock_updown=True,
                           use_spatial_transformer=False, context_dim=None, condition_key="nocond"),
                 batch=32, size=64, channels=3, sample_step=200,
                 name="LBBDM-f4 latent 64x64x3, batch 32 per GPU, UNet sampling step (BASELINE configs[2] shape)",
                 flops_per_step=7.93e12),
    "cfg4": dict(unet=dict(image_size=64, in_channels=4, model_channels=128, out_channels=4, num_res_blocks=2,
                           attention_resolutions=(32, 16, 8), channel_mult=(1, 4, 8), conv_resample=True, dims=2,
                           num_heads=8, num_head_channels=64, use_scale_shift_norm=True, resblock_updown=True,
                           use_spatial_transformer=False, context_dim=None, condition_key="nocond"),
                 batch=64, size=64, channels=4, sample_step=200,
                 name="LBBDM-f8 latent 64x64x4, batch 64, sharded sampling step (BASELINE configs[3] shape)",
                 flops_per_step=15.86e12),
    "cfg5": dict(unet=dict(image_size=64, in_channels=16, model_channels=128, out_channels=16, num_res_blocks=2,
                           attention_resolutions=(16, 8, 4), channel_mult=(1, 4, 8), conv_resample=True, dims=2,
                           num_heads=8, num_head_channels=64, use_scale_shift_norm=True, resblock_updown=True,
                           use_spatial_transformer=False, context_dim=None, condition_key="nocond"),
                 batch=8, size=64, channels=16, sample_step=200,
                 name="LBBDM-f16 latent 64x64x16, batch 8, attention-heavy UNet (BASELINE configs[4] shape)",
                 flops_per_step=2.08e12),
}
METRIC = "denoising-steps/sec (UNet fwd) at 256^2 pixel-BBDM"

# VQGAN ends of the latent configs (Template-LBBDM-f4/f8/f16.yaml ddconfigs; cfg4 / cfg5 are the scaled variants of
# SURVEY section 8: f8 at 512^2 -> 64x64x4, f16 at 1024^2 -> 64x64x16), random init (ckpt_path None)
VQGAN_ENDS = {
    "cfg3": dict(image=256, embed_dim=3, n_embed=8192,
                 ddconfig=dict(double_z=False, z_channels=3, resolution=256, in_channels=3, out_ch=3, ch=128,
                               ch_mult=(1, 2, 4), num_res_blocks=2, attn_resolutions=[], dropout=0.0)),
    "cfg4": dict(image=512, embed_dim=4, n_embed=16384,
                 ddconfig=dict(double_z=False, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128,
                               ch_mult=(1, 2, 2, 4), num_res_blocks=2, attn_resolutions=[32], dropout=0.0)),
    "cfg5": dict(image=1024, embed_dim=16, n_embed=16384,
                 ddconfig=dict(double_z=False, z_channels=16, resolution=256, in_channels=3, out_ch=3, ch=128,
                               ch_mult=(1, 1, 2, 2, 4), num_res_blocks=2, attn_resolutions=[16], dropout=0.0)),
}


def namespace(unet, sample_step):
    import argparse as ap
    ns = ap.Namespace
    params = ns(mt_type="linear", objective="grad", loss_type="l1", skip_sample=True, sample_type="linear",
                sample_step=sample_step, num_timesteps=1000, eta=1.0, max_var=1.0, UNetParams=ns(**unet))
    return ns(model_name="BrownianBridge", model_type="BBDM", latent_before_quant_conv=False,
              normalize_latent=False, only_load_latent_mean_std=False, BB=ns(params=params))


def init_weights(unet, seed=1234):
    """reference ctor init + runners/utils.py:35-45 weights_init (N(0,0.02) on every Conv2d/Linear
    weight) under seed 1234, then attention proj_out ~ N(0,0.02) so attention is live
    (BASELINE.md section 3)."""
    import torch.nn as nn
    torch.manual_seed(seed)
    for m in unet.modules():
        if isinstance(m, (nn.Conv2d, nn.Linear)):
            nn.init.normal_(m.weight.data, 0.0, 0.02)
    for name, m in unet.named_modules():
        if name.endswith("proj_out"):
            nn.init.normal_(m.weight.data, 0.0, 0.02)


def synth(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return (0.5 * torch.randn(shape, generator=g)).clamp_(-1, 1)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.2 and len(r) >= 9] or [r for _, r in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = [float(r[1]) for r in rows]
        reasons = set()
        for r in rows:
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(rows[0][2]), "reasons": sorted(reasons),
                "samples": len(rows), "power_w_max": max(float(r[3]) for r in rows)}


DUMP_BYTES = 60 * 10**6          # --dump-outputs in all: under 64 MB with the .npy headers


def dump_outputs(out_dir, arrays):
    """Write each tensor as out_dir/<name>.npy in float32.  When they exceed DUMP_BYTES in all, each is replaced by
    the same share of its elements, at flat indices drawn from a fixed seed (so two runs sample the same places)."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(t.numel() * 4 for t in arrays.values())
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if total > DUMP_BYTES:
            k = a.numel() * DUMP_BYTES // total
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:k].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle port (pure torch CPU restatement of the reference algorithm) on the host
# cores.  /root/reference is Python and does not exist on the GPU box, so kind = "port".
# ------------------------------------------------------------------------------------------
def cpu_step_time(cfg, sample_batch, n_steps, threads, budget_s=100.0):
    """Mean seconds per p_sample step of the oracle port at `sample_batch` images, after one warm-up
    step; at most n_steps timed steps and at most ~budget_s seconds of timed CPU work.
    Returns (seconds_per_step, steps_timed)."""
    from oracle import bbdm_oracle as O
    from bbdm_b200.unet import UNetModel
    torch.set_num_threads(threads)
    unet = UNetModel(**cfg["unet"])
    init_weights(unet)
    sd = {k: v.detach() for k, v in unet.state_dict().items()}
    ocfg = O.unet_cfg(**cfg["unet"])
    bufs, steps = O.make_schedule(sample_step=cfg["sample_step"])
    S, C = cfg["size"], cfg["channels"]
    y = synth((sample_batch, C, S, S), 1)
    x = synth((sample_batch, C, S, S), 2)
    ctx = None if cfg["unet"]["condition_key"] == "nocond" else y
    times = []
    with torch.no_grad():
        for i in range(max(1, n_steps) + 1):                      # first iteration = warm-up
            nz = torch.randn(x.shape)
            t0 = time.perf_counter()
            x, _ = O.p_sample(sd, ocfg, bufs, steps, 3 + i, x, y, ctx, nz, prefix="")
            times.append(time.perf_counter() - t0)
            if i >= 1 and sum(times[1:]) + times[-1] > budget_s:
                break
    timed = times[1:]
    return statistics.mean(timed), len(timed)


def host_threads():
    """All the host threads torch's CPU kernels can use productively: physical cores (SMT siblings
    only slow the fp32 conv/GEMM kernels down)."""
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
    except Exception:
        n = None
    return int(n or os.cpu_count() or 1)


def run_reference_arm(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    sb = 1 if cfg["batch"] > 4 else cfg["batch"]
    per, n_timed = cpu_step_time(cfg, sb, max(1, args.steps), threads)
    scale = cfg["batch"] / sb
    ms = per * scale * 1e3
    val = 1e3 / ms
    sample = (f"{n_timed} p_sample step(s) (bounded to ~100 s of CPU work) on {sb} of the {cfg['batch']} images (time scaled x{scale:g}), "
              f"after 1 warm-up step; oracle port (torch CPU fp32), {threads} threads")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["name"], "batch_per_gpu": cfg["batch"], "parallelism": "cpu"},
            "cpu_baseline": {"value": val, "unit": "steps/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
def run_ends(args, cfg):
    """End-to-end LBBDM sampling (BASELINE configs[2..4]): images -> VQGAN encode -> the full skip-sampling loop
    (one captured CUDA graph per step) -> quantize + VQGAN decode -> images, through
    LatentBrownianBridgeModel.sample() -- the call BBDMRunner.sample_to_eval makes (BBDMRunner.py:240) -- with the
    condition batch coming from pinned host memory and the result copied back inside the timed region.
    value = sample_step * batches / time, i.e. the same denoising-steps/s metric with both ends included."""
    import argparse as ap
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from bbdm_b200 import cabi
    from model.BrownianBridge.LatentBrownianBridgeModel import LatentBrownianBridgeModel
    vq = VQGAN_ENDS[args.config]
    ns = namespace(cfg["unet"], cfg["sample_step"])
    ns.VQGAN = ap.Namespace(params=ap.Namespace(ckpt_path=None, embed_dim=vq["embed_dim"], n_embed=vq["n_embed"],
                                                ddconfig=ap.Namespace(**vq["ddconfig"]),
                                                lossconfig=ap.Namespace(target="torch.nn.Identity")))
    torch.manual_seed(0)          # the constructor's default init (biases) too: identical weights from run to run
    net = LatentBrownianBridgeModel(ns).eval()
    init_weights(net.denoise_fn)
    torch.manual_seed(4321)
    with torch.no_grad():
        for n, p in net.vqgan.named_parameters():
            if p.dim() >= 2:
                p.normal_(0, 0.02)
        net.vqgan.quantize.embedding.weight.normal_(0, 0.5)
    net = net.to(dev)
    B, S = cfg["batch"], vq["image"]
    xc_host = synth((B, 3, S, S), 3000 + rank).pin_memory()
    out_host = torch.empty((B, 3, S, S)).pin_memory()

    def one_batch():
        xc = xc_host.to(dev, non_blocking=True)
        img = net.sample(xc, clip_denoised=False)
        out_host.copy_(img, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    import contextlib
    import io
    with contextlib.redirect_stderr(io.StringIO()):            # tqdm bars of the loop
        one_batch()                                            # warm-up: weight packing, pools, graph capture
        barrier()
        clocks = ClockSampler(local)
        clocks.start()
        time.sleep(0.3)
        n0 = cabi.LAUNCHES["n"]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        barrier()
        e0.record()
        for _ in range(args.batches):
            one_batch()
        e1.record()
        barrier()
        clk = clocks.stop(t0, time.time())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"images": out_host})
    ms = e0.elapsed_time(e1) / args.batches
    if dist is not None:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    net._bridge.backend().check_fault()
    # the ends alone (same tensors), for the breakdown
    xc = xc_host.to(dev)
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    with torch.no_grad():
        z = net.encode(xc, cond=True)
        net.decode(z, cond=False)
        torch.cuda.synchronize()
        e[0].record()
        z = net.encode(xc, cond=True)
        e[1].record()
        net.decode(z, cond=False)
        e[2].record()
    torch.cuda.synchronize()
    n_steps = cfg["sample_step"]
    if rank == 0:
        nbytes = B * 3 * S * S * 4
        val = world * n_steps * 1e3 / ms
        line = {"metric": METRIC, "value": val, "unit": "steps/s", "n_gpus": world, "steps": n_steps * args.batches,
                "warmup": n_steps, "ms_per_step": ms / n_steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16x3 / fp16x3 split tensor-core products, fp32 accumulate (fp32-class)",
                "data": "synthetic",
                "config": {"workload": cfg["name"] + " -- END TO END through LatentBrownianBridgeModel.sample(): VQGAN encode + "
                                       f"{n_steps}-step loop + quantize/decode, images {S}x{S}", "batch_per_gpu": B,
                           "parallelism": f"dp{world} (sharded sampling, no collective)",
                           "ms_per_batch": ms, "encode_ms": e[0].elapsed_time(e[1]), "decode_ms": e[1].elapsed_time(e[2]),
                           "loop_ms": ms - e[0].elapsed_time(e[2]), "images_per_s": world * B * 1e3 / ms},
                "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": nbytes / n_steps,
                        "d2h_bytes_per_step": nbytes / n_steps, "ms_per_step": ms / n_steps,
                        "note": "host images in, host images out, per sampled batch (bytes amortised over the loop's steps)"},
                "gpu_launches": (cabi.LAUNCHES["n"] - n0), "clocks": clk}
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", default="cfg2", choices=list(CONFIGS))
    ap.add_argument("--precision", default="split3", choices=["split3", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-convs", default=None, help="write per-conv-launch shape/time/TFLOPs (profiled step) to this file")
    ap.add_argument("--graph", action="store_true", help="also time CUDA-graph replays of the captured sampling step")
    ap.add_argument("--ends", action="store_true", help="latent configs: end-to-end sample() incl. VQGAN encode / decode")
    ap.add_argument("--batches", type=int, default=1, help="--ends: sampled batches in the timed region")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the native implementation only")
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        return run_reference_arm(args, cfg)
    if args.ends:
        assert args.config in VQGAN_ENDS, "--ends needs a latent config (cfg3, cfg4, cfg5)"
        return run_ends(args, cfg)
    assert args.warmup >= 3, "timing rules: W >= 3"
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from bbdm_b200 import cabi
    from bbdm_b200.bridge import BridgeOps
    from bbdm_b200.engine import UNetEngine
    from model.BrownianBridge.BrownianBridgeModel import BrownianBridgeModel

    class ProfilingBackend(cabi.CudaBackend):
        """Same kernels; optionally brackets every tcgen05 conv launch with CUDA events on the
        launching stream so the roofline numbers are measured live."""
        record = False
        events = []

        def conv_umma(self, **kw):
            if not ProfilingBackend.record:
                return super().conv_umma(**kw)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            super().conv_umma(**kw)
            e1.record()
            if kw.get("weights_per_image"):
                # Winograd F(4x4,3x3) position GEMMs (B = 36 positions, H*W = tiles): the reference algorithm is the
                # 3x3 conv over 16 pixels per tile (the kernel does 4x fewer MACs); the two transform kernels are
                # timed into the same family below (wino_input / wino_output)
                flops = 2.0 * kw["H"] * kw["W"] * 16 * kw["Cout"] * 9 * kw["Cin"]
            elif kw.get("upsample2x"):
                # reference algorithm: 3x3 conv on the 2x-upsampled tensor (the kernel does 2.25x fewer MACs)
                flops = 2.0 * kw["B"] * 4 * kw["H"] * kw["W"] * kw["Cout"] * 9 * kw["Cin"]
            else:
                flops = 2.0 * kw["B"] * kw["H"] * kw["W"] * kw["Cout"] * (kw["taps"] * kw["Cin"] + kw.get("Cin2", 0))
            ProfilingBackend.events.append((e0, e1, flops, {k: kw[k] for k in ("B", "H", "W", "Cin", "Cout", "taps")} |
                                            {"Cin2": kw.get("Cin2", 0), "up2": bool(kw.get("upsample2x")), "res": kw.get("res_mode", 0),
                                             "wino": bool(kw.get("weights_per_image"))}))

        def _timed_transform(self, name, fn, *a, **kw):
            if not ProfilingBackend.record:
                return fn(*a, **kw)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn(*a, **kw)
            e1.record()
            ProfilingBackend.events.append((e0, e1, 0.0, {"transform": name}))     # time counts, no extra FLOPs

        def wino_input(self, *a, **kw):
            return self._timed_transform("wino_input", super().wino_input, *a, **kw)

        def wino_output(self, *a, **kw):
            return self._timed_transform("wino_output", super().wino_output, *a, **kw)

    BridgeOps.backend_factory = staticmethod(lambda: ProfilingBackend())
    torch.manual_seed(0)          # the constructor's default init (biases) too: identical weights from run to run
    net = BrownianBridgeModel(namespace(cfg["unet"], cfg["sample_step"])).eval()
    init_weights(net.denoise_fn)
    net = net.to(dev)
    if args.precision != "split3":
        be = net._bridge.backend()
        object.__setattr__(net.denoise_fn, "_engine", UNetEngine(net.denoise_fn, backend=be, precision=args.precision))
    B, S, C = cfg["batch"], cfg["size"], cfg["channels"]
    y_host = synth((B, C, S, S), 1000 + rank).pin_memory()
    x_host = synth((B, C, S, S), 2000 + rank).pin_memory()
    out_host = torch.empty((B, C, S, S)).pin_memory()
    y = y_host.to(dev)
    n_sched = len(net.steps)

    def ctx_of(t):
        return None if cfg["unet"]["condition_key"] == "nocond" else t

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing: K consecutive steps of the loop ---------------------------------
    x = x_host.to(dev)
    for i in range(args.warmup):
        x, _ = net.p_sample(x, y, ctx_of(y), 5 + i)
    barrier()
    clocks = ClockSampler(local)
    clocks.start()
    time.sleep(0.3)
    n0 = cabi.LAUNCHES["n"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    e0.record()
    for i in range(args.steps):
        x, x0 = net.p_sample(x, y, ctx_of(y), (10 + i) % (n_sched - 1))
    e1.record()
    barrier()
    t_wall1 = time.time()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"x_prev": x, "x0_recon": x0})        # p_sample's (x_{t-1}, x0 estimate)
    launches = cabi.LAUNCHES["n"] - n0
    ms_dev = max_over_ranks(e0.elapsed_time(e1)) / args.steps

    # ---- end to end: host buffers, H2D of the step inputs + D2H of the result every step -----------
    for i in range(2):
        xd = x_host.to(dev, non_blocking=True)
        yd = y_host.to(dev, non_blocking=True)
        o, _ = net.p_sample(xd, yd, ctx_of(yd), 7)
        out_host.copy_(o, non_blocking=True)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for i in range(args.steps):
        xd = x_host.to(dev, non_blocking=True)
        yd = y_host.to(dev, non_blocking=True)
        o, _ = net.p_sample(xd, yd, ctx_of(yd), (10 + i) % (n_sched - 1))   # the public API call of the loop body
        out_host.copy_(o, non_blocking=True)
        torch.cuda.current_stream().synchronize()                        # the D2H must have landed before the host reads it
        x_host.copy_(out_host)                                           # next step's host-side input
    e3.record()
    barrier()
    clk = clocks.stop(t_wall0, time.time())
    ms_e2e = max_over_ranks(e2.elapsed_time(e3)) / args.steps
    net._bridge.backend().check_fault()

    # ---- CUDA-graph replay of the captured step (what p_sample_loop / sample() executes) ------------
    graph_ms = None
    if args.graph:
        st = net._bridge._step_graph(y, ctx_of(y), False)
        st["x"].copy_(x)
        st["coef"].copy_(net._bridge.coef_table()[10].to(dev))
        st["t"].fill_(int(net.steps[10]))
        for _ in range(2):
            st["noise"].normal_()
            st["graph"].replay()
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(args.steps):
            st["noise"].normal_()
            st["graph"].replay()
        g1.record()
        barrier()
        graph_ms = max_over_ranks(g0.elapsed_time(g1)) / args.steps

    # ---- roofline of the dominant kernel family (tcgen05 implicit-GEMM conv), one profiled step -----
    ProfilingBackend.record, ProfilingBackend.events = True, []
    x2, _ = net.p_sample(x, y, ctx_of(y), 20)
    torch.cuda.synchronize()
    ProfilingBackend.record = False
    conv_ms = sum(e[0].elapsed_time(e[1]) for e in ProfilingBackend.events)
    conv_flops = sum(e[2] for e in ProfilingBackend.events)
    if args.dump_convs and rank == 0:
        with open(args.dump_convs, "w") as f:
            for e0_, e1_, fl, shp in ProfilingBackend.events:
                ms_ = e0_.elapsed_time(e1_)
                f.write(json.dumps({**shp, "ms": ms_, "algo_tflops": fl / ms_ / 1e9}) + "\n")
    n_conv = sum(1 for e in ProfilingBackend.events if "transform" not in e[3])
    n_wino = sum(1 for e in ProfilingBackend.events if e[3].get("wino"))
    wino_tf_ms = sum(e[0].elapsed_time(e[1]) for e in ProfilingBackend.events if "transform" in e[3])
    peaks, peak_src = load_peaks()
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
    achieved_tf = conv_flops / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
    traffic = traffic_src = None
    for tp in ("r02_conv_traffic.json", "r01_conv_traffic.json"):
        tp = os.path.join(ROOT, "profiles", tp)
        if os.path.exists(tp):    # dram__bytes_read.sum + dram__bytes_write.sum per conv_umma launch, mean over the launches of
            traffic = json.load(open(tp)).get("dram_bytes_per_launch_mean")      # one ncu --set full capture of this command
            traffic_src = os.path.relpath(tp, ROOT)
            break
    # GPU library baseline (SURVEY 8d "the real bar"): the same architecture on stock PyTorch kernels, measured by
    # tools/bench_torchlib.py on a B200 of this pool (separate process: its fp32 row peaks at 183 GB of HBM)
    library = None
    lp = os.path.join(ROOT, "profiles", "r02_torch_library_baseline_%s.json" % args.config)
    if not os.path.exists(lp):
        lp = os.path.join(ROOT, "profiles", "r01_torch_library_baseline_%s.json" % args.config)
    if os.path.exists(lp):
        library = {"source": os.path.relpath(lp, ROOT) + " (tools/bench_torchlib.py, same pool, not this run)",
                   "rows": [{k: r.get(k) for k in ("mode", "ms_per_step", "steps_per_s")} for r in json.load(open(lp)).get("rows", [])]}
    roofline = {"bound": "tensor", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": achieved_tf / peak_tf, "traffic": traffic, "traffic_source": traffic_src,
                "kernel": "conv_umma_kernel (tcgen05 implicit-GEMM conv, %d launches/step, %d of them Winograd F(4x4,3x3) "
                          "position GEMMs whose input/output transform kernels -- %.2f ms/step -- are included in kernel_ms)"
                          % (n_conv, n_wino, wino_tf_ms),
                "algorithmic_flops_per_step": conv_flops, "kernel_ms_per_step": conv_ms,
                "share_of_step": conv_ms / ms_dev if ms_dev else None,
                "peak_source": peak_src + ", bf16 sustained",
                "note": ("algorithmic FLOPs (2*M*N*K of the reference conv); precision mode '%s' issues %dx the executed "
                         "MACs on the tensor pipe; Winograd layers execute 1/4, fused-upsample layers 1/2.25 of the "
                         "reference MACs" % (args.precision, 3 if args.precision == "split3" else 1))}

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            threads = host_threads()
            sb = 1 if B > 4 else B
            per, _ = cpu_step_time(cfg, sb, 1, threads)
            scale = B / sb
            cpu = {"value": 1.0 / (per * scale), "unit": "steps/s", "cores": threads, "kind": "port",
                   "sample": f"1 p_sample step on {sb} of the {B} images (time scaled x{scale:g}) after 1 warm-up; "
                             f"oracle port (torch CPU fp32)"}
        nbytes = B * C * S * S * 4
        line = {"metric": METRIC, "value": world * 1e3 / ms_dev, "unit": "steps/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16x3 (split-bf16 tensor-core products, fp32 accumulate: fp32-class)" if args.precision == "split3" else "bf16",
                "data": "synthetic",
                "config": {"workload": cfg["name"], "batch_per_gpu": B, "image": [C, S, S], "parallelism": f"dp{world} (sharded sampling, no collective)",
                           "precision": args.precision,
                           "l2": "working set larger than L2: every step streams the 0.95 GB of split-bf16 weights"
                                 + (" and 0.5-1.3 GB activation tensors" if args.config == "cfg2" else ""),
                           "graph_replay_ms_per_step": graph_ms,
                           "activation_pool_gb": net.denoise_fn.engine().pool_bytes() / 1e9,
                           "img_steps_per_s": world * B * 1e3 / ms_dev,
                           "unet_tflops_per_s": world * cfg["flops_per_step"] / (ms_dev * 1e-3) / 1e12},
                "e2e": {"value": world * 1e3 / ms_e2e, "unit": "steps/s", "h2d_bytes_per_step": 2 * nbytes,
                        "d2h_bytes_per_step": nbytes, "ms_per_step": ms_e2e},
                "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu, "gpu_library_baseline": library,
                "clocks": clk}
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
