"""-m gpu: the call sequence of the reference runner (runners/BaseRunner.py:59-79,173-192,405-419 and
runners/DiffusionBasedModelRunners/BBDMRunner.py:21-29,169,240-253) on a real GPU, restated here because the runner's
source is not part of this repository; the model and EMA classes are reached through the same imports the runner
makes (the namespace-package overlays): construct -> .to(device) -> apply(weights_init) -> EMA register
-> [forward, backward, optimizer step, EMA update] x n -> EMA apply_shadow -> sample -> restore -> image files ->
checkpoint round trip."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn

from _recipe import UNET_CONFIGS, bb_namespace, synth_images

pytestmark = pytest.mark.gpu
DEV = "cuda"
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def weights_init(m):                       # what runners/utils.py:35-45 does to Conv2d / Linear modules
    name = m.__class__.__name__
    if name.find("Conv2d") != -1 or name.find("Linear") != -1:
        nn.init.normal_(m.weight.data, 0.0, 0.02)


def test_runner_call_sequence_on_gpu(tmp_path):
    from PIL import Image
    from bbdm_b200 import output
    from bbdm_b200.optim import FusedAdam, FusedEMA
    from model.BrownianBridge.BrownianBridgeModel import BrownianBridgeModel
    from runners.base.EMA import EMA                        # BaseRunner's import: resolves to this repo's overlay
    assert EMA is FusedEMA and BrownianBridgeModel.__module__ == "model.BrownianBridge.BrownianBridgeModel"
    assert sys.modules[BrownianBridgeModel.__module__].__file__.startswith(REPO)
    torch.manual_seed(1234)
    ns = bb_namespace(UNET_CONFIGS["mid_pixel"], sample_step=6)
    net = BrownianBridgeModel(ns).to(DEV)
    net.apply(weights_init)
    for n, p in net.denoise_fn.named_parameters():          # make the zero-initialised attention projection live
        if n.endswith("proj_out.weight"):
            nn.init.normal_(p.data, 0.0, 0.02)
    ema = EMA(0.995)
    ema.register(net)
    assert list(ema.shadow) == [n for n, p in net.named_parameters() if p.requires_grad]
    opt = FusedAdam(net.get_parameters(), lr=1e-4, weight_decay=0.0, betas=(0.9, 0.999))
    x, x_cond = synth_images((4, 3, 32, 32), 1).to(DEV), synth_images((4, 3, 32, 32), 2).to(DEV)
    losses = []
    for step in range(3):
        net.train()
        loss, log = net(x, x_cond)
        assert loss.dim() == 0 and "x0_recon" in log
        opt.zero_grad()
        loss.backward()
        opt.step()
        ema.update(net, with_decay=step >= 1)               # BaseRunner.step_ema: no decay before start_ema_step
        losses.append(float(loss))
    assert all(np.isfinite(losses))
    before = {n: p.data_ptr() for n, p in net.named_parameters()}
    ema.apply_shadow(net)
    net.eval()
    torch.manual_seed(7)
    sample = net.sample(x_cond, clip_denoised=False)
    ema.restore(net)
    assert {n: p.data_ptr() for n, p in net.named_parameters()} == before
    assert sample.shape == x.shape and torch.isfinite(sample).all()
    net._bridge.backend().check_fault()
    # sample_to_eval's image files: one conversion launch for the batch, async writers, reference bytes
    writer = output.AsyncImageWriter(workers=2)
    names = [f"{i}.png" for i in range(4)]
    output.save_image_batch(sample, str(tmp_path), names, to_normal=True, writer=writer)
    writer.close()
    for i, n in enumerate(names):
        img = sample[i].detach().clone().mul_(0.5).add_(0.5).clamp_(0, 1.).mul_(255).add_(0.5).clamp_(0, 255)
        want = img.permute(1, 2, 0).to("cpu", torch.uint8).numpy()
        assert np.array_equal(np.asarray(Image.open(tmp_path / n)), want)
    # checkpoint round trip (BaseRunner.py:141-170): model + EMA + optimizer states reload into fresh objects
    ck = {"model": net.state_dict(), "ema": ema.shadow, "optimizer": opt.state_dict()}
    torch.save(ck, tmp_path / "ck.pth")
    ck = torch.load(tmp_path / "ck.pth", map_location="cpu")
    net2 = BrownianBridgeModel(ns).to(DEV)
    net2.load_state_dict(ck["model"])
    ema2 = EMA(0.995)
    ema2.register(net2)
    ema2.shadow = ck["ema"]
    ema2.reset_device(net2)
    opt2 = torch.optim.Adam(net2.get_parameters(), lr=1e-4)       # a stock optimizer takes the fused one's state
    opt2.load_state_dict(ck["optimizer"])
    ema2.apply_shadow(net2)
    net2.eval()
    torch.manual_seed(7)
    assert torch.equal(net2.sample(x_cond, clip_denoised=False), sample)


def test_model_on_non_default_device_index():
    """The reference's single-GPU launcher moves the model to cuda:N without set_device (main.py:124): every kernel,
    TMA descriptor, stream and captured graph must follow the tensors' device.  Needs >= 2 GPUs (skips otherwise)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    from model.BrownianBridge.BrownianBridgeModel import BrownianBridgeModel
    from _recipe import fill_state_dict
    net0 = BrownianBridgeModel(bb_namespace(UNET_CONFIGS["mid_pixel"], sample_step=5)).eval()
    shapes = {k: tuple(v.shape) for k, v in net0.denoise_fn.state_dict().items()}
    net0.denoise_fn.load_state_dict(fill_state_dict(shapes, seed=1234))
    import copy
    net1 = copy.deepcopy(net0).to("cuda:1")
    net0 = net0.to("cuda:0")
    assert torch.cuda.current_device() == 0
    y = synth_images((2, 3, 32, 32), 3)
    g = torch.Generator().manual_seed(5)
    noises = [torch.randn(2, 3, 32, 32, generator=g) for _ in range(8)]      # the same Gaussian draws on both devices

    def run(net, dev):
        it = iter(noises)
        net._bridge.noise_source = lambda like: next(it).to(like.device)
        return net.sample(y.to(dev), clip_denoised=False)

    a = run(net0, "cuda:0")
    b = run(net1, "cuda:1")
    assert b.device.index == 1
    net1._bridge.backend().check_fault(device="cuda:1")
    eps1 = net1.denoise_fn(y.to("cuda:1"), timesteps=torch.tensor([7, 500], device="cuda:1"), context=y.to("cuda:1"))
    eps0 = net0.denoise_fn(y.to("cuda:0"), timesteps=torch.tensor([7, 500], device="cuda:0"), context=y.to("cuda:0"))
    print(f"\n[cuda:1 vs cuda:0] UNet max diff {float((eps1.cpu() - eps0.cpu()).abs().max()):.3e}; "
          f"sample max diff {float((a.cpu() - b.cpu()).abs().max()):.3e}")
    # same kernels, same inputs, same noise => identical results on either device
    assert torch.equal(eps0.cpu(), eps1.cpu())
    assert torch.equal(a.cpu(), b.cpu())
