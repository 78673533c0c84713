"""Host logic of the sample_to_eval output path (bbdm_b200/output.py) through the emulation backend: byte-identical
PNG pixels with the reference expression, async writer, opt-in install into the unmodified runner modules."""
import os
import sys

import numpy as np
import pytest
import torch

from _emu_backend import EmuBackend
from bbdm_b200 import output as OUT


@pytest.fixture(autouse=True)
def _emu(monkeypatch):
    monkeypatch.setattr(OUT, "_be", EmuBackend())


def _ref_u8(image, to_normal=True):
    image = image.detach().clone()                      # runners/utils.py:67-74, verbatim expression
    if to_normal:
        image = image.mul_(0.5).add_(0.5).clamp_(0, 1.)
    return image.mul_(255).add_(0.5).clamp_(0, 255).permute(1, 2, 0).to('cpu', torch.uint8).numpy()


def test_batch_writer_produces_the_reference_bytes(tmp_path):
    from PIL import Image
    x = (0.7 * torch.randn(5, 3, 24, 20)).clamp_(-1.3, 1.3)
    w = OUT.AsyncImageWriter(workers=2, slots=2)
    names = [f"img_{i}.png" for i in range(5)]
    OUT.save_image_batch(x, str(tmp_path), names, to_normal=True, writer=w)
    OUT.save_image_batch(x[:2] * 0.5 + 0.5, str(tmp_path), ["raw0.png", "raw1.png"], to_normal=False, writer=w)
    w.close()
    for i, n in enumerate(names):
        assert np.array_equal(np.asarray(Image.open(tmp_path / n)), _ref_u8(x[i]))
    assert np.array_equal(np.asarray(Image.open(tmp_path / "raw1.png")), _ref_u8(x[1] * 0.5 + 0.5, to_normal=False))
    OUT.save_single_image(x[3], str(tmp_path), "single.png")
    assert np.array_equal(np.asarray(Image.open(tmp_path / "single.png")), _ref_u8(x[3]))


def test_install_rebinds_the_runner_functions(monkeypatch):
    """The reference's runners/utils.py defines save_single_image and BBDMRunner.py imports it by name: install()
    rebinds the name in both modules (stand-ins here, so the test needs no BBDM checkout)."""
    import types

    def save_single_image(image, save_path, file_name, to_normal=True):
        raise AssertionError("not rebound")

    for name in ("runners.utils", "runners.DiffusionBasedModelRunners.BBDMRunner"):
        mod = types.ModuleType(name)
        mod.save_single_image = save_single_image
        monkeypatch.setitem(sys.modules, name, mod)
    assert OUT.install() == 2
    assert sys.modules["runners.utils"].save_single_image is OUT.save_single_image
    assert sys.modules["runners.DiffusionBasedModelRunners.BBDMRunner"].save_single_image is OUT.save_single_image
