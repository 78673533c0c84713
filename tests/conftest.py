import importlib.util
import os
import sys
import types

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# An upstream BBDM checkout: tests/golden/make_golden*.py run it to regenerate the fixtures; the tests themselves
# run from the committed fixtures alone.
REF = os.environ.get("BBDM_REFERENCE", "")
for p in (REPO, os.path.join(REPO, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
os.environ.setdefault("PYTHONDONTWRITEBYTECODE", "1")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


def pytest_collection_modifyitems(config, items):
    import torch
    has_gpu = torch.cuda.is_available()
    for it in items:
        if "gpu" in it.keywords and not has_gpu:
            it.add_marker(pytest.mark.skip(reason="no CUDA device"))


def install_reference_shims():
    """sys.modules stubs the unmodified reference needs to import here (SURVEY section 8c).

    Nothing in the reference tree is touched.  The repo root stays AHEAD of the checkout
    on sys.path so ``model.BrownianBridge.{BrownianBridgeModel,LatentBrownianBridgeModel}``
    resolve to this repo's drop-in classes while every other reference module
    (runners.*, model.VQGAN.*, model.utils, datasets.*) resolves to the reference.
    """
    import torch.nn as nn
    if REF not in sys.path:
        sys.path.append(REF)
    if "pytorch_lightning" not in sys.modules:
        pl = types.ModuleType("pytorch_lightning")
        pl.LightningModule = nn.Module
        sys.modules["pytorch_lightning"] = pl
    if "torchsummary" not in sys.modules:
        ts = types.ModuleType("torchsummary")
        ts.summary = lambda *a, **k: None
        sys.modules["torchsummary"] = ts
    if "omegaconf" not in sys.modules:
        oc, dc, lc = (types.ModuleType(n) for n in
                      ("omegaconf", "omegaconf.dictconfig", "omegaconf.listconfig"))
        dc.DictConfig = type("DictConfig", (dict,), {})
        lc.ListConfig = type("ListConfig", (list,), {})
        oc.dictconfig, oc.listconfig = dc, lc
        sys.modules.update({"omegaconf": oc, "omegaconf.dictconfig": dc,
                            "omegaconf.listconfig": lc})
    ds = sys.modules.get("datasets")
    if ds is None or getattr(ds, "__path__", [None])[0] != REF + "/datasets":
        ds = types.ModuleType("datasets")
        ds.__path__ = [REF + "/datasets"]
        sys.modules["datasets"] = ds


def load_reference_module(alias, relpath):
    """Import a reference file under an alias (so it can coexist with the overlay)."""
    install_reference_shims()
    if alias in sys.modules:
        return sys.modules[alias]
    spec = importlib.util.spec_from_file_location(alias, os.path.join(REF, relpath))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[alias] = mod
    spec.loader.exec_module(mod)
    return mod
