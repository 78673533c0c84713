"""Training half of the N>1 path on CPU (SURVEY section 8 row a24 / 8e): two gloo ranks wrap the drop-in model in the
reference's ``DDP(net)`` (runners/BaseRunner.py:76), run the native training Functions (kernels emulated, tests only)
on their half of a fixed batch and step ``FusedAdam``.  DDP must see ordinary ``.grad`` tensors: after each step both
ranks hold bit-identical parameters, and they match a single process that trains on the whole batch."""
import os
import sys

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
STEPS, GLOBAL_BATCH = 2, 4


class _Step(torch.nn.Module):
    """forward == one p_losses call with caller-provided t / noise (BrownianBridgeModel.py:98-126), so the two
    layouts of the batch see the same randomness."""

    def __init__(self, net):
        super().__init__()
        self.net = net

    def forward(self, x, y, t, noise):
        return self.net.p_losses(x, y, y, t, noise)[0]


def _build():
    sys.path[:0] = [os.path.dirname(HERE), HERE]
    from _emu_backend import EmuBackend
    from _recipe import UNET_CONFIGS, bb_namespace, fill_state_dict
    from bbdm_b200 import optim
    from bbdm_b200.bridge import BridgeOps
    from model.BrownianBridge.BrownianBridgeModel import BrownianBridgeModel
    emu = EmuBackend()
    BridgeOps.backend_factory = staticmethod(lambda: emu)
    optim.FusedAdam.backend_factory = staticmethod(lambda: emu)
    from bbdm_b200 import train
    train.set_backend(emu)
    net = BrownianBridgeModel(bb_namespace(UNET_CONFIGS["mid_pixel"])).train()
    shapes = {k: tuple(v.shape) for k, v in net.denoise_fn.state_dict().items()}
    net.denoise_fn.load_state_dict(fill_state_dict(shapes, seed=1234))
    return net, emu, optim


def _batch(step):
    g = torch.Generator().manual_seed(100 + step)
    x = torch.randn(GLOBAL_BATCH, 3, 32, 32, generator=g).clamp_(-1, 1)
    y = torch.randn(GLOBAL_BATCH, 3, 32, 32, generator=g).clamp_(-1, 1)
    t = torch.randint(0, 1000, (GLOBAL_BATCH,), generator=g)
    nz = torch.randn(GLOBAL_BATCH, 3, 32, 32, generator=g)
    return x, y, t, nz


def _train(wrap, rows):
    net, emu, optim = _build()
    step_mod = wrap(_Step(net))
    # eps far above the gradients' rounding noise: with the default 1e-8 Adam turns the sign of a ~1e-10 gradient
    # (summation order of the two batch layouts) into a full +-lr step, which says nothing about the data path
    opt = optim.FusedAdam(net.get_parameters(), lr=1e-3, betas=(0.9, 0.999), eps=1e-3)
    for s in range(STEPS):
        x, y, t, nz = (a[rows] for a in _batch(s))
        opt.zero_grad()
        step_mod(x, y, t, nz).backward()
        opt.step()
    assert "adam_multi" in emu.calls and "conv_wgrad" in emu.calls          # the native path, not the stock graph
    return {n: p.detach().clone() for n, p in net.denoise_fn.named_parameters()}


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    per = GLOBAL_BATCH // world
    params = _train(lambda m: torch.nn.parallel.DistributedDataParallel(m), slice(rank * per, (rank + 1) * per))
    q.put((rank, {k: v.numpy() for k, v in params.items()}))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_ddp_training_matches_single_process(monkeypatch):
    from bbdm_b200 import optim, train
    from bbdm_b200.bridge import BridgeOps
    # the in-process _train() below installs the emulation backend process-wide: undo that when the test ends
    for cls in (BridgeOps, optim.FusedAdam):
        monkeypatch.setattr(cls, "backend_factory", cls.__dict__["backend_factory"])
    monkeypatch.setattr(train, "_BACKEND", train._BACKEND)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29000 + os.getpid() % 500
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = {}
    for _ in procs:
        rank, res = q.get(timeout=600)
        got[rank] = res
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    for k in got[0]:
        assert (got[0][k] == got[1][k]).all(), f"ranks diverged: {k}"
    torch.set_num_threads(2)
    want = _train(lambda m: m, slice(0, GLOBAL_BATCH))
    worst = 0.0
    for k, w in want.items():
        g = torch.from_numpy(got[0][k])
        worst = max(worst, float((g - w).abs().max()))
    assert worst < 2e-6, worst          # parameters moved by up to STEPS * lr = 2e-3
