"""N>1 path on CPU: world_size-2 gloo processes each sample their DistributedSampler shard of a
synthetic test set (no data-path collective, SURVEY section 8e); the union must equal the
single-process result for the same indices.  Kernel backend emulated by the oracle (tests only)."""
import os
import sys

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))


def _build():
    sys.path[:0] = [os.path.dirname(HERE), HERE]
    from _emu_backend import EmuBackend
    from _recipe import UNET_CONFIGS, bb_namespace, fill_state_dict
    from bbdm_b200.bridge import BridgeOps
    from model.BrownianBridge.BrownianBridgeModel import BrownianBridgeModel
    BridgeOps.backend_factory = staticmethod(lambda: EmuBackend())
    net = BrownianBridgeModel(bb_namespace(UNET_CONFIGS["tiny_latent"], sample_step=3)).eval()
    shapes = {k: tuple(v.shape) for k, v in net.denoise_fn.state_dict().items()}
    net.denoise_fn.load_state_dict(fill_state_dict(shapes, seed=1234))
    return net


def _dataset():
    g = torch.Generator().manual_seed(5)
    return torch.randn(6, 4, 16, 16, generator=g).clamp_(-1, 1) * 0.5


def _sample_indices(net, data, idxs):
    out = {}
    for i in idxs:
        torch.manual_seed(1000 + i)                       # per-item seed => order independent
        out[i] = net.sample(data[i:i + 1], clip_denoised=False)
    return out


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    net = _build()
    data = _dataset()
    sampler = torch.utils.data.distributed.DistributedSampler(data, num_replicas=world, rank=rank, shuffle=False)
    res = _sample_indices(net, data, list(iter(sampler)))
    # timing-style reduction only (what bench.py does): max over ranks of a scalar
    t = torch.tensor([float(rank + 1)])
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    assert float(t) == world
    q.put((rank, {k: v.numpy() for k, v in res.items()}))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharded_sampling_matches_single_process(monkeypatch):
    from bbdm_b200.bridge import BridgeOps
    # the in-process _build() below installs the emulation backend process-wide: undo that when the test ends
    monkeypatch.setattr(BridgeOps, "backend_factory", BridgeOps.__dict__["backend_factory"])
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 500
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = {}
    for _ in procs:
        rank, res = q.get(timeout=300)
        assert not (set(res) & set(got)), "shards overlap"
        got.update(res)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert sorted(got) == list(range(6))
    torch.set_num_threads(2)
    net = _build()
    want = _sample_indices(net, _dataset(), range(6))
    for i in range(6):
        assert torch.equal(torch.from_numpy(got[i]), want[i]), i
