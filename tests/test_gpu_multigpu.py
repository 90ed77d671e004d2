"""Multi-GPU data-plane tests (SURVEY.md §8e; VERDICT r1 "missing" #7, ADVICE r1 high/medium): world_size-2 NCCL, one
process per GPU, spawned from the test.  Skipped on machines with fewer than two GPUs.

  * per-shard parity: rank r's shard of a sharded sample() == a SINGLE-GPU run of that shard's inputs with that shard's seed
    (parallel.shard_range / rank_seed / gather_tokens used for real)
  * the weights every rank computes with are the broadcast ones: Paella and VQModel outputs on the receiving rank equal the
    source rank's bit for bit (the receiver's own parameters are deliberately DIFFERENT, so a skipped broadcast cannot pass)
  * a corrupted receive is detected by the checksum all-reduce
"""
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__))))
    from helpers import load_golden
    from paella_b200 import parallel as P
    from paella_b200 import utils as U
    from paella_b200.modules import Paella
    from paella_b200.synth import rerandomize_, synthetic_conditioning
    from paella_b200.vqgan import VQModel
    cfg, sd, g = load_golden("paella_tiny.npz")
    m = Paella(**cfg).eval()
    if rank == 0:
        m.load_state_dict(sd)               # only the source holds the real weights; receivers keep their random init
    m = m.to(dev)
    m.pack_weights(broadcast_src=0)
    vq = VQModel(levels=2, bottleneck_blocks=2, c_hidden=32, c_latent=4, codebook_size=64).eval()
    if rank == 0:
        rerandomize_(vq.state_dict(), seed=3)
    else:
        rerandomize_(vq.state_dict(), seed=99)
    vq = vq.to(dev)
    vq.pack_weights(broadcast_src=0)

    total, H = 6, 8
    kw = dict(byt5_embd=cfg["byt5_embd"], clip_embd=cfg["clip_embd"])
    cond, uncond = synthetic_conditioning(total, 5, seed=7, **kw)
    lo, hi = P.shard_range(total, rank, world)
    c = {k: v[lo:hi].to(dev) for k, v in cond.items()}
    u = {k: v[lo:hi].to(dev) for k, v in uncond.items()}
    torch.manual_seed(P.rank_seed(100, rank))
    toks = U.sample(m, c, (hi - lo, H, H), u, steps=3, renoise_steps=2)
    full = P.gather_tokens(toks, [P.shard_range(total, r, world)[1] - P.shard_range(total, r, world)[0] for r in range(world)])
    idx = torch.randint(0, 64, (2, 4, 4), device=dev, generator=torch.Generator(device=dev).manual_seed(5))
    img = vq.decode_indices(idx)
    imgs = [torch.empty_like(img) for _ in range(world)]
    dist.all_gather(imgs, img)
    # corrupted receive -> detected
    bad = m._blob.clone()
    if rank == 1:
        bad[12345 % bad.numel()] ^= 1
    caught = False
    try:
        P.assert_same_across_ranks(P.blob_checksum(bad), "blob")
    except RuntimeError:
        caught = True
    if rank == 0:
        ret["full"] = full.cpu()
        ret["vq_equal"] = bool(torch.equal(imgs[0], imgs[1]))
        ret["vq_nontrivial"] = float(imgs[0].std())
    ret[f"caught{rank}"] = caught
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_per_shard_parity_and_broadcast_weights():
    import torch.multiprocessing as mp
    from helpers import load_golden
    from paella_b200 import parallel as P
    from paella_b200 import utils as U
    from paella_b200.modules import Paella
    from paella_b200.synth import synthetic_conditioning
    world = 2
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    assert ret["caught0"] and ret["caught1"]
    assert ret["vq_equal"] and ret["vq_nontrivial"] > 1e-3
    # single-GPU reference runs of each shard with that shard's seed
    cfg, sd, g = load_golden("paella_tiny.npz")
    m = Paella(**cfg).to("cuda:0").eval()
    m.load_state_dict(sd)
    total, H = 6, 8
    cond, uncond = synthetic_conditioning(total, 5, seed=7, byt5_embd=cfg["byt5_embd"], clip_embd=cfg["clip_embd"])
    for r in range(world):
        lo, hi = P.shard_range(total, r, world)
        c = {k: v[lo:hi].to("cuda:0") for k, v in cond.items()}
        u = {k: v[lo:hi].to("cuda:0") for k, v in uncond.items()}
        torch.manual_seed(P.rank_seed(100, r))
        want = U.sample(m, c, (hi - lo, H, H), u, steps=3, renoise_steps=2).cpu()
        assert torch.equal(ret["full"][lo:hi], want), f"shard {r} differs from its single-GPU run"
