"""Multi-GPU path on hardware: images sharded by batch across ranks (one process per GPU, NCCL), the only collective is
the final all_gather of detection records -- the gathered result must equal the single-GPU run on the whole batch
(the analogue of CustomDataParallel.gather, the reference's eval.py:630-634): same counts, same class ids rank for
rank, boxes / scores / coefficients to 1e-4 (a shard of 2 images and a batch of 5 may get different tile plans from
the autotuner -- e.g. stream-K splits the reduction differently -- so the last bits of the fp32 sums differ).  Skipped with fewer than 2 GPUs; the
host logic alone is covered on CPU by tests/test_parallel_gloo.py."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def test_pack_records_kernel_matches_the_host_layout():
    from yolact_b200.parallel import pack_records, unpack_records
    g = torch.Generator().manual_seed(3)
    b, M, k = 3, 100, 32
    rec = (torch.rand(b, M, 4, generator=g), torch.rand(b, M, k, generator=g) * 2 - 1, torch.randint(0, 80, (b, M), generator=g),
           torch.rand(b, M, generator=g), torch.randint(0, M + 1, (b,), generator=g, dtype=torch.int32))
    host = pack_records(*rec)                                  # torch ops on CPU tensors
    dev = pack_records(*[t.cuda() for t in rec])               # yb_pack_detections
    assert torch.equal(dev.cpu(), host)
    for a, c in zip(rec, unpack_records(dev, M, k)):
        assert torch.equal(a, c.cpu())


def _worker(rank, world, port, q):
    os.environ.update({"MASTER_ADDR": "127.0.0.1", "MASTER_PORT": str(port), "RANK": str(rank), "WORLD_SIZE": str(world)})
    import torch.distributed as dist
    import yolact_b200
    from oracle.weights import deterministic_input, deterministic_state_dict
    from yolact_b200.config import CONFIGS
    from yolact_b200.parallel import gather_detections, shard_range
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    cfg = CONFIGS["yolact_resnet50_config"].copy()
    yolact_b200.cfg.replace(cfg.copy())
    net = yolact_b200.Yolact(cfg, precision="f16x3")
    net.detect.use_fast_nms = True
    net.load_state_dict(deterministic_state_dict(net.state_dict(), 0))
    net.eval()
    gb, size = 5, 256                                          # 5 images over `world` ranks: uneven shards, padded gather
    x = deterministic_input(gb, size, size, 77)
    s, e = shard_range(gb, rank, world)
    per_rank = (gb + world - 1) // world
    box, coef, cls, score, count, _ = net.infer_padded(x[s:e].to(dev))
    out = gather_detections(box, coef, cls, score, count, per_rank_batch=per_rank)
    torch.cuda.synchronize()
    if rank == 0:
        full = net.infer_padded(x.to(dev))[:5]                # the same images on ONE GPU
        torch.cuda.synchronize()
        # numpy arrays travel by value: a tensor's storage is shared through a socket of this process, which may
        # already have exited when the parent unpickles it
        q.put(([t.cpu().numpy() for t in out], [t.cpu().numpy() for t in full],
               [shard_range(gb, r, world) for r in range(world)], per_rank))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_run_plus_nccl_gather_equals_single_gpu():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2 if n < 4 else 4
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    gathered, full, spans, per_rank = q.get(timeout=600)
    gathered, full = [torch.from_numpy(a) for a in gathered], [torch.from_numpy(a) for a in full]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    names = ("box", "coef", "cls", "score", "count")
    for r, (a, b) in enumerate(spans):
        rows = slice(r * per_rank, r * per_rank + (b - a))     # rank-major rows of the gather <-> images [a, b)
        for name, g, f in zip(names, gathered, full):
            if name in ("cls", "count"):
                assert torch.equal(g[rows], f[a:b]), "rank %d %s differs from the single-GPU run" % (r, name)
            else:
                d = float((g[rows] - f[a:b]).abs().max())
                assert d < 1e-4, "rank %d %s differs from the single-GPU run by %.2e" % (r, name, d)
        pad = slice(r * per_rank + (b - a), (r + 1) * per_rank)
        assert int(gathered[4][pad].sum()) == 0                # padded rows of a short shard carry count 0
    assert int(full[4].min()) > 0
