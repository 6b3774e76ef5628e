"""N>1 host logic on CPU: world_size-2 gloo, sharding + the detection gather (no GPU needed)."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from yolact_b200.parallel import shard_range, pack_records, unpack_records, gather_detections


def test_shard_range_covers_batch():
    for gb in (1, 7, 8, 32, 64, 65):
        for ws in (1, 2, 4, 8):
            spans = [shard_range(gb, r, ws) for r in range(ws)]
            assert spans[0][0] == 0 and spans[-1][1] == gb
            assert all(spans[i][1] == spans[i + 1][0] for i in range(ws - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def _fake(rank, b, M=100, k=32):
    g = torch.Generator().manual_seed(100 + rank)
    return (torch.rand(b, M, 4, generator=g), torch.rand(b, M, k, generator=g) * 2 - 1,
            torch.randint(0, 80, (b, M), generator=g), torch.rand(b, M, generator=g),
            torch.randint(0, M + 1, (b,), generator=g, dtype=torch.int32))


def test_pack_unpack_roundtrip():
    rec = _fake(0, 3)
    out = unpack_records(pack_records(*rec), 100, 32)
    for a, b in zip(rec, out):
        assert torch.equal(a, b)


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    gb = 5                                   # global batch 5 over 2 ranks -> 3 + 2 (last shard padded)
    s, e = shard_range(gb, rank, world)
    mine = _fake(rank, e - s)
    out = gather_detections(*mine, per_rank_batch=3)
    if rank == 0:
        # numpy arrays travel by value: a tensor's storage is shared through a socket of this process, which may
        # already have exited when the parent unpickles it
        q.put([t.numpy().copy() for t in out])
    dist.barrier()
    dist.destroy_process_group()


def test_gather_detections_world2_gloo():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = [torch.from_numpy(a) for a in q.get(timeout=120)]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    r0, r1 = _fake(0, 3), _fake(1, 2)
    box, coef, cls, score, count = out
    assert box.shape[0] == 6
    assert torch.equal(box[:3], r0[0]) and torch.equal(box[3:5], r1[0])
    assert torch.equal(cls[:3], r0[2]) and torch.equal(cls[3:5], r1[2])
    assert torch.equal(count[:3], r0[4]) and torch.equal(count[3:5], r1[4]) and int(count[5]) == 0
    assert torch.equal(coef[3:5], r1[1]) and torch.equal(score[:3], r0[3])
