"""Pair assignment and row exchange of the device-resident multi-GPU inner product (sharding.inner_product_assignment,
inner_product_exchange_plan, exchange_inner_product_rows): pure-function checks over many shapes, and world-2 / world-3
gloo runs with tagged stand-in rows."""
import os
import sys

import torch.multiprocessing as mp

from conftest import ROOT

sys.path.insert(0, ROOT)
from temp_fhe_transciphering_b200 import sharding  # noqa: E402

SHAPES = [(nb, w) for nb in range(1, 41) for w in range(1, 9)]


def test_assignment_covers_every_pair_once_and_is_balanced():
    for nb, w in SHAPES:
        ranges = sharding.inner_product_assignment(nb, w)
        assert len(ranges) == w
        covered = sorted(p for p0, p1 in ranges for p in range(p0, p1))
        assert covered == list(range(4 * nb)), (nb, w)
        sizes = [p1 - p0 for p0, p1 in ranges]
        assert max(sizes) - min(sizes) <= 1, (nb, w, sizes)


def test_exchange_plan_delivers_exactly_the_rows_of_each_ranks_pairs():
    for nb, w in SHAPES:
        npairs = 4 * nb
        shard0 = [8 * sharding.block_range(nb, r, w)[0] for r in range(w)]
        got = {(r, which): {} for r in range(w) for which in "xy"}
        for src, dst, which, s, d, n in sharding.inner_product_exchange_plan(nb, w):
            b0, b1 = sharding.block_range(nb, src, w)
            assert 0 <= s and s + n <= 8 * (b1 - b0) and n > 0, (nb, w)
            for i in range(n):
                assert d + i not in got[(dst, which)], (nb, w, "row delivered twice")
                got[(dst, which)][d + i] = shard0[src] + s + i  # global value index
        for r, (p0, p1) in enumerate(sharding.inner_product_assignment(nb, w)):
            assert got[(r, "x")] == {i: p0 + i for i in range(p1 - p0)}, (nb, w, r)
            assert got[(r, "y")] == {i: npairs + p0 + i for i in range(p1 - p0)}, (nb, w, r)


def test_even_world_receives_half_a_shard_from_its_partner_only():
    for nb, w in SHAPES:
        if w % 2 or nb % w:
            continue
        shard = 8 * nb // w
        received = {r: {} for r in range(w)}
        for src, dst, which, s, d, n in sharding.inner_product_exchange_plan(nb, w):
            if src != dst:
                received[dst][src] = received[dst].get(src, 0) + n
        for r in range(w):
            partner = (r + w // 2) % w
            assert received[r] == {partner: shard // 2}, (nb, w, r, received[r])


def _worker(rank, world, port, nblocks, q):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from temp_fhe_transciphering_b200 import sharding
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    # stand-in transcipher output: every word of value v's rows carries v, word (bit, 1) carries the bit index
    b0, b1 = sharding.block_range(nblocks, rank, world)
    vals = torch.arange(8 * b0, 8 * b1, dtype=torch.int64).reshape(-1, 1, 1).expand(-1, 16, 2049).clone()
    vals[:, :, 1] = torch.arange(16)
    local = vals.reshape(b1 - b0, 128, 2049)
    x, y = sharding.exchange_inner_product_rows(local, nblocks, rank, world, dist)
    p0, p1 = sharding.inner_product_assignment(nblocks, world)[rank]
    npairs = 4 * nblocks
    ok = x.shape == y.shape == (p1 - p0, 16, 2049) and x.dtype == torch.int64
    if ok and p1 > p0:
        ok = (x[:, 0, 0].tolist() == list(range(p0, p1)) and y[:, 0, 0].tolist() == list(range(npairs + p0, npairs + p1))
              and bool((x[:, :, 1] == torch.arange(16)).all()) and bool((y[:, :, 1] == torch.arange(16)).all())
              and bool((x[:, :, 2:] == x[:, :1, :1]).all()) and bool((y[:, :, 2:] == y[:, :1, :1]).all()))
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_exchange_inner_product_rows_gloo():
    ctx = mp.get_context("spawn")
    for world, nblocks, port in ((2, 8, 29731), (2, 5, 29732), (3, 5, 29733), (3, 7, 29734)):
        q = ctx.Queue()
        procs = [ctx.Process(target=_worker, args=(r, world, port, nblocks, q)) for r in range(world)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(120)
            assert p.exitcode == 0
        results = dict(q.get(timeout=5) for _ in range(world))
        assert results == {r: True for r in range(world)}, (world, nblocks, results)
