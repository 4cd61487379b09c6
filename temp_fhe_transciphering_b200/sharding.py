"""Block sharding across GPUs (SURVEY.md 8(e)): every AES block is independent through all ten
rounds, so blocks are partitioned contiguously across ranks, keys are replicated per GPU, there is
no collective in the data path, and results are gathered once at the end.  The max mini-workload
reduces locally per rank and finishes with one tiny gather (16 LWE per rank).  The *_sharded_dev helpers at the end run
both mini-workloads on the transcipher output where it lies, in each rank's HBM."""
import numpy as np


def block_range(nblocks, rank, world):
    """Contiguous [b0, b1) of `nblocks` owned by `rank` (same split the stage executable uses)."""
    return nblocks * rank // world, nblocks * (rank + 1) // world


def shard_ciphertext(ct_bytes, rank, world):
    nblocks = len(ct_bytes) // 16
    b0, b1 = block_range(nblocks, rank, world)
    return bytes(ct_bytes[16 * b0:16 * b1]), b0, b1


def gather_results(local, nblocks, rank, world, dist=None, device=None):
    """Gather per-rank [b1-b0][128][2049] uint64 results to rank 0 -> [nblocks][128][2049] (None elsewhere).

    `dist` is torch.distributed (gloo on CPU tests, nccl on GPUs); with world == 1 it is not used."""
    local = np.ascontiguousarray(local, dtype=np.uint64)
    if world == 1:
        return local
    import torch
    sizes = [block_range(nblocks, r, world) for r in range(world)]
    maxb = max(b1 - b0 for b0, b1 in sizes)
    buf = torch.zeros((maxb, 128, 2049), dtype=torch.int64, device=device)
    if local.shape[0]:
        buf[: local.shape[0]] = torch.from_numpy(local.view(np.int64)).to(buf.device)
    outs = [torch.zeros_like(buf) for _ in range(world)] if rank == 0 else None
    if dist.get_backend() == "nccl":
        allb = [torch.zeros_like(buf) for _ in range(world)]
        dist.all_gather(allb, buf)
        outs = allb if rank == 0 else None
    else:
        dist.gather(buf, outs, dst=0)
    if rank != 0:
        return None
    parts = [outs[r][: sizes[r][1] - sizes[r][0]].cpu().numpy().view(np.uint64) for r in range(world)]
    return np.concatenate(parts, axis=0)


def pair_range(npairs, rank, world):
    """Contiguous [p0, p1) of the inner product's `npairs` (x_i, y_i) pairs owned by `rank`."""
    return npairs * rank // world, npairs * (rank + 1) // world


def shard_inner_product_values(lwe_bits, rank, world):
    """Rows of [nvals*16][2049] bit ciphertexts this rank needs for its partial inner product: its slice of the
    first half (x) followed by the same slice of the second half (y), i.e. again a (first half, second half) input."""
    a = np.asarray(lwe_bits, dtype=np.uint64).reshape(-1, 16, 2049)
    npairs = a.shape[0] // 2
    p0, p1 = pair_range(npairs, rank, world)
    return np.concatenate([a[p0:p1], a[npairs + p0:npairs + p1]], axis=0).reshape(-1, 2049)


def value_range(nvals, rank, world):
    """Contiguous [v0, v1) of the max workload's values owned by `rank`."""
    return nvals * rank // world, nvals * (rank + 1) // world


# ---- device-resident stage 8 across GPUs ----
#
# Each rank holds the transcipher output of its blocks, [b1-b0][128][2049] = values [8*b0, 8*b1) as [.][16][2049], in HBM.
# The max needs no exchange: every rank reduces its own values.  The inner product pairs value i (x) with value
# npairs + i (y); pair chunk k = pair_range(npairs, k, world) goes to rank sigma(k), which places the x and y rows of two
# consecutive chunks on ranks r and r + world/2 - exactly the ranks whose shards hold them when world is even and divides
# nblocks - so each rank computes one chunk and receives half of its partner's shard (DESIGN.md, "Stage 8 across GPUs").


def _sigma(k, world):
    return k // 2 if k % 2 == 0 else (world + 1) // 2 + k // 2


def inner_product_assignment(nblocks, world):
    """[(p0, p1)] per rank: the contiguous range of the 4*nblocks inner-product pairs that rank computes."""
    npairs = 4 * nblocks
    out = [None] * world
    for k in range(world):
        out[_sigma(k, world)] = pair_range(npairs, k, world)
    return out


def inner_product_exchange_plan(nblocks, world):
    """Every row range the inner product's assignment moves, as (src, dst, "x" | "y", src_off, dst_off, count): `count` values
    from value offset src_off of src's shard to value offset dst_off of dst's x or y rows.  Entries with src == dst are rows
    the rank already holds (copied locally, not sent).  Every rank derives the same list, in the same order."""
    npairs = 4 * nblocks
    shards = [tuple(8 * b for b in block_range(nblocks, r, world)) for r in range(world)]
    plan = []
    for dst, (p0, p1) in enumerate(inner_product_assignment(nblocks, world)):
        for which, base in (("x", 0), ("y", npairs)):
            lo, hi = base + p0, base + p1  # global values wanted
            for src, (v0, v1) in enumerate(shards):
                a, b = max(lo, v0), min(hi, v1)
                if a < b:
                    plan.append((src, dst, which, a - v0, a - lo, b - a))
    return plan


def exchange_inner_product_rows(local, nblocks, rank, world, dist):
    """This rank's (x, y) rows of its inner-product pairs, each [p1-p0][16][2049] on local's device.

    `local` is this rank's [b1-b0][128][2049] int64 tensor (block_range).  Rows held locally are sliced; the rest arrive
    point to point (isend/irecv; batch_isend_irecv under NCCL) from the ranks that hold them.  Under NCCL the transfers are
    ordered on torch's current stream, without a host synchronisation."""
    import torch
    p0, p1 = inner_product_assignment(nblocks, world)[rank]
    vals = local.reshape(-1, 16, local.shape[-1])
    x = torch.empty((p1 - p0, 16, local.shape[-1]), dtype=local.dtype, device=local.device)
    y = torch.empty_like(x)
    ops = []
    for src, dst, which, s, d, n in inner_product_exchange_plan(nblocks, world):
        rows = (x if which == "x" else y)[d:d + n]
        if src == dst == rank:
            rows.copy_(vals[s:s + n])
        elif src == rank:
            ops.append((dist.isend, vals[s:s + n], dst))
        elif dst == rank:
            ops.append((dist.irecv, rows, src))
    if ops and dist.get_backend() == "nccl":
        works = dist.batch_isend_irecv([dist.P2POp(op, t, peer) for op, t, peer in ops])
    else:
        works = [op(t, peer) for op, t, peer in ops]
    for w in works:
        w.wait()
    return x, y


def _combine_partials(part, rank, world, dist, combine):
    """All ranks' [16][2049] partials -> rank 0, which reduces them with combine(d_in, n, d_out); None on other ranks."""
    import torch
    if world == 1:
        return part
    allp = torch.empty((world * 16, part.shape[-1]), dtype=part.dtype, device=part.device)
    dist.all_gather(list(allp.chunk(world)), part)
    if rank != 0:
        return None
    out = torch.empty_like(part)
    combine(allp.data_ptr(), world, out.data_ptr())
    return out


def _check_stream(ctx, device):
    import torch
    assert ctx.stream == torch.cuda.current_stream(device).cuda_stream, \
        "the context must issue on torch's current stream of its device (ctx.set_stream(torch.cuda.current_stream().cuda_stream))"


def max_u16_sharded_dev(ctx, local, nblocks, rank, world, dist):
    """Encrypted max of all 8*nblocks values, each rank holding its transcipher output `local` ([b1-b0][128][2049] int64 on
    its GPU).  Every rank reduces its own values (cbs_max_u16_dev), the 16-ciphertext partials are gathered on the device
    and rank 0 combines them; returns the [16][2049] device tensor on rank 0, None elsewhere.  A rank without values
    contributes the trivial encryption of 0.  No ciphertext passes through host memory.

    The context's stream must be torch's current stream on that device (Context.set_stream): library calls and NCCL
    transfers are then ordered without host synchronisation.  `dist` is torch.distributed (unused when world == 1)."""
    import torch
    _check_stream(ctx, local.device)
    b0, b1 = block_range(nblocks, rank, world)
    part = torch.zeros((16, local.shape[-1]), dtype=torch.int64, device=local.device)
    if b1 > b0:
        ctx.max_u16_dev(local.data_ptr(), 8 * (b1 - b0), part.data_ptr())
    return _combine_partials(part, rank, world, dist, ctx.max_u16_dev)


def inner_product_u16_sharded_dev(ctx, local, nblocks, rank, world, dist, rows=None):
    """Encrypted sum_i (x_i * y_i mod 2^16) mod 2^16 over the 8*nblocks values (x = first half, y = second half), `local`
    as for max_u16_sharded_dev.  Each rank computes its pairs (inner_product_assignment) from the rows
    exchange_inner_product_rows brings it - or from `rows`, the (x, y) of an earlier exchange - and rank 0 sums the
    partials (cbs_sum_u16_dev); returns the [16][2049] device tensor on rank 0, None elsewhere.  Same stream requirement."""
    import torch
    _check_stream(ctx, local.device)
    x, y = rows if rows is not None else exchange_inner_product_rows(local, nblocks, rank, world, dist)
    part = torch.zeros((16, local.shape[-1]), dtype=torch.int64, device=local.device)
    if x.shape[0]:
        ctx.inner_product_u16_dev(x.data_ptr(), y.data_ptr(), x.shape[0], part.data_ptr())
    return _combine_partials(part, rank, world, dist, ctx.sum_u16_dev)
