"""Device-resident stage 8 (cbs_max_u16_dev, cbs_max_u16_lut_dev, cbs_sum_u16_dev, cbs_inner_product_u16_dev) and its
multi-GPU composition (sharding.max_u16_sharded_dev / inner_product_u16_sharded_dev): bit-identical to the host-buffer
calls, correct after decryption, chained behind a device-resident transcipher with no host hop, asynchronous, and
rejecting bad arguments."""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu

V = 16 * 2049  # words of one u16 value (16 big LWE)


def _encrypt(keyset, vals, seed):
    bits = np.array([(v >> (15 - i)) & 1 for v in vals for i in range(16)], dtype=np.uint8)
    return keyset.encrypt_bits_big(bits, seed)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()


def _host(t):
    return t.cpu().numpy().view(np.uint64).reshape(-1, 2049)


def _decrypt(ct, keyset):
    import ref_io
    return ref_io.bits_to_u16(ref_io.decode_bit(ref_io.lwe_phase(np.asarray(ct).reshape(-1, 2049), keyset.glwe_sk)))


def _ip(vals):
    h = len(vals) // 2
    return sum((x * y) % 65536 for x, y in zip(vals[:h], vals[h:])) % 65536


def _rand_vals(n, seed):
    return np.random.default_rng(seed).integers(0, 65536, n).tolist()


@pytest.fixture
def sctx(ctx):
    """The session context issuing on a torch stream that is also torch's current stream (ordering without syncs)."""
    s = torch.cuda.Stream()
    ctx.set_stream(s.cuda_stream)
    with torch.cuda.stream(s):
        yield ctx
    ctx.set_stream(None)


def _out():
    return torch.empty((16, 2049), dtype=torch.int64, device="cuda")


def test_dev_calls_bit_identical_to_host_calls(sctx, keyset):
    ctx = sctx
    cases = [("max_u16", 8), ("max_u16", 33), ("max_u16_lut", 5), ("max_u16_lut", 33), ("sum_u16", 5), ("sum_u16", 33)]
    for k, (name, n) in enumerate(cases):
        vals = _rand_vals(n, 300 + k)
        lwe = _encrypt(keyset, vals, 400 + k)
        want = getattr(ctx, name)(lwe)
        d_in, d_out = _dev(lwe), _out()
        getattr(ctx, name + "_dev")(d_in.data_ptr(), n, d_out.data_ptr())
        got = _host(d_out)
        assert (got == want).all(), (name, n)
        expect = sum(vals) % 65536 if name == "sum_u16" else max(vals)
        assert _decrypt(got, keyset) == [expect], (name, n)
    for k, n in enumerate((8, 64)):
        vals = _rand_vals(n, 500 + k)
        lwe = _encrypt(keyset, vals, 600 + k)
        want = ctx.inner_product_u16(lwe)
        d_x, d_y, d_out = _dev(lwe[: n // 2 * 16]), _dev(lwe[n // 2 * 16:]), _out()  # two separate allocations
        ctx.inner_product_u16_dev(d_x.data_ptr(), d_y.data_ptr(), n // 2, d_out.data_ptr())
        got = _host(d_out)
        assert (got == want).all(), n
        assert _decrypt(got, keyset) == [_ip(vals)], n


def test_chained_after_ctr_transcipher_without_host_hop(sctx, keyset, aes_key):
    import aes_clear
    ctx = sctx
    nb = 8
    iv = bytes(range(16))
    pt = bytes(np.random.default_rng(71).integers(0, 256, 16 * nb, dtype=np.uint8))
    ct = aes_clear.ctr_crypt(aes_key, iv, pt)
    ctx.upload_fwd_trans_key(*keyset.gen_forward_transciphering_keys(aes_key, 55))
    counters = b"".join(((int.from_bytes(iv, "big") + b) % (1 << 128)).to_bytes(16, "big") for b in range(nb))
    d_ctr = torch.frombuffer(bytearray(counters), dtype=torch.uint8).cuda()
    d_ct = torch.frombuffer(bytearray(ct), dtype=torch.uint8).cuda()
    d_out = torch.empty((nb, 128, 2049), dtype=torch.int64, device="cuda")
    m, ip = _out(), _out()
    ctx.ctr_transcipher_dev(d_ctr.data_ptr(), d_ct.data_ptr(), nb, d_out.data_ptr())
    ctx.max_u16_dev(d_out.data_ptr(), 8 * nb, m.data_ptr())
    ctx.inner_product_u16_dev(d_out.data_ptr(), d_out.data_ptr() + 4 * nb * V * 8, 4 * nb, ip.data_ptr())
    vals = _decrypt(_host(d_out), keyset)
    assert len(vals) == 8 * nb
    assert _decrypt(_host(m), keyset) == [max(vals)]
    assert _decrypt(_host(ip), keyset) == [_ip(vals)]


def test_repeated_calls_reuse_and_replace_cached_plans(sctx, keyset):
    ctx = sctx
    vals = _rand_vals(64, 81)
    lwe = _dev(_encrypt(keyset, vals, 82))
    first = None
    for npairs in (32, 32, 4, 32):
        d_out = _out()
        # x = the first npairs values, y = the npairs after them
        ctx.inner_product_u16_dev(lwe.data_ptr(), lwe.data_ptr() + npairs * V * 8, npairs, d_out.data_ptr())
        got = _host(d_out)
        assert _decrypt(got, keyset) == [_ip(vals[: 2 * npairs])], npairs
        if npairs == 32:
            first = got if first is None else first
            assert (got == first).all()
    for n in (3, 8, 5):  # the ladder max's pair tables grow once and serve smaller counts
        d_out = _out()
        ctx.max_u16_dev(lwe.data_ptr(), n, d_out.data_ptr())
        assert _decrypt(_host(d_out), keyset) == [max(vals[:n])], n


def test_inner_product_dev_is_asynchronous(sctx, keyset):
    ctx = sctx
    stream = torch.cuda.current_stream()
    vals = _rand_vals(512, 91)
    lwe = _dev(_encrypt(keyset, vals, 92))
    d_out = _out()
    args = (lwe.data_ptr(), lwe.data_ptr() + 256 * V * 8, 256, d_out.data_ptr())
    ctx.inner_product_u16_dev(*args)  # warm: plan, tables and workspaces
    stream.synchronize()
    ctx.inner_product_u16_dev(*args)
    assert stream.query() is False
    assert _decrypt(_host(d_out), keyset) == [_ip(vals)]


def test_dev_argument_errors(sctx, cbs):
    ctx = sctx
    d_in, d_out = torch.zeros((4, 16, 2049), dtype=torch.int64, device="cuda"), _out()
    p, o = d_in.data_ptr(), d_out.data_ptr()
    calls = [lambda: ctx.max_u16_dev(0, 4, o), lambda: ctx.max_u16_dev(p, 4, 0), lambda: ctx.sum_u16_dev(p, 0, o),
             lambda: ctx.max_u16_lut_dev(p, -1, o), lambda: ctx.inner_product_u16_dev(p, p + 2 * V * 8, 0, o),
             lambda: ctx.inner_product_u16_dev(p, 0, 2, o), lambda: ctx.max_u16_dev(p, 4, p + 3 * V * 8 + 8),
             lambda: ctx.sum_u16_dev(p, 4, p), lambda: ctx.inner_product_u16_dev(p, p + 2 * V * 8, 2, p + 3 * V * 8)]
    for call in calls:
        with pytest.raises(cbs.CbsError, match=r"\(code 1\)"):
            call()
    assert torch.cuda.current_stream().query() is True  # nothing was queued


def _two_gpu_worker(rank, world, port, nb, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch
    import torch.distributed as dist
    import aes_clear
    import temp_fhe_transciphering_b200 as cbs
    from temp_fhe_transciphering_b200 import sharding
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    ks = cbs.KeySet.generate(20261018)
    ctx = cbs.Context(ks, rank)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    key, iv = aes_clear.harness_aes_key(None), bytes(range(16))
    pt = bytes(np.random.default_rng(nb).integers(0, 256, 16 * nb, dtype=np.uint8))
    ct = aes_clear.ctr_crypt(key, iv, pt)
    ctx.upload_fwd_trans_key(*ks.gen_forward_transciphering_keys(key, 4242))
    b0, b1 = sharding.block_range(nb, rank, world)
    counters = b"".join(((int.from_bytes(iv, "big") + b) % (1 << 128)).to_bytes(16, "big") for b in range(b0, b1))
    d_ctr = torch.frombuffer(bytearray(counters), dtype=torch.uint8).cuda()
    d_ct = torch.frombuffer(bytearray(ct[16 * b0:16 * b1]), dtype=torch.uint8).cuda()
    local = torch.empty((b1 - b0, 128, 2049), dtype=torch.int64, device="cuda")
    ctx.ctr_transcipher_dev(d_ctr.data_ptr(), d_ct.data_ptr(), b1 - b0, local.data_ptr())
    res_max = sharding.max_u16_sharded_dev(ctx, local, nb, rank, world, dist)
    res_ip = sharding.inner_product_u16_sharded_dev(ctx, local, nb, rank, world, dist)
    stream.synchronize()
    q.put(("vals", rank, _decrypt(_host(local), ks)))
    if rank == 0:
        q.put(("res", _decrypt(_host(res_max), ks), _decrypt(_host(res_ip), ks)))
    else:
        assert res_max is None and res_ip is None
    dist.barrier()
    ctx.close()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_sharded_max_and_inner_product():
    import torch.multiprocessing as mp
    mpc = mp.get_context("spawn")
    q = mpc.Queue()
    procs = [mpc.Process(target=_two_gpu_worker, args=(r, 2, 29841, 16, q)) for r in range(2)]
    for p in procs:
        p.start()
    msgs = [q.get(timeout=600) for _ in range(3)]
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    vals = dict((m[1], m[2]) for m in msgs if m[0] == "vals")
    allv = vals[0] + vals[1]
    assert len(allv) == 128
    (res,) = [m for m in msgs if m[0] == "res"]
    assert res[1] == [max(allv)] and res[2] == [_ip(allv)]
