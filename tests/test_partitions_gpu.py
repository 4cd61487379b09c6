"""How work is split must not change what is computed.

* Transciphering runs blocks in chunks of CBS_CHUNK_BLOCKS (64), each chunk as CBS_LANES (2) block-aligned parts on side
  streams; a one-block chunk runs on the context stream with the workspaces stage 8 also uses.  With the blind-rotation
  kernel pinned (CBS_BR_LOWLAT=0, read once per process, so in a worker process), every block must come out bit-identical
  under every split, equal to the block transciphered alone, and decrypt to its plaintext.
* The stage-8 LUT circuits run each layer in sub-batches of at most CBS_PLAN_CAP (8192) circuit bootstraps; a bit used in
  two sub-batches is bootstrapped twice.  With the team kernel pinned (CBS_BR_LOWLAT=2) every cap gives the same bits.
* Stage 8 at its edge counts (1, 2, 3, 8 and 9 values, where the maximum switches from the CMux ladder to the LUT circuit)
  and edge values, through the host-buffer and the device-resident calls, which must agree bit for bit."""
import hashlib
import os
import sys
import traceback

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

SPLITS = [(64, 2), (3, 2), (1, 1), (2, 3), (4, 4), (5, 2)]  # (CBS_CHUNK_BLOCKS, CBS_LANES)
NB = 7
IV = bytes([0xFF] * 15 + [0xFC])  # the counter carries through all 128 bits between blocks 3 and 4


def _digests(out):
    out = np.ascontiguousarray(out, dtype=np.uint64).reshape(-1, 128 * 2049)
    return [hashlib.sha256(b.tobytes()).hexdigest() for b in out]


def _counters(iv, nb):
    return b"".join(((int.from_bytes(iv, "big") + b) % (1 << 128)).to_bytes(16, "big") for b in range(nb))


def _summary(out, ks):
    """per-block digests, decrypted bytes and output noise (log2 std, log2 max) of a transcipher output."""
    import ref_io
    bits, std, mx = ref_io.noise_stats(np.asarray(out).reshape(-1, 2049), ks.glwe_sk)
    return {"digests": _digests(out), "bytes": np.packbits(bits).tobytes(), "std": std, "max": mx}


def _setup_worker(mode):
    os.environ["CBS_BR_LOWLAT"] = str(mode)
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))


def _transcipher_worker(q):
    try:
        _setup_worker(0)
        import torch
        import aes_clear
        import temp_fhe_transciphering_b200 as cbs
        ks = cbs.KeySet.generate(20261018)
        key = aes_clear.harness_aes_key(None)
        tk = ks.gen_transciphering_keys(key, 99)
        kf = ks.gen_forward_transciphering_keys(key, 55)
        pt = bytes(np.random.default_rng(7).integers(0, 256, 16 * 65, dtype=np.uint8))
        res = {"pt": pt}

        def context(chunk, lanes):
            os.environ["CBS_CHUNK_BLOCKS"], os.environ["CBS_LANES"] = str(chunk), str(lanes)
            return cbs.Context(ks, 0)

        p7 = pt[:16 * NB]
        ecb, ctr = aes_clear.ecb_encrypt(key, p7), aes_clear.ctr_crypt(key, IV, p7)
        for split in SPLITS:
            c = context(*split)
            res["ecb", split] = _summary(c.aes_to_lwe_transciphering(ecb, *tk), ks)
            res["ctr", split] = _summary(c.aes_ctr_to_lwe_transciphering(ctr, IV, *kf), ks)
            c.upload_fwd_trans_key(*kf)
            d_ctr = torch.frombuffer(bytearray(_counters(IV, NB)), dtype=torch.uint8).cuda()
            d_ct = torch.frombuffer(bytearray(ctr), dtype=torch.uint8).cuda()
            d_out = torch.zeros((NB, 128, 2049), dtype=torch.int64, device="cuda")
            torch.cuda.synchronize()
            c.ctr_transcipher_dev(d_ctr.data_ptr(), d_ct.data_ptr(), NB, d_out.data_ptr())
            c.synchronize()
            res["ctr_dev", split] = _summary(d_out.cpu().numpy().view(np.uint64), ks)
            if split == SPLITS[0]:
                for b in range(NB):
                    blk = slice(16 * b, 16 * b + 16)
                    res["ecb", "alone", b] = _summary(c.aes_to_lwe_transciphering(ecb[blk], *tk), ks)
                    res["ctr", "alone", b] = _summary(
                        c.aes_ctr_to_lwe_transciphering(ctr[blk], _counters(IV, b + 1)[-16:], *kf), ks)
            c.close()
        ecb, ctr = aes_clear.ecb_encrypt(key, pt), aes_clear.ctr_crypt(key, IV, pt)
        for split in ((64, 2), (65, 2)):
            c = context(*split)
            res["ecb65", split] = _summary(c.aes_to_lwe_transciphering(ecb, *tk), ks)
            res["ctr65", split] = _summary(c.aes_ctr_to_lwe_transciphering(ctr, IV, *kf), ks)
            c.close()
        q.put(("ok", res))
    except BaseException:
        q.put(("error", traceback.format_exc()))
        raise


def _vals(n, seed):
    return np.random.default_rng(seed).integers(0, 65536, n).tolist()


def _encrypt(ks, vals, seed):
    bits = np.array([(v >> (15 - i)) & 1 for v in vals for i in range(16)], dtype=np.uint8)
    return ks.encrypt_bits_big(bits, seed)


def _decrypt(ct, ks):
    import ref_io
    return ref_io.bits_to_u16(ref_io.decode_bit(ref_io.lwe_phase(np.asarray(ct).reshape(-1, 2049), ks.glwe_sk)))


def _ip(vals):
    h = len(vals) // 2
    return sum((x * y) % 65536 for x, y in zip(vals[:h], vals[h:])) % 65536


def _dev_call(ctx, fn, *arrays, count):
    """fn(*device pointers, count, d_out) on device copies of `arrays`, with the context's stream ordered after the
    copies and synchronised before the result is read."""
    import torch
    ins = [torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda() for a in arrays]
    d_out = torch.zeros((16, 2049), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    fn(*[t.data_ptr() for t in ins], count, d_out.data_ptr())
    ctx.synchronize()
    return d_out.cpu().numpy().view(np.uint64)


def _plan_cap_worker(q):
    try:
        _setup_worker(2)
        import temp_fhe_transciphering_b200 as cbs
        ks = cbs.KeySet.generate(20261018)
        v20, v33 = _vals(20, 901), _vals(33, 902)
        l20, l33 = _encrypt(ks, v20, 903), _encrypt(ks, v33, 904)
        res = {"v20": v20, "v33": v33}
        for cap in (8192, 64, 16):
            os.environ["CBS_PLAN_CAP"] = str(cap)
            c = cbs.Context(ks, 0)
            outs = {"ip": c.inner_product_u16(l20), "sum": c.sum_u16(l33), "max_lut": c.max_u16_lut(l33),
                    "ip_dev": _dev_call(c, c.inner_product_u16_dev, l20[:10 * 16], l20[10 * 16:], count=10),
                    "sum_dev": _dev_call(c, c.sum_u16_dev, l33, count=33),
                    "max_lut_dev": _dev_call(c, c.max_u16_lut_dev, l33, count=33)}
            for k, o in outs.items():
                res[cap, k] = (hashlib.sha256(o.tobytes()).hexdigest(), _decrypt(o, ks))
            c.close()
        q.put(("ok", res))
    except BaseException:
        q.put(("error", traceback.format_exc()))
        raise


def _run_worker(target, timeout=1200):
    """target(queue) in a spawned process -> its payload; the process is joined, or killed if it does not answer."""
    import torch.multiprocessing as mp
    mpc = mp.get_context("spawn")
    q = mpc.Queue()
    p = mpc.Process(target=target, args=(q,))
    p.start()
    try:
        status, payload = q.get(timeout=timeout)
        p.join(120)
    finally:
        if p.is_alive():
            p.kill()
            p.join()
    assert status == "ok", payload
    assert p.exitcode == 0, p.exitcode
    return payload


@pytest.fixture(scope="module")
def splits():
    return _run_worker(_transcipher_worker)


@pytest.mark.parametrize("mode", ["ecb", "ctr", "ctr_dev"])
def test_transcipher_bit_identical_across_chunk_and_lane_splits(splits, mode):
    """7 blocks as one chunk of two uneven lanes (3 + 4); chunks of 3 + 3 + 1 (1 + 2 lanes, the last chunk on the un-laned
    path); one block per chunk; chunks of 2 with three lanes (more lanes than blocks); chunks of 4 + 3 over four lanes; chunks
    of 5 + 2, whose partial last chunk runs on the same two lanes as the full one with fewer blocks per lane."""
    pt = splits["pt"][:16 * NB]
    base = splits[mode, SPLITS[0]]
    alone = [splits[mode[:3], "alone", b]["digests"][0] for b in range(NB)]
    for split in SPLITS:
        r = splits[mode, split]
        assert r["bytes"] == pt, (split, r["bytes"].hex(), pt.hex())
        bad = [b for b in range(NB) if r["digests"][b] != base["digests"][b]]
        assert not bad, f"{mode} {split}: blocks {bad} differ from the (64, 2) run"
    bad = [b for b in range(NB) if base["digests"][b] != alone[b]]
    assert not bad, f"{mode}: blocks {bad} differ from the same block transciphered alone"
    for b in range(NB):
        assert splits[mode[:3], "alone", b]["bytes"] == pt[16 * b:16 * b + 16], b


@pytest.mark.parametrize("mode", ["ecb65", "ctr65"])
def test_transcipher_65_blocks_one_or_two_chunks(splits, mode):
    """64 + 1 blocks (the one-block chunk on the context stream) against one chunk of 65 blocks, v4 kernel pinned."""
    a, b = splits[mode, (64, 2)], splits[mode, (65, 2)]
    assert a["bytes"] == b["bytes"] == splits["pt"]
    bad = [k for k in range(65) if a["digests"][k] != b["digests"][k]]
    assert not bad, f"blocks {bad} differ"


@pytest.mark.parametrize("mode", ["ecb", "ctr"])
def test_transcipher_65_blocks_default_kernels(keyset, aes_key, trans_key, monkeypatch, mode):
    """The same two splits in the default blind-rotation mode, where the one-block chunk's 128 ciphertexts take the team
    kernel: equal decryption and the output-noise bounds of the other transcipher tests."""
    import aes_clear
    import temp_fhe_transciphering_b200 as cbs
    pt = bytes(np.random.default_rng(7).integers(0, 256, 16 * 65, dtype=np.uint8))
    kf = keyset.gen_forward_transciphering_keys(aes_key, 55)
    got = {}
    for chunk in (64, 65):
        monkeypatch.setenv("CBS_CHUNK_BLOCKS", str(chunk))
        c = cbs.Context(keyset, 0)
        try:
            if mode == "ecb":
                out = c.aes_to_lwe_transciphering(aes_clear.ecb_encrypt(aes_key, pt), *trans_key)
            else:
                out = c.aes_ctr_to_lwe_transciphering(aes_clear.ctr_crypt(aes_key, IV, pt), IV, *kf)
        finally:
            c.close()
        got[chunk] = _summary(out, keyset)
    for chunk, r in got.items():
        assert r["bytes"] == pt, chunk
        assert r["std"] < 58.5 and r["max"] < 61.0, (chunk, r["std"], r["max"])


@pytest.fixture(scope="module")
def plan_caps():
    return _run_worker(_plan_cap_worker)


@pytest.mark.parametrize("name", ["ip", "sum", "max_lut"])
def test_lut_circuit_sub_batches_bit_identical(plan_caps, name):
    """Caps of 8192 (one sub-batch per layer), 64 and 16 circuit bootstraps, host and device calls."""
    v20, v33 = plan_caps["v20"], plan_caps["v33"]
    want = {"ip": _ip(v20), "sum": sum(v33) % 65536, "max_lut": max(v33)}[name]
    ref = plan_caps[8192, name][0]
    for cap in (8192, 64, 16):
        for k in (name, name + "_dev"):
            digest, dec = plan_caps[cap, k]
            assert dec == [want], (cap, k, dec, want)
            assert digest == ref, f"{k} with a cap of {cap} differs from the host call with one sub-batch per layer"


# ---- stage 8 at its edge counts, in this process --------------------------------------------------------------------

def _patterns(n, seed):
    rng = np.random.default_rng(seed)
    lo = rng.integers(0, 60000, n).tolist()
    top = max(lo) + 1
    tied, last_bit = list(lo), list(lo)
    if n >= 2:
        tied[0] = tied[n - 1] = top          # the maximum twice, at both ends
        last_bit[n // 2], last_bit[n - 1] = top, top ^ 1  # a runner-up that differs in the last bit only
    return {"equal": [12345] * n, "zeros": [0] * n, "ones": [65535] * n, "tied": tied, "last_bit": last_bit}


@pytest.mark.parametrize("n", [1, 2, 3, 8, 9])
def test_max_edge_counts_and_values(ctx, keyset, monkeypatch, n):
    monkeypatch.delenv("CBS_MAX_VARIANT", raising=False)
    for k, (pattern, vals) in enumerate(_patterns(n, 700 + n).items()):
        lwe = _encrypt(keyset, vals, 710 + 10 * n + k)
        variants = [None, "ladder", "lut"] if n == 9 else [None]
        for variant in variants:
            if variant:
                monkeypatch.setenv("CBS_MAX_VARIANT", variant)
            calls = [(ctx.max_u16, ctx.max_u16_dev)] + ([(ctx.max_u16_lut, ctx.max_u16_lut_dev)] if not variant else [])
            for fn, dev in calls:
                host = fn(lwe)
                assert np.array_equal(_dev_call(ctx, dev, lwe, count=n), host), (n, pattern, variant, fn.__name__)
                assert _decrypt(host, keyset) == [max(vals)], (n, pattern, variant, fn.__name__)
                if n == 1 and fn == ctx.max_u16:
                    assert np.array_equal(host, lwe)  # the maximum of one value is that value
            monkeypatch.delenv("CBS_MAX_VARIANT", raising=False)


def test_sum_edge_counts(ctx, keyset):
    for k, vals in enumerate(([0], [65535], [40000, 30000], [65535, 65535], [1, 65535], [0, 0])):
        lwe = _encrypt(keyset, vals, 800 + k)
        host = ctx.sum_u16(lwe)
        assert np.array_equal(_dev_call(ctx, ctx.sum_u16_dev, lwe, count=len(vals)), host), vals
        assert _decrypt(host, keyset) == [sum(vals) % 65536], vals


def test_inner_product_dev_edge_pair_counts(ctx, keyset):
    for k, (x, y) in enumerate((([65535], [65535]), ([0], [41234]), ([65535, 0, 12345], [65535, 777, 54321]),
                                ([3, 0, 65535], [0, 9, 2]))):
        lwe = _encrypt(keyset, x + y, 850 + k)
        host = ctx.inner_product_u16(lwe)
        dev = _dev_call(ctx, ctx.inner_product_u16_dev, lwe[:16 * len(x)], lwe[16 * len(x):], count=len(x))
        assert np.array_equal(dev, host), (x, y)
        assert _decrypt(host, keyset) == [_ip(x + y)], (x, y)
