"""The bootstrapping stages at the batch sizes they run at.

Every kernel on the bootstrap path computes each ciphertext on its own, so an output must not depend on the batch size
or on where the ciphertext sits in the batch: the same input gives the same bits alone, in a batch of 2 or 3, in any slot
of a many-wave launch and in the partial last CTA.  That check needs no oracle and is exact at any size; with the oracle
parity of tests/test_gpu_parity.py at small sizes it ties every large launch to the oracle.  On top of it each stage is
compared with the oracle at about 16 positions of its largest batch, and every output of that batch is decrypted with the
secret key against a bound on its WORST error, so that one corrupted ciphertext cannot hide behind a good mean.

Sentinel inputs go where kernels go wrong: first and last position, around every wave boundary (multiples of the SM
count times the items one CTA holds, which also covers kernels with several resident CTAs per SM) and the whole last CTA
with the item before it.  The largest batch is also run again without its first item, which moves every item to another
slot of its CTA and of the grid.

The blind rotation runs k_blind_rotate_ll (the team kernel) for small batches and small tails and k_blind_rotate_v4
otherwise.  CBS_BR_LOWLAT (read once per process) forces either, so those checks run in worker processes, one per mode.
On a B200 the two kernels give bit-identical accumulators (test_team_and_v4_kernels_agree), so the default mode, where
a batch of 1 to 3 and a batch of 300 take different kernels, is compared bit for bit as well."""
import os
import sys
import traceback

import numpy as np
import pytest

from conftest import ROOT, glwe_phase, log2max, sdiff

N = 1024


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _bits(n, seed):
    return np.random.default_rng(seed).integers(0, 2, n, dtype=np.uint8)


# ---- exact phase of many GLWE at once ------------------------------------------------------------------------------

def _negacyclic(s):
    """M with (a * s mod X^N + 1)[j] = sum_i a[i] M[i, j]; entries 0 / +-1."""
    i, j = np.arange(N)[:, None], np.arange(N)[None, :]
    return s[(j - i) % N].astype(np.float64) * np.where(j >= i, 1.0, -1.0)


def fast_glwe_phase(glwe, glwe_sk):
    """conftest.glwe_phase, exact, as float64 matrix products: the masks are split into 16-bit limbs, so every dot
    product of 1024 terms stays below 2^26 and is exact; the limbs are recombined mod 2^64."""
    g = np.asarray(glwe, dtype=np.uint64).reshape(-1, 3, N)
    s = np.asarray(glwe_sk, dtype=np.uint64).reshape(2, N)
    out = g[:, 2].copy()
    for c in range(2):
        m = _negacyclic(s[c])
        for limb in range(4):
            part = ((g[:, c] >> np.uint64(16 * limb)) & np.uint64(0xFFFF)).astype(np.float64) @ m
            out -= np.rint(part).astype(np.int64).view(np.uint64) << np.uint64(16 * limb)
    return out


def test_fast_glwe_phase_matches_glwe_phase():
    rng = np.random.default_rng(5)
    g = rng.integers(0, 2 ** 64, (3, 3, N), dtype=np.uint64)
    sk = rng.integers(0, 2, 2 * N, dtype=np.uint64)
    assert (fast_glwe_phase(g, sk) == glwe_phase(g, sk)).all()


# ---- sentinel slots and the invariance check -------------------------------------------------------------------------

def slots(n, per_item, per_cta, sms):
    """Positions of an n-item launch that matter, for a kernel with per_item work units per item and per_cta units per
    CTA: first and last, every wave boundary, and the last CTA with the item before it."""
    units = n * per_item
    pos = {0, n - 1}
    last = (units - 1) // per_cta * per_cta // per_item
    pos |= set(range(last - 1, n))
    for w in range(sms * per_cta, units, sms * per_cta):
        pos |= {(w - 1) // per_item, w // per_item}
    return sorted(p for p in pos if 0 <= p < n)


def check_invariance(run, filler, sents, counts, per_item, per_cta):
    """run(batch) -> outputs, one per item.  Sentinels alone, in batches of 2 and 3, and in the slots of filler batches
    of each count must give bit-identical outputs; the largest batch run without its first item must give the same
    outputs as before for the other items.  Returns (batch, out, slot list) of the largest count."""
    sms = _sms()
    alone = [run(s[None])[0] for s in sents]
    pair, trio = run(np.stack(sents[:2])), run(np.stack(sents))
    for k in range(len(sents)):
        assert np.array_equal(trio[k], alone[k]), ("batch of 3", k)
        if k < 2:
            assert np.array_equal(pair[k], alone[k]), ("batch of 2", k)
    big = None
    for n in counts:
        batch = np.array(filler[:n], copy=True)
        where = slots(n, per_item, per_cta, sms)
        for i, p in enumerate(where):
            batch[p] = sents[i % len(sents)]
        out = run(batch)
        for i, p in enumerate(where):
            k = i % len(sents)
            assert np.array_equal(out[p], alone[k]), f"count {n}: sentinel {k} at position {p} differs"
        big = (batch, out, where)
    batch, out, _ = big
    shifted = run(batch[1:])
    bad = [i + 1 for i in range(len(shifted)) if not np.array_equal(shifted[i], out[i + 1])]
    assert not bad, f"{len(bad)} outputs change when their item moves one slot: {bad[:16]}"
    return big


def probe_positions(n, where, k=16):
    """about k positions of an n-item batch: the sentinel slots' extremes and an even spread."""
    pick = set(where[:4]) | set(where[-4:]) | set(np.linspace(0, n - 1, k - 8).astype(int).tolist())
    return sorted(pick)


# ---- stages in this process (default blind-rotation mode) ----------------------------------------------------------

@pytest.mark.gpu
def test_keyswitch_batch_shapes(ctx, orc, orc_keys, keyset):
    import ref_io
    n = 8193
    bits = _bits(n, 101)
    filler = keyset.encrypt_bits_big(bits, 102)
    sbits = np.array([1, 0, 1], dtype=np.uint8)
    sents = list(keyset.encrypt_bits_big(sbits, 103))
    batch, out, where = check_invariance(ctx.keyswitch_lwe_ciphertext_by_glwe_keyswitch, filler, sents, (1, 3, n),
                                         1, 2)
    for p in probe_positions(n, where):
        d = sdiff(out[p], orc.lwe_keyswitch(orc_keys, batch[p][None])[0])
        assert log2max(d) < 30, (p, log2max(d))
    want = bits.copy()
    for i, p in enumerate(where):
        want[p] = sbits[i % 3]
    ph = ref_io.lwe_phase(out, keyset.lwe_sk_small)
    assert (ref_io.decode_bit(ph) == want).all()
    assert log2max(ref_io.bit_error(ph, want)) < 58.5


@pytest.mark.gpu
def test_glev_from_acc_batch_shapes(ctx, orc):
    rng = np.random.default_rng(111)
    filler = rng.integers(0, 2 ** 64, (1000, 3072), dtype=np.uint64)
    sents = list(rng.integers(0, 2 ** 64, (3, 3072), dtype=np.uint64))
    batch, out, _ = check_invariance(ctx.glev_from_acc, filler, sents, (1, 1000), 1, 1)
    assert (out == orc.glev_from_acc(batch)).all()


@pytest.fixture(scope="module")
def glwe_pool(ctx, keyset):
    """~620 trace inputs: the GLEV rows of blind-rotated encryptions of random bits."""
    acc = ctx.blind_rotate(keyset.encrypt_bits_small(_bits(89, 121), 122))
    return ctx.glev_from_acc(acc).reshape(-1, 3072)


@pytest.mark.gpu
def test_trace_batch_shapes(ctx, orc, orc_keys, keyset, glwe_pool):
    sms = _sms()
    counts = (1, 3, 2 * sms - 1, 2 * sms + 1, 600)
    sents = list(glwe_pool[-3:])
    batch, out, where = check_invariance(ctx.trace_assign, glwe_pool[:-3], sents, counts, 1, 2)
    for p in probe_positions(600, where):
        d = sdiff(out[p], orc.trace(orc_keys, batch[p][None])[0])
        assert log2max(d) < 30, (p, log2max(d))
    ph = fast_glwe_phase(out, keyset.glwe_sk).astype(np.int64).astype(np.float64)
    worst = np.log2(np.abs(ph[:, 1:]).max(axis=1) + 1)
    assert worst.max() < 42, (int(worst.argmax()), worst.max())


@pytest.mark.gpu
def test_scheme_switch_batch_shapes(ctx, orc, orc_keys, keyset):
    sms = _sms()
    n = 200
    glev = ctx.lwe_msb_bit_to_glev_by_trace_with_preprocessing(keyset.encrypt_bits_small(_bits(n + 3, 131), 132))
    counts = (1, 3, 4 * sms // 7 + 5, n)
    batch, out, where = check_invariance(ctx.switch_scheme, glev[:n], list(glev[n:]), counts, 7, 4)
    for p in probe_positions(n, where):
        d = sdiff(out[p], orc.scheme_switch(orc_keys, batch[p][None])[0])
        assert log2max(d) < 40, (p, log2max(d))
    # rows k of the GGSW are the GLEV itself
    assert (out.reshape(-1, 7, 3, 3072)[:, :, 2] == batch.reshape(-1, 7, 3072)).all()


def ggsw_worst_row_error(ggsw, bits, glwe_sk):
    """log2 of the worst coefficient error over every row of every level of each GGSW: row r < 2 of level l encrypts
    -b S_r 2^(64-2(l+1)), row 2 encrypts b 2^(64-2(l+1))."""
    g = np.asarray(ggsw, dtype=np.uint64).reshape(-1, 7, 3, 3, N)
    ph = fast_glwe_phase(g.reshape(-1, 3, N), glwe_sk).reshape(-1, 7, 3, N)
    sk = np.asarray(glwe_sk, dtype=np.uint64).reshape(2, N)
    want = np.zeros_like(ph)
    for lvl in range(7):
        sh = np.uint64(64 - 2 * (lvl + 1))
        with np.errstate(over="ignore"):
            for r in range(2):
                want[:, lvl, r] = ((np.uint64(0) - sk[r]) << sh)[None] * bits.astype(np.uint64)[:, None]
            want[:, lvl, 2, 0] = bits.astype(np.uint64) << sh
    return np.log2(np.abs(sdiff(ph, want)).reshape(len(bits), -1).max(axis=1) + 1)


@pytest.mark.gpu
def test_circuit_bootstrap_batch_shapes(ctx, keyset):
    """Default mode: batches of 1 to 3 run the team blind rotation, 300 (more than 2 per SM, less than one v4 wave) run
    v4; with the trace from the accumulator (from_acc) and the scheme switch into the Fourier and standard GGSW."""
    n = 300
    bits = _bits(n, 141)
    filler = keyset.encrypt_bits_small(bits, 142)
    sbits = np.array([1, 0, 1], dtype=np.uint8)
    sents = list(keyset.encrypt_bits_small(sbits, 143))
    run = ctx.circuit_bootstrap_lwe_ciphertext_by_trace_with_preprocessing
    batch, out, where = check_invariance(run, filler, sents, (1, 3, n), 1, 4)
    want = bits.copy()
    for i, p in enumerate(where):
        want[p] = sbits[i % 3]
    worst = ggsw_worst_row_error(out, want, keyset.glwe_sk)
    assert worst.max() < 52.5, (int(worst.argmax()), worst.max())


@pytest.fixture(scope="module")
def byte_pool(ctx, keyset):
    """GGSWs of 16 bytes (bits LSB first per byte, as cbs_lut8_eval takes them) and their values."""
    vals = np.random.default_rng(151).integers(0, 256, 16)
    bits = np.array([(v >> i) & 1 for v in vals for i in range(8)], dtype=np.uint8)
    ggsw = ctx.circuit_bootstrap_lwe_ciphertext_by_trace_with_preprocessing(keyset.encrypt_bits_small(bits, 152))
    return ggsw.reshape(16, 8, -1), vals


@pytest.mark.gpu
@pytest.mark.parametrize("nluts", [4, 3, 1])
def test_lut8_batch_shapes(ctx, orc, keyset, trans_key, aes_key, byte_pool, nluts):
    """accs_per_byte = 2 nluts = 8, 6, 2: 4, 3 and 2 jobs per CTA, the shapes of the inverse and forward middle rounds
    and of the last round."""
    import ref_io
    sms = _sms()
    ggsw, vals = byte_pool
    n = sms // 2 + 6  # past one wave of 2 CTAs per byte for 4 and 3 LUTs
    if nluts == 4:
        tab = trans_key[1].reshape(-1, 4, 16, 2, 3072)  # [round][m][byte]
    elif nluts == 3:
        tab = keyset.gen_forward_transciphering_keys(aes_key, 55)[1].reshape(-1, 3, 16, 2, 3072)
    else:
        tab = trans_key[2].reshape(1, 1, 16, 2, 3072)
    items = [(b % 16, (7 * b) % len(tab), (5 * b + 3) % 16) for b in range(n + 3)]  # (ggsw byte, round, state byte)

    def item(k):
        g, r, s = items[k]
        return np.concatenate([ggsw[g].reshape(-1), tab[r, :, s].reshape(-1)])

    gw = 8 * ggsw.shape[2]

    def run(batch):
        b = np.asarray(batch).reshape(len(batch), -1)
        return ctx.evaluate_8_to_8_cipher_lut(b[:, :gw], b[:, gw:])

    filler = np.stack([item(k) for k in range(n)])
    sents = [item(k) for k in range(n, n + 3)]
    batch, out, where = check_invariance(run, filler, sents, (1, 2, n), 2 * nluts, {8: 4, 6: 3, 2: 2}[2 * nluts])
    b = batch.reshape(n, -1)
    luts = b[:, gw:].reshape(n, nluts, 2, 3072)
    gf = {}
    for p in probe_positions(n, where):
        key = b[p, :gw].tobytes()
        gf.setdefault(key, orc.ggsw_to_fourier(b[p, :gw].reshape(8, -1)))
        for m in range(nluts):
            d = sdiff(out[p, m], orc.lut8_eval(gf[key], luts[p, m]))
            assert log2max(d) < 52, (p, m, log2max(d))
    # every output decrypts to its table entry
    src = list(range(n))
    for i, p in enumerate(where):
        src[p] = n + i % 3
    value = vals[[items[k][0] for k in src]]
    cols = 2048 + 256 * np.arange(4)[None, :] + value[:, None]  # [n][t]
    want = np.stack([(np.take_along_axis(luts[:, :, a], cols[:, None, :].repeat(nluts, 1), axis=2) >> np.uint64(63))
                     for a in range(2)], axis=2).reshape(n, nluts, 8).astype(np.uint8)
    ph = ref_io.lwe_phase(out, keyset.glwe_sk)
    assert (ref_io.decode_bit(ph) == want).all()
    assert log2max(ref_io.bit_error(ph, want)) < 60.5


# ---- blind rotation and circuit bootstrap under a forced kernel (worker processes) -------------------------------------

def _forced_worker(mode, outdir, q):
    try:
        os.environ["CBS_BR_LOWLAT"] = str(mode)
        sys.path.insert(0, ROOT)
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import torch
        import temp_fhe_transciphering_b200 as cbs
        ks = cbs.KeySet.generate(20261018)
        ctx = cbs.Context(ks, 0)
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        for name, run, n, per_cta in (("br", ctx.blind_rotate, 2 * 4 * sms + 3, 4),
                                      ("cbs", ctx.circuit_bootstrap_lwe_ciphertext_by_trace_with_preprocessing, 300, 4)):
            small = ks.encrypt_bits_small(_bits(n + 3, 161), 162)
            sents, filler = small[n:], small[:n]
            outs = {"alone": np.stack([run(s[None])[0] for s in sents]), "trio": run(sents)}
            for count in (3, n):
                batch = filler[:count].copy()
                where = slots(count, 1, per_cta, sms)
                for i, p in enumerate(where):
                    batch[p] = sents[i % 3]
                outs[f"out{count}"] = run(batch)
                outs[f"where{count}"] = np.array(where)
                outs[f"in{count}"] = batch
            outs["shifted"] = run(batch[1:])
            np.savez(os.path.join(outdir, f"{name}.npz"), **outs)
        ctx.close()
        q.put("ok")
    except BaseException:
        q.put(traceback.format_exc())
        raise


def run_worker(target, *args, timeout=900):
    """target(*args, queue) in a spawned process: its message (or traceback), with the process joined or killed."""
    import torch.multiprocessing as mp
    mpc = mp.get_context("spawn")
    q = mpc.Queue()
    p = mpc.Process(target=target, args=(*args, q))
    p.start()
    try:
        msg = q.get(timeout=timeout)
        p.join(120)
    finally:
        if p.is_alive():
            p.kill()
            p.join()
    assert msg == "ok", msg
    assert p.exitcode == 0, p.exitcode
    return msg


@pytest.fixture(scope="module")
def forced(tmp_path_factory):
    """{mode: {"br": npz, "cbs": npz}} for CBS_BR_LOWLAT = 0 (v4 always) and 2 (team kernel always)."""
    res = {}
    for mode in (0, 2):
        d = str(tmp_path_factory.mktemp(f"lowlat{mode}"))
        run_worker(_forced_worker, mode, d)
        res[mode] = {k: dict(np.load(os.path.join(d, f"{k}.npz"))) for k in ("br", "cbs")}
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 2])
@pytest.mark.parametrize("stage", ["br", "cbs"])
def test_forced_kernel_batch_invariance(forced, keyset, mode, stage):
    r = forced[mode][stage]
    big = max(int(k[3:]) for k in r if k.startswith("out"))
    assert np.array_equal(r["trio"], r["alone"])
    for count in (3, big):
        out, where = r[f"out{count}"], r[f"where{count}"]
        for i, p in enumerate(where):
            assert np.array_equal(out[p], r["alone"][i % 3]), (count, int(p))
    bad = np.flatnonzero((r["shifted"] != r[f"out{big}"][1:]).reshape(big - 1, -1).any(axis=1))
    assert bad.size == 0, (bad[:16] + 1).tolist()
    # every output decrypts: accumulator coefficient l holds b 2^(64-2(l+1)) - 2^(63-2(l+1)); GGSW rows as above
    inp = r[f"in{big}"]
    bits = _bits(big + 3, 161)[:big].copy()
    sbits = _bits(big + 3, 161)[big:]
    for i, p in enumerate(r[f"where{big}"]):
        bits[p] = sbits[i % 3]
    assert inp.shape[0] == big
    if stage == "br":
        ph = fast_glwe_phase(r[f"out{big}"], keyset.glwe_sk)
        for lvl in range(7):
            val = ph[:, lvl] + np.uint64(1 << (63 - 2 * (lvl + 1)))
            assert log2max(sdiff(val, bits.astype(np.uint64) << np.uint64(64 - 2 * (lvl + 1)))) < 52
    else:
        worst = ggsw_worst_row_error(r[f"out{big}"], bits, keyset.glwe_sk)
        assert worst.max() < 52.5, (int(worst.argmax()), worst.max())


@pytest.mark.gpu
@pytest.mark.parametrize("stage", ["br", "cbs"])
def test_team_and_v4_kernels_agree(forced, keyset, stage):
    """The same inputs through k_blind_rotate_v4 (mode 0) and the team kernel (mode 2) give the same bits: both run the
    same decomposition and FFT arithmetic per ciphertext, only the thread layout differs."""
    a, b = forced[0][stage], forced[2][stage]
    big = max(int(k[3:]) for k in a if k.startswith("out"))
    assert np.array_equal(a[f"in{big}"], b[f"in{big}"])
    bad = np.flatnonzero((a[f"out{big}"] != b[f"out{big}"]).reshape(big, -1).any(axis=1))
    assert bad.size == 0, f"{bad.size} of {big} outputs differ between the kernels: {bad[:16].tolist()}"
