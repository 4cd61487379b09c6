"""The exact integer reference (tests/exact_ref.py) against big-int arithmetic, and the oracle against the reference.

With small keys every FP64 product the FFT evaluates is an integer far below 2^53, so the FP64 path of the oracle must
equal the exact reference bit for bit.  The key bounds (worst case |sum| = max digit x max key word x number of terms,
which must stay far below 2^52 so that the FFT round-off, about 2^-44 of it, leaves every output within 1/8 of its
integer):
  * bootstrap key |k| <= 2^8:     2^22 (B = 2^23 digits) x 2^8 x 3 rows x 1024        < 2^41.6
  * scheme-switch key |k| <= 2^16: 2^16 (B = 2^17)        x 2^16 x 2 levels x 3 x 1024 < 2^44.6
  * LWE keyswitch key |k| <= 2^30: 2^3 (B = 2^4)          x 2^30 x 8 x 3 levels x 256  < 2^45.6
  * automorphism key 0 <= k < 2^20: 2^12 (B = 2^13)       x 2^20 x 2 x 3 levels x 1024 < 2^44.6
    The automorphism key is converted split at bit 41 (lo = the UNSIGNED low 41 bits, hi = the rest), so its words must
    be non-negative: a negative word has a lo limb near 2^41 and nothing is exact.
  * LUT-ladder GGSW |g| <= 2^24:  2 (B = 2^2)             x 2^24 x 7 levels x 3 x 1024 < 2^39.4
With the real seeded keys the oracle's distance to the exact reference is the FP64 error of the algorithm itself; the
GPU budgets in tests/test_exact_gpu.py are set against it."""
import ctypes

import numpy as np
import pytest

import exact_ref as ex
from conftest import log2max, sdiff

N = 1024
EDGE = [0, 1, (1 << 63) - 1, 1 << 63, (1 << 64) - 1]


def tie_words(base_log, level):
    """words at the rounding tie of the closest representable value and at the balanced-digit ties of every level"""
    nr = 64 - base_log * level
    half = 1 << (nr - 1)
    out = [half, half - 1, (1 << 64) - half, (1 << 64) - half - 1]
    for t in range(level):
        b = 1 << (nr + base_log * t + base_log - 1)  # raw digit B/2 at level t
        for nxt in (0, 1 << min(63, nr + base_log * (t + 1) + base_log - 1)):
            for w in (b, b + half, b - half, b + half - 1):
                out.append((w + nxt) % (1 << 64))
    return out


# ---- the reference against big ints --------------------------------------------------------------------------------

def schoolbook(a, d):
    n = len(a)
    out = [0] * n
    for i, di in enumerate(d):
        if di == 0:
            continue
        for j, aj in enumerate(a):
            k = i + j
            if k < n:
                out[k] += di * aj
            else:
                out[k - n] -= di * aj
    return [v % (1 << 64) for v in out]


@pytest.mark.parametrize("n", [8, 256, 1024])
def test_negacyclic_mul_matches_bigint(n):
    rng = np.random.default_rng(n)
    for trial in range(3):
        a = rng.integers(0, 2 ** 64, n, dtype=np.uint64)
        a[: len(EDGE)] = EDGE
        if trial == 0:
            d = rng.integers(-(1 << 22), (1 << 22) + 1, n)
        elif trial == 1:
            d = rng.integers(0, 2 ** 64, n, dtype=np.uint64).view(np.int64)  # full 64-bit both sides
        else:
            d = np.zeros(n, dtype=np.int64)
            d[[0, n - 1]] = [-1, (1 << 62)]
        got = ex.negacyclic_mul(a, d.astype(np.int64))
        assert got.tolist() == schoolbook([int(x) for x in a], [int(x) for x in d])


@pytest.mark.parametrize("base_log,level", [(23, 1), (13, 3), (17, 2), (2, 7), (4, 3)])
def test_decompose_matches_definition_and_oracle(orc, base_log, level):
    rng = np.random.default_rng(base_log)
    words = EDGE + tie_words(base_log, level) + rng.integers(0, 2 ** 64, 2000, dtype=np.uint64).tolist()
    x = np.array(words, dtype=np.uint64)
    got = ex.decompose(x, base_log, level)
    want = np.array([ex.decompose_bigint(int(w), base_log, level) for w in words]).T
    assert (got == want).all()
    assert np.abs(got).max() <= 1 << (base_log - 1)
    # digits reconstruct the closest representable value mod 2^64
    nr = 64 - base_log * level
    for w, col in zip(words[:200], got.T[:200]):
        rec = sum(int(col[t]) << (nr + base_log * t) for t in range(level)) % (1 << 64)
        assert rec == ((w + (1 << (nr - 1))) >> nr << nr) % (1 << 64)
    # the oracle's decomposer (tfhe's carry form) on the same words
    n = len(words)
    dig = np.zeros((level, n), dtype=np.int64)
    orc.lib().orc_decompose(dig.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                            x.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), n, base_log, level)
    assert (dig == got).all()


def test_building_blocks_match_oracle(orc):
    L = orc.lib()
    u = ctypes.POINTER(ctypes.c_uint64)
    rng = np.random.default_rng(7)
    p = rng.integers(0, 2 ** 64, N, dtype=np.uint64)
    q = np.zeros(N, dtype=np.uint64)
    for d in (0, 1, 8, 511, 1023, 1024, 1025, 2040, 2047, 2048):
        L.orc_mono_mul(q.ctypes.data_as(u), p.ctypes.data_as(u), N, d)
        assert (ex.mono_mul(p, d) == q).all(), d
    for i in range(1, 11):
        kappa = N // (1 << (i - 1)) + 1
        L.orc_eval_x_k(q.ctypes.data_as(u), p.ctypes.data_as(u), N, kappa)
        assert (ex.eval_x_k(p, kappa) == q).all(), kappa
    g = rng.integers(0, 2 ** 64, 3 * N, dtype=np.uint64)
    lwe = np.zeros(2 * N + 1, dtype=np.uint64)
    for t in (0, 1, 256, 768, 1023):
        L.orc_sample_extract(lwe.ctypes.data_as(u), g.ctypes.data_as(u), 2, N, t)
        assert (ex.sample_extract(g, 2, N, t) == lwe).all(), t
    small = rng.integers(0, 2 ** 64, 8 * 256 + 1, dtype=np.uint64)
    emb = np.zeros(9 * 256, dtype=np.uint64)
    L.orc_const_embed(emb.ctypes.data_as(u), small.ctypes.data_as(u), 8, 256)
    assert (ex.const_embed(small, 8, 256) == emb).all()
    assert (ex.sample_extract(emb, 8, 256, 0) == small).all()
    # modulus switch: every rounding boundary of the 2^56 grid, both sides
    for w in EDGE + [k << 56 for k in range(256)] + [(k << 56) + (1 << 55) + s for k in range(256) for s in (-1, 0)]:
        w %= 1 << 64
        assert ex.modswitch(w) == orc.modswitch(w), hex(w)
        assert ex.modswitch(w) % 8 == 0 and 0 <= ex.modswitch(w) <= 2048
    # accumulator build against the oracle's blind rotation with an all-zero mask (no step runs)
    keys = orc.Keys(np.zeros(768 * 9 * N, np.uint64), np.zeros(8 * 3 * 4 * 256, np.uint64),
                    np.zeros(10 * 2 * 3 * 3 * N, np.uint64), np.zeros(2 * 2 * 3 * 3 * N, np.uint64))
    for b in (0, 1 << 55, (1 << 56) * 37, 1 << 63, (1 << 64) - 1):
        lwe = np.zeros(769, dtype=np.uint64)
        lwe[768] = b
        assert (ex.br_accumulator(b).reshape(-1) == orc.blind_rotate(keys, lwe)[0]).all()


# ---- small keys: the oracle's FP64 path is exact ------------------------------------------------------------------

def small_keys(seed=2026):
    rng = np.random.default_rng(seed)

    def signed(bound, shape):
        return rng.integers(-bound, bound + 1, shape).astype(np.int64).view(np.uint64)

    bsk = signed(1 << 8, (768, 1, 3, 3, N))
    ksk = signed(1 << 30, (8, 3, 4, 256))
    auto = rng.integers(0, 1 << 20, (10, 2, 3, 3, N), dtype=np.uint64)
    ss = signed(1 << 16, (2, 2, 3, 3, N))
    return bsk, ksk, auto, ss


def small_ggsw(rng, count, bound=1 << 24):
    return rng.integers(-bound, bound + 1, (count, 7 * 3 * 3 * N)).astype(np.int64).view(np.uint64)


@pytest.fixture(scope="module")
def small(orc):
    k = small_keys()
    return k, orc.Keys(*k)


def br_inputs(rng):
    """single mask words at both sides of modulus-switch boundaries (including the 2048 -> identity wrap), plus one full
    random LWE"""
    rows = []
    for i, w in enumerate([1 << 55, (1 << 55) - 1, (5 << 56) + (1 << 55), (5 << 56) + (1 << 55) - 1, 1 << 63,
                           (1 << 64) - (1 << 55), (1 << 64) - (1 << 55) - 1, (1 << 64) - 1]):
        lwe = np.zeros(769, dtype=np.uint64)
        lwe[(97 * i + 3) % 768] = w
        lwe[768] = rng.integers(0, 2 ** 64, dtype=np.uint64)
        rows.append(lwe)
    rows.append(rng.integers(0, 2 ** 64, 769, dtype=np.uint64))
    return np.stack(rows)


def test_small_keys_blind_rotation_exact(small, orc):
    (bsk, ksk, auto, ss), K = small
    lwe = br_inputs(np.random.default_rng(1))
    got = orc.blind_rotate(K, lwe)
    for i in range(len(lwe)):
        assert (ex.blind_rotate(bsk, lwe[i]) == got[i]).all(), i


def test_small_keys_lwe_keyswitch_exact(small, orc):
    (bsk, ksk, auto, ss), K = small
    rng = np.random.default_rng(2)
    lwe = rng.integers(0, 2 ** 64, (6, 2049), dtype=np.uint64)
    lwe[0] = 0
    lwe[1, :len(EDGE) * 100] = np.repeat(np.array(EDGE, dtype=np.uint64), 100)
    lwe[2, : 2048] = np.resize(np.array(tie_words(4, 3), dtype=np.uint64), 2048)
    got = orc.lwe_keyswitch(K, lwe)
    for i in range(len(lwe)):
        assert (ex.lwe_keyswitch(ksk, lwe[i]) == got[i]).all(), i


def test_small_keys_trace_and_auto_steps_exact(small, orc):
    (bsk, ksk, auto, ss), K = small
    rng = np.random.default_rng(3)
    g = rng.integers(0, 2 ** 64, 3 * N, dtype=np.uint64)
    g[:1000] = np.resize(np.array(tie_words(13, 3), dtype=np.uint64), 1000)
    for i in range(1, 11):
        assert (ex.auto_step(auto, i, g) == orc.auto_step(K, i, g)).all(), i
    assert (ex.trace(auto, g) == orc.trace(K, g)[0]).all()


def test_small_keys_scheme_switch_exact(small, orc):
    (bsk, ksk, auto, ss), K = small
    rng = np.random.default_rng(4)
    glev = rng.integers(0, 2 ** 64, (7, 3 * N), dtype=np.uint64)
    glev[0, :2000] = np.resize(np.array(tie_words(17, 2), dtype=np.uint64), 2000)
    assert (ex.scheme_switch(ss, glev) == orc.scheme_switch(K, glev)[0]).all()


def test_small_keys_lut_ladder_exact(orc):
    rng = np.random.default_rng(5)
    ggsw = small_ggsw(rng, 8)
    lut = rng.integers(0, 2 ** 64, (2, 3 * N), dtype=np.uint64)
    lut[0, :2048] = 0  # trivial accumulator next to a non-trivial one
    lut[0, 2048:2048 + 500] = np.resize(np.array(tie_words(2, 7), dtype=np.uint64), 500)
    got = orc.lut8_eval(orc.ggsw_to_fourier(ggsw), lut)
    assert (ex.lut8_eval(ggsw, lut) == got).all()


def test_small_keys_circuit_bootstrap_exact(small, orc):
    (bsk, ksk, auto, ss), K = small
    lwe = np.random.default_rng(6).integers(0, 2 ** 64, (1, 769), dtype=np.uint64)
    want = ex.circuit_bootstrap((bsk, auto, ss), lwe[0], orc.glev_from_acc)
    assert (orc.circuit_bootstrap(K, lwe)[0] == want).all()


# ---- real keys: the oracle's own FP64 error ------------------------------------------------------------------------

def oracle_br_step(orc, bsk_i, acc, a_i):
    """one blind-rotation CMux of the oracle (its FP64 external product) on a given accumulator"""
    L = orc.lib()
    u, dp = ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_double)
    f = np.zeros(9 * N)
    b = np.ascontiguousarray(bsk_i, dtype=np.uint64).reshape(-1)
    L.orc_ggsw_to_fourier(f.ctypes.data_as(dp), b.ctypes.data_as(u), 2, N, 1)
    out = np.array(acc, dtype=np.uint64).reshape(3, N)
    with np.errstate(over="ignore"):
        ct1 = np.ascontiguousarray(ex.mono_mul(out, ex.modswitch(a_i) % (2 * N)) - out)
    L.orc_external_product_add(out.ctypes.data_as(u), f.ctypes.data_as(dp), ct1.ctypes.data_as(u), 2, N, 23, 1)
    return out


def test_real_keys_oracle_error_of_each_external_product(orc, orc_keys, keyset):
    """log2 max |oracle - exact| per kind of external product with the seeded keys (KeySet.generate(20261018)).
    Measured on x86-64 (gcc -O3 -mfma), seeds 8 / 9 / 10 of the inputs: blind-rotation step on uniform accumulators
    40.43 (median 40.00 over 40 steps, seed 8), 8-CMux LUT ladder 21.75 / 21.85 / 21.91 (B = 2^2 digits are tiny), scheme switch 35.05 / 34.92 / 34.73, LWE keyswitch
    21.32 / 21.28 / 21.03, automorphism step 8.55 / 7.95 / 8.13 (the split key multiplies 41- and 23-bit limbs).  These
    numbers sit next to the GPU budgets of tests/test_exact_gpu.py."""
    rng = np.random.default_rng(8)
    err = {}
    # after a few steps an accumulator is uniform: 40 steps on uniform accumulators
    e = []
    for i in range(40):
        acc = rng.integers(0, 2 ** 64, (3, N), dtype=np.uint64)
        a = rng.integers(0, 2 ** 64, dtype=np.uint64)
        e.append(log2max(sdiff(oracle_br_step(orc, keyset.bsk[i], acc, a), ex.br_step(acc, keyset.bsk[i], a))))
    err["br_step"] = max(e)
    ggsw = rng.integers(0, 2 ** 64, (8, 7 * 9 * N), dtype=np.uint64)
    lut = rng.integers(0, 2 ** 64, (2, 3 * N), dtype=np.uint64)
    got = orc.lut8_eval(orc.ggsw_to_fourier(ggsw), lut)
    want = ex.lut8_eval(ggsw, lut)
    err["lut_ladder"] = log2max(sdiff(got, want))
    glev = rng.integers(0, 2 ** 64, (7, 3 * N), dtype=np.uint64)
    err["scheme_switch"] = log2max(sdiff(orc.scheme_switch(orc_keys, glev)[0], ex.scheme_switch(keyset.ss, glev)))
    big = rng.integers(0, 2 ** 64, (1, 2049), dtype=np.uint64)
    err["lwe_keyswitch"] = log2max(sdiff(orc.lwe_keyswitch(orc_keys, big)[0], ex.lwe_keyswitch(keyset.ksk, big[0])))
    g = rng.integers(0, 2 ** 64, 3 * N, dtype=np.uint64)
    err["auto_step"] = log2max(sdiff(orc.auto_step(orc_keys, 3, g), ex.auto_step(keyset.auto_std, 3, g)))
    print({k: round(v, 1) for k, v in err.items()})
    limits = {"br_step": 41, "lut_ladder": 23, "scheme_switch": 36, "lwe_keyswitch": 22.5, "auto_step": 10}
    for k, v in err.items():
        assert v < limits[k], (k, v)
