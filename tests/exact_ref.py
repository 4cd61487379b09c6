"""Exact integer reference of the FP64 external-product stages (test helper, not a conftest).

Every operation is restated in integer arithmetic mod 2^64 with numpy's wrapping uint64: Z/2^64 is a ring, so a product
of two words read as two's complement and summed with wrap-around is the exact product mod 2^64, whatever the size of the
words.  The negacyclic product is one np.convolve of the two coefficient vectors (wrapping uint64 multiply-add, N^2
terms, no floating point) folded by X^N = -1.  No limb splitting is needed and no FFT is involved, so nothing has to be
certified: the reference is exact by construction, for any key.  tests/test_exact_ref_cpu.py checks it against Python
big-int schoolbook arithmetic.

With small keys every FP64 product inside the kernels and the oracle is an exactly representable integer (the bounds
are derived in tests/test_exact_ref_cpu.py), so there both must equal this reference bit for bit.  With real keys the
difference to this reference is the FP64 error of the evaluation.

Layouts follow oracle/cbs_oracle.h: LWE [a_0..a_{n-1}, b], GLWE [k masks][body] of N coefficients, GGSW std
[level (coarsest first)][row][poly][N], decomposition digits [level][...] finest first.
"""
import numpy as np

U64 = np.uint64
N = 1024
LWE_N = 768


def u64(x):
    return np.asarray(x, dtype=np.uint64)


def neg(x):
    return U64(0) - u64(x)


# ---- ring arithmetic ---------------------------------------------------------------------------------------------------

def negacyclic_mul(a, b):
    """a * b mod (X^n + 1) mod 2^64; a, b: [n] words (signed values as two's complement).  Exact."""
    a = np.ascontiguousarray(a, dtype=np.int64).view(np.uint64) if np.asarray(a).dtype == np.int64 else u64(a)
    b = np.ascontiguousarray(b, dtype=np.int64).view(np.uint64) if np.asarray(b).dtype == np.int64 else u64(b)
    n = a.shape[-1]
    with np.errstate(over="ignore"):
        full = np.convolve(a, b)
        out = full[:n].copy()
        out[: n - 1] -= full[n:]
    return out


def mono_mul(p, d):
    """p * X^d mod (X^n + 1), d taken mod 2n; p: [..., n]."""
    p = u64(p)
    n = p.shape[-1]
    d %= 2 * n
    out = np.roll(p, d % n, axis=-1)
    with np.errstate(over="ignore"):
        out[..., : d % n] = neg(out[..., : d % n])
        if d >= n:
            out = neg(out)
    return out


def eval_x_k(p, kappa):
    """p(X^kappa) mod (X^n + 1) for odd kappa; p: [..., n]."""
    p = u64(p)
    n = p.shape[-1]
    e = (np.arange(n) * kappa) % (2 * n)
    out = np.zeros_like(p)
    with np.errstate(over="ignore"):
        out[..., e % n] = np.where(e >= n, neg(p), p)
    return out


def sample_extract(glwe, k, n, t):
    """LWE of coefficient t of GLWE(k, n): mask c, position j = m_c[t - j] (negated when it wraps), body = b[t]."""
    g = u64(glwe).reshape(k + 1, n)
    j = np.arange(n)
    src = (t - j) % n
    with np.errstate(over="ignore"):
        mask = np.where(j <= t, g[:k, src], neg(g[:k, src]))
    return np.concatenate([mask.reshape(-1), g[k, t:t + 1]])


def const_embed(lwe, k, n):
    """GLWE(k, n) whose constant coefficient decrypts like the LWE(k n): inverse of sample_extract at t = 0."""
    lwe = u64(lwe)
    a = lwe[: k * n].reshape(k, n)
    out = np.zeros((k + 1, n), dtype=np.uint64)
    out[:k, 0] = a[:, 0]
    out[:k, 1:] = neg(a[:, :0:-1])
    out[k, 0] = lwe[k * n]
    return out.reshape(-1)


# ---- tfhe SignedDecomposer ---------------------------------------------------------------------------------------------

def decompose(x, base_log, level):
    """Balanced signed digits of the closest representable value, finest level first: [level][...] int64.

    closest: round x to the nearest multiple of 2^(64 - base_log level), halves up (carry out of 2^64 dropped).
    digits, from the finest: raw = the next base_log bits; a raw above B/2 becomes raw - B with a carry into the rest;
    exactly B/2 does the same only when the rest's next raw digit is B/2 or more (tfhe's tie rule), so the last
    level keeps +B/2."""
    x = u64(x)
    B = 1 << base_log
    nr = 64 - base_log * level
    rest = (x >> U64(nr)) + ((x >> U64(nr - 1)) & U64(1))  # < 2^(base_log level) + 1
    out = np.empty((level,) + x.shape, dtype=np.int64)
    for t in range(level):
        raw = (rest & U64(B - 1)).astype(np.int64)
        rest = rest >> U64(base_log)
        nxt = (rest & U64(B - 1)).astype(np.int64)
        carry = (raw > B // 2) | ((raw == B // 2) & (nxt >= B // 2))
        out[t] = raw - carry * B
        rest = rest + carry.astype(np.uint64)
    return out


def decompose_bigint(x, base_log, level):
    """The same definition on one Python int, for the checks of decompose()."""
    B = 1 << base_log
    nr = 64 - base_log * level
    v = ((x + (1 << (nr - 1))) >> nr) % (1 << (base_log * level))
    digits = []
    for _ in range(level):
        raw, v = v % B, v // B
        if raw > B // 2 or (raw == B // 2 and v % B >= B // 2):
            raw -= B
            v += 1
        digits.append(raw)
    return digits


# ---- modulus switch and blind rotation ---------------------------------------------------------------------------------

def modswitch(x):
    """tfhe fast_pbs_modulus_switch(N = 1024, log_lut_count 3): round(x / 2^56) * 8, a multiple of 8 in [0, 2048]."""
    return (((int(x) >> 55) + 1) >> 1) << 3


def br_accumulator(body):
    """trivial GLWE: the test polynomial of lwe_msb_bit_to_glev_by_trace_with_preprocessing times X^-modswitch(b)."""
    i = np.arange(N)
    val = np.array([(1 << 64) - (1 << (63 - 2 * (k % 8 + 1))) for k in range(8)], dtype=np.uint64)[i % 8]
    val[: N // 2] = neg(val[: N // 2])
    tv = np.roll(val, -N // 2)
    acc = np.zeros((3, N), dtype=np.uint64)
    acc[2] = mono_mul(tv, 2 * N - modswitch(body))
    return acc


def external_product(ggsw, glwe, base_log, level):
    """sum_r sum_t digit_t(glwe_r) * ggsw[level - 1 - t][r][c] for every output polynomial c: [k+1][n].
    ggsw [level][k+1][k+1][n] (coarsest level first), glwe [k+1][n]."""
    g = u64(ggsw)
    rows = g.shape[1]
    glwe = u64(glwe).reshape(rows, -1)
    out = np.zeros_like(glwe)
    with np.errstate(over="ignore"):
        for r in range(rows):
            dig = decompose(glwe[r], base_log, level)
            for t in range(level):
                if not dig[t].any():
                    continue
                for c in range(rows):
                    out[c] += negacyclic_mul(g[level - 1 - t, r, c], dig[t])
    return out


def cmux_step(acc, ggsw, shift, base_log, level):
    """acc + ggsw (x) (acc X^shift - acc), acc [3][n]."""
    acc = u64(acc).reshape(3, -1)
    with np.errstate(over="ignore"):
        diff = mono_mul(acc, shift) - acc
        return acc + external_product(ggsw, diff, base_log, level)


def br_step(acc, bsk_i, a_i):
    """one CMux of the blind rotation: rotation by modswitch(a_i) under bsk_i [1][3][3][N] (B = 2^23, l = 1).
    A rotation of 0 or 2N leaves the accumulator as it is."""
    d = modswitch(a_i) % (2 * N)
    if d == 0:
        return u64(acc).reshape(3, N).copy()
    return cmux_step(acc, bsk_i, d, 23, 1)


def blind_rotate(bsk, lwe, steps=LWE_N):
    """accumulator build and the first `steps` CMux steps; bsk [768][1][3][3][N], lwe [769]."""
    lwe = u64(lwe)
    acc = br_accumulator(lwe[LWE_N])
    for i in range(steps):
        if lwe[i] != 0:
            acc = br_step(acc, bsk[i], lwe[i])
    return acc.reshape(-1)


# ---- GLWE keyswitches --------------------------------------------------------------------------------------------------

def glwe_keyswitch(key, glwe, base_log, level):
    """keyswitch_glwe_ciphertext with the full key [in_k][level][out_size][n] (coarsest level first):
    body copied to the last output polynomial, plus sum_i sum_t digit_t(mask_i) * key[i][level - 1 - t]."""
    key = u64(key)
    in_k, _, out_size, n = key.shape
    g = u64(glwe).reshape(in_k + 1, n)
    out = np.zeros((out_size, n), dtype=np.uint64)
    out[out_size - 1] = g[in_k]
    with np.errstate(over="ignore"):
        for i in range(in_k):
            dig = decompose(g[i], base_log, level)
            for t in range(level):
                if not dig[t].any():
                    continue
                for c in range(out_size):
                    out[c] += negacyclic_mul(key[i, level - 1 - t, c], dig[t])
    return out.reshape(-1)


def lwe_keyswitch(ksk, lwe):
    """LWE(2048) -> LWE(768) over the ring N' = 256: const-embed, keyswitch (B = 2^4, l = 3), extract 0."""
    g = const_embed(lwe, 8, 256)
    out = glwe_keyswitch(u64(ksk).reshape(8, 3, 4, 256), g, 4, 3)
    return sample_extract(out, 3, 256, 0)


def auto_step(auto_std, i, glwe):
    """automorphism X -> X^kappa, kappa = N / 2^(i-1) + 1 (i = 1..10), then the keyswitch (B = 2^13, l = 3)."""
    kappa = N // (1 << (i - 1)) + 1
    pw = eval_x_k(u64(glwe).reshape(3, N), kappa)
    return glwe_keyswitch(u64(auto_std)[i - 1], pw, 13, 3)


def trace(auto_std, glwe, steps=10):
    g = u64(glwe).reshape(-1).copy()
    with np.errstate(over="ignore"):
        for i in range(1, steps + 1):
            g = g + auto_step(auto_std, i, g)
    return g


def scheme_switch(ss, glev):
    """GLEV [7][3][N] -> GGSW std [7][3][3][N]: rows 0, 1 = ss_i (x) GLEV level (B = 2^17, l = 2), row 2 = the GLEV."""
    glev = u64(glev).reshape(7, 3, N)
    ss = u64(ss).reshape(2, 2, 3, 3, N)
    out = np.zeros((7, 3, 3, N), dtype=np.uint64)
    for col in range(7):
        for i in range(2):
            out[col, i] = external_product(ss[i], glev[col], 17, 2)
        out[col, 2] = glev[col]
    return out.reshape(-1)


def circuit_bootstrap(keys, lwe, glev_from_acc):
    """LWE(768) -> GGSW std; keys = (bsk, auto_std, ss); glev_from_acc is the oracle's integer stage (bit-exact)."""
    bsk, auto_std, ss = keys
    acc = blind_rotate(bsk, lwe)
    glev = u64(glev_from_acc(acc)).reshape(7, 3 * N)
    traced = np.stack([trace(auto_std, glev[l]) for l in range(7)])
    return scheme_switch(ss, traced)


# ---- 8-bit LUT ladder --------------------------------------------------------------------------------------------------

def lut_cmux(acc, ggsw, i):
    """selector i of evaluate_8_to_8_cipher_lut: acc + ggsw_i (x) (acc X^-(2^i) - acc), B = 2^2, l = 7."""
    return cmux_step(acc, u64(ggsw).reshape(7, 3, 3, N), 2 * N - (1 << i), 2, 7)


def lut8_eval(ggsw8, lut2, selectors=8):
    """8 CMux selectors (LSB first) on both accumulators, then 4 extractions each -> [8][2049], bit t of acc a at 4a+t."""
    ggsw8 = u64(ggsw8).reshape(8, -1)
    out = np.zeros((8, 2 * N + 1), dtype=np.uint64)
    for a in range(2):
        acc = u64(lut2).reshape(2, 3, N)[a]
        for i in range(selectors):
            acc = lut_cmux(acc, ggsw8[i], i)
        for t in range(4):
            out[4 * a + t] = sample_extract(acc, 2, N, 256 * t)
    return out
