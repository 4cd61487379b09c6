"""The FP64 external-product kernels against exact integer arithmetic (tests/exact_ref.py).

(a) Small keys (bounds derived in tests/test_exact_ref_cpu.py): every FP64 product is an exact integer, so the GPU must
    equal the exact reference bit for bit, compared with ==.  The one deliberate exception is torus_from_scaled at
    f = +2^63 (DESIGN.md section 2), reached by a constructed LUT-ladder case and asserted exactly.
(b) The seeded real keys: the distance to the exact reference is the FP64 error of the kernel, bounded by a budget
    measured on one NVIDIA B200; each budget sits next to the oracle's own error from tests/test_exact_ref_cpu.py.
(c) The integer helpers of the kernels, exhaustively on the device (tests/device_helpers.cu)."""
import os
import subprocess
import sys
import traceback

import numpy as np
import pytest

import exact_ref as ex
from conftest import ROOT, log2max, sdiff
from test_batch_shapes_gpu import run_worker
from test_exact_ref_cpu import EDGE, oracle_br_step, small_ggsw, small_keys, tie_words

pytestmark = pytest.mark.gpu

N = 1024
CSRC = os.path.join(ROOT, "temp_fhe_transciphering_b200", "csrc")


@pytest.fixture(scope="module")
def small_ctx(cbs):
    c = cbs.Context(cbs.KeySet.from_arrays(*small_keys()), 0)
    yield c
    c.close()


def first_last_spread(n, k=64):
    return sorted(set(range(min(n, 8))) | set(range(max(0, n - 8), n)) | set(np.linspace(0, n - 1, k).astype(int).tolist()))


# ---- (a) small keys: bit-exact ------------------------------------------------------------------------------------

def test_small_keys_lwe_keyswitch(small_ctx):
    ksk = small_keys()[1]
    rng = np.random.default_rng(31)
    lwe = rng.integers(0, 2 ** 64, (8193, 2049), dtype=np.uint64)
    words = np.array(EDGE + tie_words(4, 3), dtype=np.uint64)
    lwe[::2] = words[rng.integers(0, len(words), (4097, 2049))]
    for n in (1, 2, 8193):
        got = small_ctx.keyswitch_lwe_ciphertext_by_glwe_keyswitch(lwe[:n])
        for p in first_last_spread(n):
            assert (got[p] == ex.lwe_keyswitch(ksk, lwe[p])).all(), (n, p)


def br_small_inputs():
    """every rotation 0, 8, ..., 2048 on one mask word with a body at every rotation; mask words at both sides of
    modulus-switch boundaries; two full random LWE"""
    rows = []
    for r in range(0, 2049, 8):
        lwe = np.zeros(769, dtype=np.uint64)
        w = (r // 8) << 56 if r < 2048 else (1 << 64) - 1
        lwe[(3 * r // 8) % 768] = w
        lwe[768] = ((256 - r // 8) % 256) << 56
        rows.append(lwe)
    for k in (0, 1, 2, 127, 128, 255):
        for s in (-1, 0):
            lwe = np.zeros(769, dtype=np.uint64)
            lwe[(11 * k) % 768] = ((k << 56) + (1 << 55) + s) % (1 << 64)
            lwe[768] = ((k << 56) + (1 << 55) + s) % (1 << 64)
            rows.append(lwe)
    rng = np.random.default_rng(32)
    rows += list(rng.integers(0, 2 ** 64, (2, 769), dtype=np.uint64))
    return np.stack(rows)


def _br_worker(mode, outdir, q):
    try:
        os.environ["CBS_BR_LOWLAT"] = str(mode)
        sys.path.insert(0, ROOT)
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import torch
        import temp_fhe_transciphering_b200 as cbs
        ctx = cbs.Context(cbs.KeySet.from_arrays(*small_keys()), 0)
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        inp = br_small_inputs()
        wave = np.resize(np.arange(len(inp)), 4 * sms + 5)  # one v4 wave plus a tail
        np.savez(os.path.join(outdir, "br.npz"), all=ctx.blind_rotate(inp), one=ctx.blind_rotate(inp[:1]),
                 six=ctx.blind_rotate(inp[-6:]), wave=ctx.blind_rotate(inp[wave]), wave_idx=wave)
        ctx.close()
        q.put("ok")
    except BaseException:
        q.put(traceback.format_exc())
        raise


@pytest.fixture(scope="module")
def br_exact():
    bsk = small_keys()[0]
    return np.stack([ex.blind_rotate(bsk, x) for x in br_small_inputs()])


@pytest.mark.parametrize("mode", [0, 2])
def test_small_keys_blind_rotation_both_kernels(tmp_path, br_exact, mode):
    """CBS_BR_LOWLAT = 0: k_blind_rotate_v4 for every batch; 2: the team kernel k_blind_rotate_ll."""
    run_worker(_br_worker, mode, str(tmp_path))
    r = np.load(tmp_path / "br.npz")
    want = br_exact
    bad = np.flatnonzero((r["all"] != want).any(axis=1))
    assert bad.size == 0, bad[:16].tolist()
    assert (r["one"] == want[:1]).all() and (r["six"] == want[-6:]).all()
    bad = np.flatnonzero((r["wave"] != want[r["wave_idx"]]).any(axis=1))
    assert bad.size == 0, bad[:16].tolist()


def test_small_keys_trace_scheme_switch_and_circuit_bootstrap(small_ctx, orc):
    bsk, ksk, auto, ss = small_keys()
    rng = np.random.default_rng(33)
    g = rng.integers(0, 2 ** 64, (3, 3 * N), dtype=np.uint64)
    g[0, :1000] = np.resize(np.array(tie_words(13, 3), dtype=np.uint64), 1000)
    got = small_ctx.trace_assign(g)
    for i in range(3):
        assert (got[i] == ex.trace(auto, g[i])).all(), i
    glev = rng.integers(0, 2 ** 64, (2, 7, 3 * N), dtype=np.uint64)
    glev[0, 0, :2000] = np.resize(np.array(tie_words(17, 2), dtype=np.uint64), 2000)
    got = small_ctx.switch_scheme(glev)
    for i in range(2):
        assert (got[i] == ex.scheme_switch(ss, glev[i])).all(), i
    lwe = rng.integers(0, 2 ** 64, (2, 769), dtype=np.uint64)
    got = small_ctx.circuit_bootstrap_lwe_ciphertext_by_trace_with_preprocessing(lwe)
    for i in range(2):
        assert (got[i] == ex.circuit_bootstrap((bsk, auto, ss), lwe[i], orc.glev_from_acc)).all(), i


@pytest.mark.parametrize("trivial", [True, False])
def test_small_entry_lut_ladder(small_ctx, trivial):
    """each selector alone (the other GGSWs all-zero keep the accumulator exactly as it is), then all 8 together; trivial
    accumulators (zero masks: the first CMux skips the mask transforms) and non-trivial ones"""
    rng = np.random.default_rng(34 + trivial)
    full = small_ggsw(rng, 8).reshape(8, -1)
    ggsw = np.zeros((9, 8, full.shape[1]), dtype=np.uint64)
    for i in range(8):
        ggsw[i, i] = full[i]
    ggsw[8] = full
    luts = rng.integers(0, 2 ** 64, (9, 1, 2, 3 * N), dtype=np.uint64)
    if trivial:
        luts[:, :, :, :2 * N] = 0
    got = small_ctx.evaluate_8_to_8_cipher_lut(ggsw, luts)
    for b in range(9):
        assert (got[b, 0] == ex.lut8_eval(ggsw[b], luts[b, 0])).all(), b


def test_lut_ladder_reaches_f_plus_2_63(small_ctx):
    """The body row [-2^62, 2^62, ..., 2^62] times X^-1 minus itself is 2^63 at coefficient 0 and 0 elsewhere: one digit
    +2 at the coarsest level, whose transform is exact.  A GGSW whose only word is 2^62 at (level 0, row 2, column 2,
    coefficient 0) makes the inverse transform output exactly 2^63.  tfhe rounds it to 2^63; torus_from_scaled gives
    2^63 - 1 (DESIGN.md section 2): the GPU must differ from the exact reference by exactly -1 there and nowhere else."""
    ggsw = np.zeros((1, 8, 7, 3, 3, N), dtype=np.uint64)
    ggsw[0, 0, 0, 2, 2, 0] = 1 << 62
    lut = np.zeros((1, 1, 2, 3, N), dtype=np.uint64)
    lut[..., 2, :] = 1 << 62
    lut[..., 2, 0] = (1 << 64) - (1 << 62)
    got = small_ctx.evaluate_8_to_8_cipher_lut(ggsw.reshape(1, 8, -1), lut.reshape(1, 1, 2, -1))[0, 0]
    want = ex.lut8_eval(ggsw[0], lut[0, 0])
    assert int(want[0, 2048]) == 1 << 62 and int(want[4, 2048]) == 1 << 62  # -2^62 + 2^63
    d = sdiff(got, want)
    assert d[0, 2048] == -1 and d[4, 2048] == -1
    d[0, 2048] = d[4, 2048] = 0
    assert not d.any()


# ---- (b) real keys: FP64 error budgets ------------------------------------------------------------------------------

def test_real_keys_blind_rotation_every_step(ctx, orc, keyset):
    """The 769 prefixes of one LWE (mask words 0..i kept, the rest zero, so later steps are skipped) in one batch: the
    first 4 x 148 run k_blind_rotate_v4, the tail the team kernel.  Step i + 1 must equal the exact step applied to the
    GPU's accumulator i, within the budget; the build (no step) is exact."""
    rng = np.random.default_rng(41)
    lwe = rng.integers(0, 2 ** 64, 769, dtype=np.uint64)
    pre = np.zeros((769, 769), dtype=np.uint64)
    for i in range(769):
        pre[i, :i] = lwe[:i]
        pre[i, 768] = lwe[768]
    acc = ctx.blind_rotate(pre).reshape(769, 3, N)
    assert (acc[0] == ex.br_accumulator(lwe[768])).all()
    bsk = keyset.bsk
    err, orc_err = np.zeros(768), np.zeros(768)
    for i in range(768):
        want = ex.br_step(acc[i], bsk[i], lwe[i])
        err[i] = log2max(sdiff(acc[i + 1], want))
        orc_err[i] = log2max(sdiff(oracle_br_step(orc, bsk[i], acc[i], lwe[i]), want))
    print(f"blind rotation step: max {err.max():.2f} (step {int(err.argmax())}), median {np.median(err):.2f}; "
          f"oracle on the same accumulators: max {orc_err.max():.2f}, median {np.median(orc_err):.2f}")
    # measured on one B200 (1000 W, 1965 MHz): max 40.53 (step 445), median 39.97; oracle - exact on uniform
    # accumulators 40.43 (tests/test_exact_ref_cpu.py).  Budget: measured + 1 bit, and at most the oracle's + 1 bit.
    assert err.max() < 41.5, (int(err.argmax()), err.max())
    assert err.max() <= orc_err.max() + 1.0, (err.max(), orc_err.max())


def test_real_keys_lut_cmux_and_ladder(ctx):
    """uniform 64-bit GGSW words: one CMux per selector position (the other GGSWs zero), the whole ladder against the exact
    chain, and the worst-case magnitudes (GGSW words +-2^63, 2^63 - 1; accumulator differences with digits +-B/2 at
    every level)."""
    rng = np.random.default_rng(42)
    full = rng.integers(0, 2 ** 64, (8, 7 * 9 * N), dtype=np.uint64)
    ggsw = np.zeros((10, 8, full.shape[1]), dtype=np.uint64)
    for i in range(8):
        ggsw[i, i] = full[i]
    ggsw[8] = full
    ext = np.array([1 << 63, (1 << 63) - 1, (1 << 64) - (1 << 63) + 1], dtype=np.uint64)
    ggsw[9] = ext[rng.integers(0, 3, full.shape)]
    luts = rng.integers(0, 2 ** 64, (10, 1, 2, 3 * N), dtype=np.uint64)
    # digits +-2 at every level: words of the form sum_t (+-2) 4^t 2^50 (alternating, so every difference is large)
    big = sum(2 << (50 + 2 * t) for t in range(7)) % (1 << 64)
    luts[9, 0, :, :] = np.where(np.arange(3 * N) % 2 == 0, np.uint64(big), np.uint64(0) - np.uint64(big))
    got = ctx.evaluate_8_to_8_cipher_lut(ggsw, luts)
    err = [log2max(sdiff(got[b, 0], ex.lut8_eval(ggsw[b], luts[b, 0]))) for b in range(10)]
    print("LUT CMux per selector", [round(e, 2) for e in err[:8]], "ladder", round(err[8], 2), "extreme", round(err[9], 2))
    # measured on one B200: per selector 20.42 .. 20.73, ladder 21.98, extreme words 22.12; oracle - exact on the ladder
    # 21.75 .. 21.91.  Budgets: measured + 1 bit.
    assert max(err[:8]) < 21.8 and err[8] < 23.0, err
    assert err[9] < 23.2, err


def test_real_keys_scheme_switch_keyswitch_and_trace(ctx, keyset):
    rng = np.random.default_rng(43)
    glev = rng.integers(0, 2 ** 64, (2, 7, 3 * N), dtype=np.uint64)
    got = ctx.switch_scheme(glev)
    e_ss = max(log2max(sdiff(got[i], ex.scheme_switch(keyset.ss, glev[i]))) for i in range(2))
    big = rng.integers(0, 2 ** 64, (64, 2049), dtype=np.uint64)
    got = ctx.keyswitch_lwe_ciphertext_by_glwe_keyswitch(big)
    e_ks = max(log2max(sdiff(got[i], ex.lwe_keyswitch(keyset.ksk, big[i]))) for i in range(64))
    g = rng.integers(0, 2 ** 64, (3, 3 * N), dtype=np.uint64)
    got = ctx.trace_assign(g)
    e_tr = max(log2max(sdiff(got[i], ex.trace(keyset.auto_std, g[i]))) for i in range(3))
    print(f"scheme switch {e_ss:.2f}, LWE keyswitch {e_ks:.2f}, 10-step trace {e_tr:.2f}")
    # measured on one B200: scheme switch 34.84, LWE keyswitch 22.08, 10-step trace 15.66 (no digit flip: the chain stays
    # within 2^16 of the exact chain); oracle - exact: scheme switch 35.05, LWE keyswitch 21.32, one automorphism step
    # 8.55.  Budgets: measured + 1 bit.
    assert e_ss < 35.9 and e_ks < 23.1 and e_tr < 16.7, (e_ss, e_ks, e_tr)


# ---- (c) device helpers ---------------------------------------------------------------------------------------------

def test_device_helpers_exhaustive(tmp_path):
    exe = tmp_path / "device_helpers"
    subprocess.check_call(["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17",
                           "-I", CSRC, os.path.join(ROOT, "tests", "device_helpers.cu"), "-o", str(exe)])
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    print(out.stdout)
    assert out.returncode == 0, out.stdout + out.stderr
