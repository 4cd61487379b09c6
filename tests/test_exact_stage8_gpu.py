"""The stage-8 FP64 external-product kernels k_max_ladder and k_lut8_gather, through cbs_max_of_two and cbs_lut8_gather_eval,
against the exact integer reference of tests/exact_stage8_ref.py.

(a) Small GGSW (|g| <= 2^24, bound in tests/test_exact_ref_cpu.py): every FP64 product is an exact integer, so the GPU must
    equal the exact reference bit for bit (==), except for torus_from_scaled at f = +2^63 (DESIGN.md section 2), reached by a
    constructed case and asserted exactly.
(b) Uniform 64-bit GGSW: the distance to the exact reference is the FP64 error of the kernel, bounded by a budget measured on
    one NVIDIA B200.
(c) Whole stage-8 calls with the seeded keyset, against the exact ladders fed by the GPU's own keyswitch and circuit
    bootstrap (pinned to exact arithmetic in tests/test_exact_gpu.py, batch-shape independent by
    tests/test_batch_shapes_gpu.py).
Host-side argument checks of the two entry points run first: nothing out of range reaches a kernel."""
import ctypes
import multiprocessing
import os
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

import exact_ref as ex
import exact_stage8_ref as s8
from conftest import log2max, sdiff
from test_exact_gpu import first_last_spread
from test_exact_ref_cpu import EDGE, small_ggsw, small_keys, tie_words
from test_partitions_gpu import _decrypt, _encrypt

pytestmark = pytest.mark.gpu

N = 1024
GGSW_WORDS = 7 * 9 * N


@pytest.fixture(scope="module")
def small_ctx(cbs):
    c = cbs.Context(cbs.KeySet.from_arrays(*small_keys()), 0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def pool():
    """the exact side is CPU-bound numpy (one external product ~ 30 ms): its independent ladders run in worker processes"""
    with ProcessPoolExecutor(max_workers=min(16, os.cpu_count() or 1), mp_context=multiprocessing.get_context("spawn")) as p:
        yield p


@pytest.fixture(scope="module")
def plan_lib(tmp_path_factory):
    return s8.build_plan_lib(tmp_path_factory.mktemp("plan_dump"))


def _ladder_bits(pool, ggsw, op, pairs):
    """exact max_of_two output bits for (va, vb, j) triples, e0 = "a" (the GPU's start)"""
    pairs = list(pairs)
    return dict(zip(pairs, pool.map(s8.max_of_two_bit, [ggsw[a] for a, b, j in pairs], [ggsw[b] for a, b, j in pairs],
                                    [op[a, j] for a, b, j in pairs], [op[b, j] for a, b, j in pairs], ["a"] * len(pairs))))


# ---- argument checks ------------------------------------------------------------------------------------------------

def _p(a, ctype):
    return None if a is None else a.ctypes.data_as(ctypes.POINTER(ctype))


def test_entry_points_reject_bad_arguments_before_queueing(cbs, small_ctx):
    L, h = cbs.lib(), small_ctx._h
    u64, i32 = ctypes.c_uint64, ctypes.c_int32
    g = np.zeros((2, 16, GGSW_WORDS), dtype=np.uint64)
    op = np.zeros((2, 16, 3 * N), dtype=np.uint64)
    out = np.zeros((1, 16, 2 * N + 1), dtype=np.uint64)
    zero, one, two, neg = (np.array([v], dtype=np.int32) for v in (0, 1, 2, -1))

    def mo2(ggsw=g, o=op, nvals=2, a=zero, b=one, npairs=1, dst=out):
        return L.cbs_max_of_two(h, _p(ggsw, u64), _p(o, u64), nvals, _p(a, i32), _p(b, i32), npairs, _p(dst, u64))

    before = small_ctx.launch_count
    bad = [dict(ggsw=None), dict(o=None), dict(a=None), dict(b=None), dict(dst=None), dict(nvals=-1), dict(npairs=-1),
           dict(a=two), dict(b=two), dict(a=neg), dict(b=neg), dict(nvals=0), dict(nvals=1, b=one)]
    for kw in bad:
        assert mo2(**kw) == 1, kw  # CBS_ERR_ARG
    assert mo2(npairs=0) == 0
    assert small_ctx.launch_count == before

    lut = np.zeros((2, 3 * N), dtype=np.uint64)
    sel = np.full((2, 8), -1, dtype=np.int32)
    sel[0, 3] = 1
    li, oi = np.array([0, 1], dtype=np.int32), np.array([0, 4], dtype=np.int32)
    rows = np.zeros((8, 2 * N + 1), dtype=np.uint64)

    def gat(ggsw=g.reshape(-1, GGSW_WORDS)[:2], nbits=2, s=sel, luts=lut, nluts=2, lidx=li, oidx=oi, njobs=2, dst=rows, nout=8):
        return L.cbs_lut8_gather_eval(h, _p(ggsw, u64), nbits, _p(s, i32), _p(luts, u64), nluts, _p(lidx, i32), _p(oidx, i32),
                                      njobs, _p(dst, u64), nout)

    def with_sel(j, i, v):
        s = sel.copy()
        s[j, i] = v
        return s

    bad = [dict(ggsw=None), dict(s=None), dict(luts=None), dict(lidx=None), dict(oidx=None), dict(dst=None),
           dict(nbits=-1), dict(nluts=-1), dict(njobs=-1), dict(nout=-1),
           dict(s=with_sel(1, 7, 2)), dict(s=with_sel(0, 0, -2)), dict(nbits=1),            # selector outside [-1, nbits)
           dict(lidx=np.array([0, 2], np.int32)), dict(lidx=np.array([-1, 0], np.int32)), dict(nluts=1),
           dict(oidx=np.array([0, 5], np.int32)), dict(oidx=np.array([-1, 4], np.int32)), dict(nout=7),  # window outside
           dict(oidx=np.array([0, 3], np.int32)), dict(oidx=np.array([4, 4], np.int32))]                # overlapping
    for kw in bad:
        assert gat(**kw) == 1, kw
    assert gat(njobs=0) == 0
    assert small_ctx.launch_count == before
    # the valid calls: the GGSW transform and the ladder kernel, counted
    assert mo2() == 0 and small_ctx.launch_count == before + 2
    assert gat() == 0 and small_ctx.launch_count == before + 4


# ---- (a) small GGSW: bit-exact ------------------------------------------------------------------------------------

PAIRS19 = [(0, 1), (1, 0), (2, 2), (3, 4), (4, 3), (1, 1), (0, 4), (4, 0), (2, 3), (3, 2), (1, 4), (4, 1), (0, 2), (2, 0),
           (3, 3), (4, 4), (0, 3), (1, 2), (2, 4)]  # 19 x 16 groups at 2 per CTA: one 296-group wave + an 8-group tail


def test_small_max_of_two(small_ctx, pool):
    """5 values (small GGSW); operands uniform, EDGE words and the B = 2^2, l = 7 rounding and digit ties; npairs = 1 and 19
    with self-pairs, a value in several pairs and both orders of a pair"""
    rng = np.random.default_rng(91)
    ggsw = small_ggsw(rng, 5 * 16).reshape(5, 16, -1)
    op = rng.integers(0, 2 ** 64, (5, 16, 3 * N), dtype=np.uint64)
    words = np.array(EDGE + tie_words(2, 7), dtype=np.uint64)
    op[1] = words[rng.integers(0, len(words), op[1].shape)]
    op[3, ::2] = words[rng.integers(0, len(words), op[3, ::2].shape)]
    one = small_ctx.max_of_two(ggsw, op, [4], [3])
    got = small_ctx.max_of_two(ggsw, op, [a for a, b in PAIRS19], [b for a, b in PAIRS19])
    assert one.shape == (1, 16, 2 * N + 1) and got.shape == (19, 16, 2 * N + 1)
    assert (one[0] == got[PAIRS19.index((4, 3))]).all()  # the same pair alone and inside the 19-pair batch
    checks = [(0, one[0], (4, 3), j) for j in (0, 15)]
    for f in sorted(set(first_last_spread(19 * 16, 12)) | {16 * PAIRS19.index((1, 0)) + 15, 16 * PAIRS19.index((2, 2)) + 7}):
        p, j = divmod(f, 16)
        checks.append((p, got[p], PAIRS19[p], j))
    want = _ladder_bits(pool, ggsw, op, {(a, b, j) for _, _, (a, b), j in checks})
    for p, rows, (a, b), j in checks:
        assert (rows[j] == want[a, b, j]).all(), (p, a, b, j)


def _gather_jobs(rng, njobs, nbits, nluts):
    """all 8 selectors (the last GGSW index among them), none (pure extraction), the same GGSW twice, each selector alone,
    then random selector sets with -1 gaps; non-monotone LUT indices"""
    jobs = [rng.permutation(nbits)[:8].tolist(), [-1] * 8]
    jobs[0][int(rng.integers(0, 8))] = nbits - 1
    twice = rng.integers(0, nbits, 8).tolist()
    twice[2] = twice[6] = int(rng.integers(0, nbits))
    jobs.append(twice)
    for i in range(8):
        jobs.append([int(rng.integers(0, nbits)) if k == i else -1 for k in range(8)])
    while len(jobs) < njobs:
        jobs.append([int(rng.integers(0, nbits)) if rng.random() < 0.75 else -1 for _ in range(8)])
    lut_index = rng.integers(0, nluts, len(jobs))
    lut_index[:3] = [nluts - 1, 0, 2]
    return np.array(jobs[:njobs], dtype=np.int32), lut_index[:njobs].astype(np.int32)


def _windows(rng, njobs):
    """permuted output windows with holes: slot k starts at 5 k + (k & 1), so windows are two rows apart or adjacent"""
    starts = np.array([5 * k + (k & 1) for k in range(njobs)], dtype=np.int32)
    return starts[rng.permutation(njobs)], 5 * njobs + 3


def test_small_gathered_ladder(small_ctx, pool):
    """njobs 1, 3, 4, 5 and 597 (4 groups per CTA: one 592-job wave + a tail); trivial and non-trivial accumulators; rows no
    job writes are zero"""
    rng = np.random.default_rng(92)
    nbits, nluts = 12, 6
    ggsw = small_ggsw(rng, nbits)
    luts = rng.integers(0, 2 ** 64, (nluts, 3 * N), dtype=np.uint64)
    luts[[0, 3], :2 * N] = 0  # trivial accumulators
    luts[4, 2 * N:2 * N + 500] = np.resize(np.array(tie_words(2, 7), dtype=np.uint64), 500)
    sel, lut_index = _gather_jobs(rng, 597, nbits, nluts)
    checked = set()
    runs = []
    for njobs in (1, 3, 4, 5, 597):
        out_index, nout = _windows(rng, njobs)
        got = small_ctx.evaluate_gathered_luts(ggsw, sel[:njobs], luts, lut_index[:njobs], out_index, nout)
        written = np.zeros(nout, dtype=bool)
        for o in out_index:
            written[o:o + 4] = True
        assert not got[~written].any(), njobs
        jobs = range(njobs) if njobs < 597 else sorted(set(first_last_spread(njobs, 16)) | set(range(11)))
        runs.append((got, out_index, jobs))
        checked.update(jobs)
    order = sorted(checked)
    want = dict(zip(order, pool.map(s8.lut8_gather, [ggsw] * len(order), [sel[j].tolist() for j in order],
                                    [luts[lut_index[j]] for j in order])))
    for got, out_index, jobs in runs:
        for j in jobs:
            o = out_index[j]
            assert (got[o:o + 4] == want[j]).all(), (len(out_index), j, sel[j].tolist(), int(lut_index[j]))


def test_small_gathered_ladder_reaches_f_plus_2_63(small_ctx):
    """the construction of test_exact_gpu.py::test_lut_ladder_reaches_f_plus_2_63 with selector 0 only, as two jobs: the
    GPU differs from exact by exactly -1 at the two body words (torus_from_scaled gives 2^63 - 1, DESIGN.md section 2)"""
    ggsw = np.zeros((1, 7, 3, 3, N), dtype=np.uint64)
    ggsw[0, 0, 2, 2, 0] = 1 << 62
    lut = np.zeros((1, 3, N), dtype=np.uint64)
    lut[0, 2, :] = 1 << 62
    lut[0, 2, 0] = (1 << 64) - (1 << 62)
    sel = np.array([[0] + [-1] * 7] * 2, dtype=np.int32)
    got = small_ctx.evaluate_gathered_luts(ggsw, sel, lut, [0, 0], [0, 4], 8)
    want = s8.lut8_gather(ggsw.reshape(1, -1), [0] + [-1] * 7, lut[0])
    assert int(want[0, 2048]) == 1 << 62
    d = sdiff(got, np.concatenate([want, want]))
    assert d[0, 2048] == -1 and d[4, 2048] == -1
    d[0, 2048] = d[4, 2048] = 0
    assert not d.any()


# ---- (b) uniform 64-bit GGSW: FP64 budgets --------------------------------------------------------------------------

def test_real_max_of_two_every_output_bit(ctx, pool):
    rng = np.random.default_rng(93)
    ggsw = rng.integers(0, 2 ** 64, (2, 16, GGSW_WORDS), dtype=np.uint64)
    op = rng.integers(0, 2 ** 64, (2, 16, 3 * N), dtype=np.uint64)
    got = ctx.max_of_two(ggsw, op, [0], [1])[0]
    want = _ladder_bits(pool, ggsw, op, [(0, 1, j) for j in range(16)])
    err = [log2max(sdiff(got[j], want[0, 1, j])) for j in range(16)]
    print("max_of_two, uniform GGSW, log2 max |GPU - exact| per output bit:", [round(e, 2) for e in err])
    assert max(err) < MAX_OF_TWO_BUDGET, err


def test_real_gathered_ladder(ctx, orc):
    """one job per single selector position, a full ladder, and GGSW words of the worst-case magnitudes (+-2^63, 2^63 - 1);
    the oracle on the same inputs (zero GGSW at the -1 positions) gives the error the GPU is held to as well"""
    rng = np.random.default_rng(94)
    ggsw = rng.integers(0, 2 ** 64, (16, GGSW_WORDS), dtype=np.uint64)
    ext = np.array([1 << 63, (1 << 63) - 1, (1 << 64) - (1 << 63) + 1], dtype=np.uint64)
    ggsw[8:] = ext[rng.integers(0, 3, ggsw[8:].shape)]
    luts = rng.integers(0, 2 ** 64, (3, 3 * N), dtype=np.uint64)
    sel = [[k if i == k else -1 for i in range(8)] for k in range(8)] + [list(range(8)), list(range(8, 16))]
    lut_index = [k % 3 for k in range(10)]
    got = ctx.evaluate_gathered_luts(ggsw, sel, luts, lut_index, [4 * k for k in range(10)], 40).reshape(10, 4, -1)
    err, orc_err = [], []
    for k in range(10):
        want = s8.lut8_gather(ggsw, sel[k], luts[lut_index[k]])
        g8 = np.stack([ggsw[s] if s >= 0 else np.zeros(GGSW_WORDS, np.uint64) for s in sel[k]])
        o = orc.lut8_eval(orc.ggsw_to_fourier(g8), np.stack([luts[lut_index[k]]] * 2))[:4]
        err.append(log2max(sdiff(got[k], want)))
        orc_err.append(log2max(sdiff(o, want)))
    print("gathered ladder, log2 max |GPU - exact|: per selector", [round(e, 2) for e in err[:8]], "ladder",
          round(err[8], 2), "extreme", round(err[9], 2), "| oracle:", [round(e, 2) for e in orc_err])
    assert max(err[:8]) < GATHER_SINGLE_BUDGET and err[8] < GATHER_LADDER_BUDGET and err[9] < GATHER_EXTREME_BUDGET, err
    for k in range(10):
        assert err[k] <= orc_err[k] + 1.0, (k, err[k], orc_err[k])


# ---- (c) whole calls, seeded keyset ---------------------------------------------------------------------------------

def _gpu_bootstrap(ctx):
    def boot(rows):
        ks = ctx.keyswitch_lwe_ciphertext_by_glwe_keyswitch(np.stack(rows))
        return (ctx.circuit_bootstrap_lwe_ciphertext_by_trace_with_preprocessing(ks),
                ctx.lwe_msb_bit_to_glev_by_trace_with_preprocessing(ks))
    return boot


MAX_PATTERNS = {"equal": [46803] * 4, "prefix": [40014, 40015, 40015, 40014], "distinct": [20962, 64797, 2177, 44457]}
LADDER_BITS = (0, 7, 14, 15)


@pytest.mark.parametrize("pattern", list(MAX_PATTERNS))
def test_max_u16_ladder_against_exact(ctx, keyset, pool, monkeypatch, pattern):
    """cbs_max_u16 with CBS_MAX_VARIANT=ladder at 2, 3 (the odd value carried with its GGSW and operand) and 4 values: every
    ladder of the tree against the exact ladder (e0 = "a") on the GPU's keyswitch + circuit bootstrap of the ladder's
    inputs, operands = 2 x GLEV index 0; a later tree level takes the GPU's own maxima of the level below"""
    import ref_io
    monkeypatch.setenv("CBS_MAX_VARIANT", "ladder")
    vals = MAX_PATTERNS[pattern]
    lwe = _encrypt(keyset, vals, 960 + len(pattern)).reshape(4, 16, -1)
    out = {n: ctx.max_u16(lwe[:n]) for n in (2, 3, 4)}
    m23 = ctx.max_u16(lwe[2:4])
    for n in (2, 3, 4):
        assert _decrypt(out[n], keyset) == [max(vals[:n])], (pattern, n)
    # (GPU output, input a rows, input b rows, cleartext a, cleartext b)
    ladders = [(out[2], lwe[0], lwe[1], vals[0], vals[1]), (out[3], out[2], lwe[2], max(vals[:2]), vals[2]),
               (m23, lwe[2], lwe[3], vals[2], vals[3]), (out[4], out[2], m23, max(vals[:2]), max(vals[2:]))]
    boot = _gpu_bootstrap(ctx)
    tasks = []
    for k, (_, ra, rb, va, vb) in enumerate(ladders):
        ggsw, glev = boot(list(ra) + list(rb))
        op = np.stack([s8.glev_to_operand(g) for g in glev])
        # each operand decrypts to its bit at 2^63: "level 1" is GLEV index 0
        bits = np.array([(v >> (15 - j)) & 1 for v in (va, vb) for j in range(16)], dtype=np.uint8)
        ph = ref_io.lwe_phase(np.stack([ex.sample_extract(o, 2, N, 0) for o in op]), keyset.glwe_sk)
        assert (ref_io.decode_bit(ph) == bits).all(), (pattern, k)
        ggsw, op = ggsw.reshape(2, 16, -1), op.reshape(2, 16, -1)
        tasks += [(ggsw[0], ggsw[1], op[0, j], op[1, j]) for j in LADDER_BITS]
    refs = list(pool.map(s8.max_of_two_bit, *zip(*tasks)))
    err = np.array([[log2max(sdiff(ladders[k][0][j], refs[k * len(LADDER_BITS) + i])) for i, j in enumerate(LADDER_BITS)]
                    for k in range(len(ladders))])
    print(f"max_u16 ladder ({pattern}), log2 max |GPU - exact| per ladder x bit {LADDER_BITS}:", err.round(2).tolist())
    assert err.max() < WHOLE_LADDER_BUDGET, err


@pytest.mark.parametrize("name,n", [("max_lut", 2), ("max_lut", 3), ("sum", 2), ("sum", 3), ("ip", 2), ("ip", 4)])
def test_lut_circuits_against_exact(ctx, keyset, pool, plan_lib, name, n):
    """cbs_max_u16_lut, cbs_sum_u16 and cbs_inner_product_u16 (1 and 2 pairs) against the plan executor with exact ladders,
    adds, gathers and refreshes and the GPU's keyswitch + circuit bootstrap of the executor's own rows"""
    vals = {2: [40014, 40015], 3: [65535, 1, 65534], 4: [65535, 12345, 65535, 54321]}[n]
    lwe = _encrypt(keyset, vals, 970 + n)
    kind, fn = {"max_lut": (s8.PLAN_MAX, ctx.max_u16_lut), "sum": (s8.PLAN_SUM, ctx.sum_u16),
                "ip": (s8.PLAN_IP, ctx.inner_product_u16)}[name]
    got = fn(lwe)
    h = n // 2
    want_val = {"max_lut": max(vals), "sum": sum(vals) % 65536,
                "ip": sum((x * y) % 65536 for x, y in zip(vals[:h], vals[h:])) % 65536}[name]
    assert _decrypt(got, keyset) == [want_val], (name, n)
    ref = np.stack(s8.run_plan(s8.get_plan(plan_lib, kind, n), list(lwe), _gpu_bootstrap(ctx), s8.ExactOps(map=pool.map)))
    assert _decrypt(ref, keyset) == [want_val], (name, n)
    err = [log2max(sdiff(got[i], ref[i])) for i in range(16)]
    print(f"{name} of {n}: log2 max |GPU - exact| per result row (MSB first):", [round(e, 2) for e in err])
    assert max(err) < WHOLE_LUT_BUDGET, err


# Budgets: the value measured on one NVIDIA B200 (1000 W power limit, 1965 MHz max SM clock) + 1 bit.
#   max_of_two, uniform GGSW, every output bit: max 23.36 (22.82 .. 23.36).
#   gathered ladder: per selector 20.28 .. 20.92, full ladder 21.90, extreme words 23.25; the oracle on the same inputs
#   20.16 .. 20.53, 21.84, 22.95.
#   cbs_max_u16 ladders (3 patterns x 4 ladders x 4 bits): 22.68 .. 23.48.
#   LUT circuits (max_lut 2, 3; sum 2, 3; ip 1, 2 pairs), every result row: 21.28 .. 22.11, one ladder's error: the
#   reference's rows and the GPU's internal rows differ by the ladders' FP64 error, which reaches a bootstrap output only
#   through a keyswitch digit or modulus-switch rounding.
MAX_OF_TWO_BUDGET = 24.4
GATHER_SINGLE_BUDGET = 21.9
GATHER_LADDER_BUDGET = 22.9
GATHER_EXTREME_BUDGET = 24.3
WHOLE_LADDER_BUDGET = 24.5
WHOLE_LUT_BUDGET = 23.1
