"""The exact stage-8 reference (tests/exact_stage8_ref.py) against what is already pinned: the oracle's max_of_two and LUT
ladder (bit-exact with small GGSW, bounds in tests/test_exact_ref_cpu.py), the exact 8-selector ladder of tests/exact_ref.py,
the C++ dry runs of the circuit plans (inner_product_plan_check, max_plan_check) and the C++ LUT tables."""
import multiprocessing
import os
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

import exact_ref as ex
import exact_stage8_ref as s8
from test_exact_ref_cpu import small_ggsw
from test_partitions_gpu import _patterns

N = 1024


@pytest.fixture(scope="module")
def plan_lib(tmp_path_factory):
    return s8.build_plan_lib(tmp_path_factory.mktemp("plan_dump"))


@pytest.fixture(scope="module")
def pool():
    with ProcessPoolExecutor(max_workers=min(8, os.cpu_count() or 1), mp_context=multiprocessing.get_context("spawn")) as p:
        yield p


def test_max_of_two_matches_oracle_reset_e(orc, pool):
    """e0 = "zero" on const-embedded LWE operands is the oracle's max_of_two(reset_e=1), which restates
    server_encrypted_compute.rs:34-98 (golden pin A): the step equations, the crossed operand naming and the bit order."""
    rng = np.random.default_rng(81)
    ga, gb = small_ggsw(rng, 16), small_ggsw(rng, 16)
    lwe_a, lwe_b = rng.integers(0, 2 ** 64, (2, 16, 2 * N + 1), dtype=np.uint64)
    want = orc.max_of_two(ga, gb, lwe_a, lwe_b, reset_e=True)
    bits = (0, 1, 14, 15)
    got = list(pool.map(s8.max_of_two_bit, [ga] * 4, [gb] * 4, [ex.const_embed(lwe_a[j], 2, N) for j in bits],
                        [ex.const_embed(lwe_b[j], 2, N) for j in bits], ["zero"] * 4))
    for k, j in enumerate(bits):
        assert (got[k] == want[j]).all(), j
    # the entry point of the whole value: the same bits through max_of_two
    assert (s8.max_of_two(ga, gb, [ex.const_embed(x, 2, N) for x in lwe_a], [ex.const_embed(x, 2, N) for x in lwe_b],
                          "zero", bits=[15])[0] == want[15]).all()


def test_lut8_gather_every_selector_is_lut8_eval():
    """selector i -> GGSW sel[i] through a permuted index table: the same 8 CMuxes as exact_ref.lut8_eval"""
    rng = np.random.default_rng(82)
    ggsw = small_ggsw(rng, 8)
    perm = rng.permutation(8)
    stored = np.empty_like(ggsw)
    stored[perm] = ggsw  # GGSW i stored at perm[i]
    lut2 = rng.integers(0, 2 ** 64, (2, 3 * N), dtype=np.uint64)
    lut2[0, :2 * N] = 0
    want = ex.lut8_eval(ggsw, lut2)
    for a in range(2):
        assert (s8.lut8_gather(stored, perm.tolist(), lut2[a]) == want[4 * a:4 * a + 4]).all(), a


@pytest.mark.parametrize("missing", [(0,), (7,), (1, 2, 5), tuple(range(8))])
def test_lut8_gather_constant_zero_selectors(orc, missing):
    """-1 skips the CMux: the same as an all-zero GGSW there, in exact_ref.lut8_eval and in the oracle (FP64, exact here)"""
    rng = np.random.default_rng(83 + len(missing))
    ggsw = small_ggsw(rng, 8)
    zeroed = ggsw.copy()
    zeroed[list(missing)] = 0
    sel = [-1 if i in missing else i for i in range(8)]
    lut2 = rng.integers(0, 2 ** 64, (2, 3 * N), dtype=np.uint64)
    want = ex.lut8_eval(zeroed, lut2)
    assert (orc.lut8_eval(orc.ggsw_to_fourier(zeroed), lut2) == want).all()
    for a in range(2):
        assert (s8.lut8_gather(ggsw, sel, lut2[a]) == want[4 * a:4 * a + 4]).all(), a
    if len(missing) == 8:  # no CMux at all: pure extraction
        assert (s8.lut8_gather(ggsw, sel, lut2[0]) == np.stack([ex.sample_extract(lut2[0], 2, N, 256 * t)
                                                                  for t in range(4)])).all()


def test_glue_operand_and_refresh():
    rng = np.random.default_rng(84)
    glev = rng.integers(0, 2 ** 64, (7, 3 * N), dtype=np.uint64)
    with np.errstate(over="ignore"):
        assert (s8.glev_to_operand(glev) == glev[0] << np.uint64(1)).all()
    assert (s8.glev_to_lwe(glev) == ex.sample_extract(glev[0] * np.uint64(2), 2, N, 0)).all()


def test_lut_accumulators_decode_to_the_library_tables(plan_lib):
    assert plan_lib.plan_num_luts() == s8.NUM_LUTS
    for lut in range(s8.NUM_LUTS):
        for idx in range(256):
            assert s8.ip_lut_value(lut, idx) == plan_lib.plan_lut_value(lut, idx), (lut, idx)
    acc = s8.lut_accumulators().reshape(s8.NUM_LUTS, 2, 3, N)
    assert not acc[:, :, :2].any()  # trivial: zero masks
    body = acc[:, :, 2]
    assert not (body & np.uint64((1 << 63) - 1)).any()
    for lut in range(s8.NUM_LUTS):
        for a in range(2):
            for i in range(N):
                want = (plan_lib.plan_lut_value(lut, i % 256) >> (4 * a + i // 256)) & 1
                assert int(body[lut, a, i] >> np.uint64(63)) == want, (lut, a, i)


def _clear_rows(vals):
    return [(v >> (15 - w)) & 1 for v in vals for w in range(16)]


def _clear_bootstrap(rows):
    return list(rows), list(rows)


def _run_clear(plan, vals):
    out = s8.run_plan(plan, _clear_rows(vals), _clear_bootstrap, s8.ClearOps())
    return sum(b << (15 - i) for i, b in enumerate(out))


def _value_sets(n, seed):
    rng = np.random.default_rng(seed)
    return list(_patterns(n, seed).values()) + [rng.integers(0, 65536, n).tolist() for _ in range(3)]


@pytest.mark.parametrize("n", range(1, 10))
def test_run_plan_clear_matches_the_cpp_dry_runs(cbs, plan_lib, n):
    """the Python executor on the C++ plan equals the C++ dry run: result, bootstraps, layers and ladders"""
    plans = {"sum": s8.get_plan(plan_lib, s8.PLAN_SUM, n), "max": s8.get_plan(plan_lib, s8.PLAN_MAX, n)}
    if n % 2 == 0:
        plans["ip"] = s8.get_plan(plan_lib, s8.PLAN_IP, n)
    for k, vals in enumerate(_value_sets(n, 900 + n)):
        for name, plan in plans.items():
            got = _run_clear(plan, vals)
            counts = (sum(len(L.cbs) for L in plan.layers), len(plan.layers), sum(len(L.jobs) for L in plan.layers))
            if name == "sum":
                assert got == sum(vals) % 65536, (n, k, vals)
                continue
            res = (cbs.inner_product_plan_check if name == "ip" else cbs.max_plan_check)(vals)
            assert (got,) + counts == res, (name, n, k, vals, got, counts, res)
            h = n // 2
            want = sum((x * y) % 65536 for x, y in zip(vals[:h], vals[h:])) % 65536 if name == "ip" else max(vals)
            assert got == want, (name, n, vals)


def _trivial_bootstrap(rows):
    """noiseless circuit bootstrap of trivial LWE rows: GGSW level l (l = 1..7) holds bit * 2^(64 - 2 l) on its diagonal,
    GLEV level 1 holds bit * 2^62 in the constant body coefficient"""
    ggsw = np.zeros((len(rows), 7, 3, 3, N), dtype=np.uint64)
    glev = np.zeros((len(rows), 7, 3, N), dtype=np.uint64)
    for k, r in enumerate(rows):
        assert not r[:2 * N].any() and not (r[2 * N] & np.uint64((1 << 63) - 1))
        bit = int(r[2 * N] >> np.uint64(63))
        for lev in range(7):
            for c in range(3):
                ggsw[k, lev, c, c, 0] = bit << (64 - 2 * (lev + 1))
        glev[k, 0, 2, 0] = bit << 62
    return ggsw.reshape(len(rows), -1), glev.reshape(len(rows), -1)


@pytest.mark.parametrize("name,vals", [("sum", [40000, 30001]), ("max", [513, 512])])
def test_run_plan_exact_on_trivial_ciphertexts(plan_lib, pool, name, vals):
    """the exact executor (gathered ladders on the restated accumulators, refreshes, adds) on noiseless trivial ciphertexts
    ends in trivial ciphertexts of the cleartext result"""
    plan = s8.get_plan(plan_lib, s8.PLAN_SUM if name == "sum" else s8.PLAN_MAX, len(vals))
    rows = []
    for b in _clear_rows(vals):
        r = np.zeros(2 * N + 1, dtype=np.uint64)
        r[2 * N] = b << 63
        rows.append(r)
    out = s8.run_plan(plan, rows, _trivial_bootstrap, s8.ExactOps(map=pool.map))
    want = sum(vals) % 65536 if name == "sum" else max(vals)
    for i, r in enumerate(out):
        assert not r[:2 * N].any() and int(r[2 * N]) == ((want >> (15 - i)) & 1) << 63, i
