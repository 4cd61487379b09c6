"""Exact integer reference of stage 8: the max_of_two CMux ladder, the gathered LUT ladder, their integer glue and the
executor of the LUT-circuit plans (test helper, not a conftest).

Built from the exact ring operations of tests/exact_ref.py (wrapping uint64, no floating point), so with small GGSW the
GPU must equal it bit for bit and with real GGSW the difference is the FP64 error of the kernels.  The plans come from
csrc/host/ip_plan.h itself through the ctypes shim tests/plan_dump.cpp (build_plan_lib); the LUT tables and accumulators
are restated here from their definition, not read out of the library.
"""
import ctypes
import os
import subprocess
from collections import namedtuple

import numpy as np

from exact_ref import N, U64, external_product, lut_cmux, sample_extract, u64

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LWE_BIG = 2 * N + 1
BASE_LOG, LEVEL = 2, 7  # the stage-8 GGSW (circuit bootstrap output)
PLAN_IP, PLAN_SUM, PLAN_MAX = 0, 1, 2


# ---- max_of_two ----------------------------------------------------------------------------------------------------

def _ext(ggsw, diff):
    return external_product(u64(ggsw).reshape(LEVEL, 3, 3, N), diff, BASE_LOG, LEVEL)


def max_of_two_bit(ga16, gb16, op_a, op_b, e0="a"):
    """output bit j of max_of_two for operands op_a = op_a16[j], op_b = op_b16[j] ([3][N] GLWE) -> [2049].
    for i = 15..0: m0 = e + Gb[i] (x) (op_b - e); m1 = op_a + Gb[i] (x) (e - op_a); e = m0 + Ga[i] (x) (m1 - m0).
    e0 = "a": e starts from op_a (the GPU, DESIGN.md section 4a); "zero": from 0 (the oracle's reset_e=1)."""
    ga16, gb16 = u64(ga16).reshape(16, -1), u64(gb16).reshape(16, -1)
    a, b = u64(op_a).reshape(3, N), u64(op_b).reshape(3, N)
    e = a.copy() if e0 == "a" else np.zeros((3, N), dtype=np.uint64)
    with np.errstate(over="ignore"):
        for i in range(15, -1, -1):
            m0 = e + _ext(gb16[i], b - e)
            m1 = a + _ext(gb16[i], e - a)
            e = m0 + _ext(ga16[i], m1 - m0)
    return sample_extract(e, 2, N, 0)


def max_of_two(ggsw_a16, ggsw_b16, op_a16, op_b16, e0="a", bits=range(16)):
    """max_of_two of two values (GGSW [16] MSB first, operands [16][3N]) -> the LWE of each output bit in `bits`."""
    oa, ob = u64(op_a16).reshape(16, -1), u64(op_b16).reshape(16, -1)
    return np.stack([max_of_two_bit(ggsw_a16, ggsw_b16, oa[j], ob[j], e0) for j in bits])


# ---- gathered LUT ladder and the integer glue -------------------------------------------------------------------------

def lut8_gather(ggsw, sel8, lut):
    """one CMux (exact_ref.lut_cmux, rotation 2^i) per selector sel8[i] >= 0 with ggsw[sel8[i]], none for -1; then the 4
    extractions at 0, 256, 512, 768 -> [4][2049]"""
    acc = u64(lut).reshape(3, N)
    for i, s in enumerate(sel8):
        if s >= 0:
            acc = lut_cmux(acc, ggsw[s], i)
    return np.stack([sample_extract(acc, 2, N, 256 * t) for t in range(4)])


def glev_to_operand(glev):
    """2 x GLEV index 0 (level 1: bit * 2^62 after the trace) -> GLWE [3N] encrypting bit * 2^63"""
    with np.errstate(over="ignore"):
        return u64(glev).reshape(LEVEL, 3 * N)[0] * U64(2)


def glev_to_lwe(glev):
    return sample_extract(glev_to_operand(glev), 2, N, 0)


def ip_lut_value(lut, idx):
    """the LUT tables of csrc/host/ip_plan.h restated: 0 nibble product, 1 population count, 2 nibble sum, 3 nibble
    compare (bit 0: a > b, bit 1: a == b; a = idx & 15, b = idx >> 4), 4 select (d AND [a > b] from the compare bits)"""
    a, b = idx & 15, idx >> 4
    if lut == 0:
        return a * b
    if lut == 1:
        return bin(idx).count("1")
    if lut == 2:
        return a + b
    if lut == 3:
        return int(a > b) | (2 if a == b else 0)
    gt0, gt1, eq1, gt2, eq2, gt3, eq3, d = ((idx >> k) & 1 for k in range(8))
    return d & (gt3 | (eq3 & (gt2 | (eq2 & (gt1 | (eq1 & gt0))))))


NUM_LUTS = 5


def lut_accumulators():
    """[NUM_LUTS * 2][3N] trivial GLWE, index 2 lut + acc: body coefficient i = bit 4 acc + i // 256 of
    ip_lut_value(lut, i % 256), at 2^63"""
    out = np.zeros((NUM_LUTS * 2, 3, N), dtype=np.uint64)
    for lut in range(NUM_LUTS):
        for acc in range(2):
            out[2 * lut + acc, 2] = [((ip_lut_value(lut, i % 256) >> (4 * acc + i // 256)) & 1) << 63 for i in range(N)]
    return out.reshape(NUM_LUTS * 2, 3 * N)


# ---- the circuit plans (csrc/host/ip_plan.h through tests/plan_dump.cpp) ----------------------------------------------

Plan = namedtuple("Plan", "nvals pool_size nin_bits result layers")
Layer = namedtuple("Layer", "pre cbs refresh jobs post")  # jobs: (sel[8], lut, acc, out)


def build_plan_lib(outdir):
    so = os.path.join(str(outdir), "libplan_dump.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-I",
                           os.path.join(ROOT, "temp_fhe_transciphering_b200", "csrc", "host"),
                           os.path.join(ROOT, "tests", "plan_dump.cpp"), "-o", so])
    lib = ctypes.CDLL(so)
    lib.plan_lut_value.restype = ctypes.c_uint
    return lib


def get_plan(lib, kind, nvals):
    n = lib.plan_dump(kind, nvals, None, 0)
    assert n > 0, (kind, nvals, n)
    buf = (ctypes.c_int * n)()
    assert lib.plan_dump(kind, nvals, buf, n) == n
    v = list(buf)
    pos = 0

    def take(k):
        nonlocal pos
        pos += k
        return v[pos - k:pos]

    def groups(width):
        cnt = take(1)[0]
        return [tuple(take(width)) for _ in range(cnt)]

    nv, pool_size, nin_bits, nlayers = take(4)
    result = take(16)
    layers = []
    for _ in range(nlayers):
        pre = groups(3)
        cbs = take(take(1)[0])
        refresh = groups(2)
        jobs = [(j[:8], j[8], j[9], j[10]) for j in groups(11)]
        layers.append(Layer(pre, cbs, refresh, jobs, groups(3)))
    assert pos == n
    return Plan(nv, pool_size, nin_bits, result, layers)


# ---- the executor of run_lut_plan -----------------------------------------------------------------------------------

class ExactOps:
    """Ciphertext operations of the executor: LWE rows [2049], exact gathered ladders on the restated accumulators.
    `map` evaluates the ladders of a layer (e.g. a process pool's map); each task carries only the GGSWs it uses."""

    def __init__(self, map=map):
        self.map = map
        self.luts = lut_accumulators()

    @staticmethod
    def zero():
        return np.zeros(LWE_BIG, dtype=np.uint64)

    @staticmethod
    def add(a, b):
        with np.errstate(over="ignore"):
            return u64(a) + u64(b)

    @staticmethod
    def refresh(glev):
        return glev_to_lwe(glev)

    def ladders(self, ggsw, jobs):
        tasks = []
        for sel, lut, acc in jobs:
            used = sorted({s for s in sel if s >= 0})
            tasks.append(([u64(ggsw[s]) for s in used], [used.index(s) if s >= 0 else -1 for s in sel],
                          self.luts[2 * lut + acc]))
        return list(self.map(lut8_gather, *zip(*tasks))) if tasks else []


class ClearOps:
    """The same executor on cleartext bits: a bootstrap returns the bit itself as both GGSW and GLEV."""

    @staticmethod
    def zero():
        return 0

    @staticmethod
    def add(a, b):
        return a ^ b

    @staticmethod
    def refresh(glev):
        return glev

    @staticmethod
    def ladders(ggsw, jobs):
        out = []
        for sel, lut, acc in jobs:
            idx = sum(ggsw[s] << i for i, s in enumerate(sel) if s >= 0)
            val = ip_lut_value(lut, idx) >> (4 * acc)
            out.append([(val >> q) & 1 for q in range(4)])
        return out


def run_plan(plan, rows, bootstrap, ops=None):
    """run_lut_plan's executor: per layer the pre-adds, bootstrap(rows of layer.cbs) -> (GGSW, GLEV) per row, the refreshes
    pool[dst] = glev_to_lwe(GLEV[pos]), the gathered ladders into the pool, the post-adds; then result[15..0] (MSB first,
    -1: a zero row).  rows: the plan.nin_bits input rows ([value][bit MSB first])."""
    ops = ops or ExactOps()
    pool = [None] * plan.pool_size
    assert len(rows) == plan.nin_bits
    pool[:plan.nin_bits] = list(rows)
    for L in plan.layers:
        for dst, a, b in L.pre:
            pool[dst] = ops.add(pool[a], pool[b])
        ggsw, glev = bootstrap([pool[i] for i in L.cbs])
        for p, dst in L.refresh:
            pool[dst] = ops.refresh(glev[p])
        outs = ops.ladders(ggsw, [(sel, lut, acc) for sel, lut, acc, _ in L.jobs])
        for (_, _, _, o), rows4 in zip(L.jobs, outs):
            pool[o:o + 4] = list(rows4)
        for dst, a, b in L.post:
            pool[dst] = ops.add(pool[a], pool[b])
    return [pool[plan.result[15 - i]] if plan.result[15 - i] >= 0 else ops.zero() for i in range(16)]
