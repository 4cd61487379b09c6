"""Exact integer reference of LWE-to-GLWE packing (test helper, not a conftest).

A direct restatement of the semantics cbs_pack_lwes implements, built from the exact ring operations and the exact GLWE
keyswitch of tests/exact_ref.py (wrapping uint64, no floating point).  With small keys the GPU must equal it bit for
bit; with real keys the difference is the FP64 error of the kernel.
"""
import numpy as np

from exact_ref import N, U64, const_embed, eval_x_k, glwe_keyswitch, mono_mul, u64


def pack_lwes(auto_std, lwes):
    """LWE-to-GLWE packing (Chen-Dai-Kim-Song 2020): big LWE i [2049] -> coefficient i % 1024 of GLWE i // 1024.
    Level 0: p[j] = const_embed(lwe_j >> 10) (the zero GLWE for a missing slot).  Level L = 1..10, stride s = 1024 >> L,
    kappa = 2^L + 1 = the automorphism of auto_std[10 - L]: q[t] = (e + X^s o) + keyswitch(eval_x_k(e - X^s o, kappa)) with
    e = p[t], o = p[t + s], for t < s.  After level 10 item 0 is the packed GLWE.  -> [ceil(count / 1024)][3072]"""
    lwes = u64(lwes).reshape(-1, 2 * N + 1)
    out = []
    with np.errstate(over="ignore"):
        for g0 in range(0, len(lwes), N):
            grp = lwes[g0:g0 + N]
            p = [const_embed(x >> U64(10), 2, N) for x in grp] + [np.zeros(3 * N, dtype=np.uint64)] * (N - len(grp))
            for L in range(1, 11):
                s = N >> L
                q = []
                for t in range(s):
                    xo = mono_mul(p[t + s].reshape(3, N), s).reshape(-1)
                    pw = eval_x_k((p[t] - xo).reshape(3, N), (1 << L) + 1)
                    q.append(p[t] + xo + glwe_keyswitch(u64(auto_std)[10 - L], pw, 13, 3))
                p = q
            out.append(p[0])
    return np.stack(out)
