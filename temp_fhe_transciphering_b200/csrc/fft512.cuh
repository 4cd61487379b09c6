// fft512.cuh — negacyclic FP64 transform for N = 1024 (512 complex points) on a 64-thread group.
//
// B200 design notes
//   * 64 threads (2 warps) own one polynomial; each thread keeps 8 complex points in registers and
//     the 512-point DFT is 3 radix-8 passes (8 x 8 x 8) with two shared-memory transposes through
//     one 8 KB scratch tile.  Transposes are done IN PLACE with an XOR swizzle so every 128-bit
//     shared access is bank-conflict free (quarter-warp = 8 consecutive 16 B slots).
//   * forward = decimation in frequency, inverse = decimation in time, so no bit-reversal pass is
//     ever executed: the Fourier-domain order is "register slot major":
//         value held by thread u (= 8*k1 + k2) in register slot k3  <->  DFT bin k1 + 8*k2 + 64*k3
//     and Fourier polynomials are stored in HBM as F[k3][u] (coalesced 16 B per thread).
//   * the negacyclic twist exp(i*pi*j/N) is folded into pass 1: a compile-time constant
//     c_m = exp(2*pi*i*m/32) on the inputs and a per-thread table T1[k1] = w^t * W512^(t*k1).
//   * all scaling (1/512 of the inverse, 2^64 of the torus) is folded into the Fourier-domain key
//     material, so the inverse ends with: z * conj(T1), IDFT-8, * conj(c_m), round.
//
// The arithmetic mirrors tfhe's fft64 wrapper semantics used by the reference
// (cbs_lib/src/fourier_glwe_keyswitch.rs:301,331; SURVEY.md Appendix A): fold N reals into N/2
// complex, twist, complex DFT with forward sign "-".
//
// Every phase function is __host__ __device__ so tests/test_fft_emulation (CPU) executes the
// very same code by looping over the 64 logical threads between the barrier points.
#pragma once
#ifdef __CUDACC__
#include <cuda_runtime.h>
#endif
#include <stdint.h>

#ifdef __CUDACC__
#define CBS_HD __host__ __device__ __forceinline__
#else
#define CBS_HD inline
#endif

namespace cbs {

constexpr int kN = 1024;          // polynomial size
constexpr int kHalf = 512;        // complex points
constexpr int kGroup = 64;        // threads per polynomial
constexpr double kSqrtHalf = 0.70710678118654752440;

struct cplx {
    double x, y;
};

CBS_HD cplx cmul(cplx a, cplx b) { return {a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x}; }
CBS_HD cplx cmul_conj(cplx a, cplx b) { return {a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y}; }  // a * conj(b)
CBS_HD cplx cadd(cplx a, cplx b) { return {a.x + b.x, a.y + b.y}; }
CBS_HD cplx csub(cplx a, cplx b) { return {a.x - b.x, a.y - b.y}; }
CBS_HD void cfma(cplx &acc, cplx a, cplx b)
{
    acc.x += a.x * b.x;
    acc.x -= a.y * b.y;
    acc.y += a.x * b.y;
    acc.y += a.y * b.x;
}

// c_m = exp(2*pi*i*m/32), m = 0..7  (twist part that depends on the register slot)
#define CBS_CM_RE {1.0, 0.98078528040323044913, 0.92387953251128675613, 0.83146961230254523708, \
                   0.70710678118654752440, 0.55557023301960222474, 0.38268343236508977173, 0.19509032201612826785}
#define CBS_CM_IM {0.0, 0.19509032201612826785, 0.38268343236508977173, 0.55557023301960222474, \
                   0.70710678118654752440, 0.83146961230254523708, 0.92387953251128675613, 0.98078528040323044913}

// 8-point DFT, natural order in and out.  INV = false: W = exp(-2*pi*i/8); true: exp(+2*pi*i/8).
// The two odd eighth roots (+-1 +- i)/sqrt2 are applied WITHOUT their 1/sqrt2 in stage 1; the factor is folded
// into the last stage as fused multiply-adds (8 DFMA replace 8 DADD + 4 DMUL: the FP64 pipe is the unit
// these kernels keep busiest).
template <bool INV>
CBS_HD void dft8(cplx v[8])
{
    // stage 1
    cplx b0 = cadd(v[0], v[4]), b4 = csub(v[0], v[4]);
    cplx b1 = cadd(v[1], v[5]), d1 = csub(v[1], v[5]);
    cplx b2 = cadd(v[2], v[6]), d2 = csub(v[2], v[6]);
    cplx b3 = cadd(v[3], v[7]), d3 = csub(v[3], v[7]);
    cplx b5, b6, b7;  // b5, b7 are sqrt2 times the true values
    if (!INV) {
        b5 = {d1.x + d1.y, d1.y - d1.x};     // * (1 - i)
        b6 = {d2.y, -d2.x};                  // * (-i)
        b7 = {d3.y - d3.x, -(d3.x + d3.y)};  // * (-1 - i)
    } else {
        b5 = {d1.x - d1.y, d1.x + d1.y};     // * (1 + i)
        b6 = {-d2.y, d2.x};                  // * (+i)
        b7 = {-(d3.x + d3.y), d3.x - d3.y};  // * (-1 + i)
    }
    // stage 2 (two 4-point DFTs)
    cplx c0 = cadd(b0, b2), c2 = csub(b0, b2);
    cplx c1 = cadd(b1, b3), e3 = csub(b1, b3);
    cplx c4 = cadd(b4, b6), c6 = csub(b4, b6);
    cplx c5 = cadd(b5, b7), e7 = csub(b5, b7);  // sqrt2 times the true values
    cplx c3, c7;
    if (!INV) {
        c3 = {e3.y, -e3.x};
        c7 = {e7.y, -e7.x};
    } else {
        c3 = {-e3.y, e3.x};
        c7 = {-e7.y, e7.x};
    }
    // stage 3
    v[0] = cadd(c0, c1);
    v[4] = csub(c0, c1);
    v[2] = cadd(c2, c3);
    v[6] = csub(c2, c3);
    v[1] = {c4.x + kSqrtHalf * c5.x, c4.y + kSqrtHalf * c5.y};
    v[5] = {c4.x - kSqrtHalf * c5.x, c4.y - kSqrtHalf * c5.y};
    v[3] = {c6.x + kSqrtHalf * c7.x, c6.y + kSqrtHalf * c7.y};
    v[7] = {c6.x - kSqrtHalf * c7.x, c6.y - kSqrtHalf * c7.y};
}

// physical slot of logical (k1, a, b): position a + 8*b inside block k1, XOR-swizzled
CBS_HD int slot(int k1, int a, int b) { return k1 * 64 + 8 * b + (a ^ b); }

// Per-thread twiddles (loaded once per kernel from the table built by make_twiddle_table()).
struct Twiddles {
    cplx t1[8];  // thread t:            exp(i*pi*t/1024) * exp(-2*pi*i*t*k1/512), k1 = 0..7
    cplx t2[8];  // thread u, t' = u&7:  exp(-2*pi*i*t'*k2/64),                    k2 = 0..7
};

// table layout: [64][8] t1 then [8][8] t2 (complex doubles), then the same two tables of the
// shuffle-exchange variant ("x", see below): [64][8] t1x, [8][8] t2x
constexpr int kTwiddleTableDoubles = (64 * 8 + 8 * 8) * 2 * 2;
constexpr int kTwiddleXOffset = (64 * 8 + 8 * 8) * 2;

CBS_HD void load_twiddles(Twiddles &tw, const double *table, int t)
{
    for (int k = 0; k < 8; k++) {
        tw.t1[k] = {table[(t * 8 + k) * 2], table[(t * 8 + k) * 2 + 1]};
        tw.t2[k] = {table[(512 + (t & 7) * 8 + k) * 2], table[(512 + (t & 7) * 8 + k) * 2 + 1]};
    }
}

// ---------------------------------------------------------------------------------------------
// forward: v[m] holds the folded input point j = t + 64*m as (coef[j], coef[j + 512]).
// fwd_p1 .. [group barrier] .. fwd_p2 .. [group barrier] .. fwd_p3 -> v[k3] = bin(k1+8*k2+64*k3)
CBS_HD void fwd_p1(cplx v[8], cplx *scr, const Twiddles &tw, int t)
{
    const double cr[8] = CBS_CM_RE, ci[8] = CBS_CM_IM;
#pragma unroll
    for (int m = 1; m < 8; m++) v[m] = cmul(v[m], cplx{cr[m], ci[m]});
    dft8<false>(v);
    const int a = t & 7, b = t >> 3;
#pragma unroll
    for (int k1 = 0; k1 < 8; k1++) scr[slot(k1, a, b)] = cmul(v[k1], tw.t1[k1]);
}

CBS_HD void fwd_p2(cplx v[8], cplx *scr, const Twiddles &tw, int t)
{
    const int k1 = t >> 3, tp = t & 7;
#pragma unroll
    for (int mp = 0; mp < 8; mp++) v[mp] = scr[slot(k1, tp, mp)];
    dft8<false>(v);
    scr[slot(k1, tp, 0)] = v[0];
#pragma unroll
    for (int k2 = 1; k2 < 8; k2++) scr[slot(k1, tp, k2)] = cmul(v[k2], tw.t2[k2]);
}

CBS_HD void fwd_p3(cplx v[8], const cplx *scr, int t)
{
    const int k1 = t >> 3, k2 = t & 7;
#pragma unroll
    for (int tp = 0; tp < 8; tp++) v[tp] = scr[slot(k1, tp, k2)];
    dft8<false>(v);
}

// inverse: v[k3] = bin(k1+8*k2+64*k3) for thread u = 8*k1+k2 (unnormalised).
// inv_p3 .. [barrier] .. inv_p2 .. [barrier] .. inv_p1 -> v[m] = (coef[t+64m], coef[t+64m+512])
CBS_HD void inv_p3(cplx v[8], cplx *scr, int t)
{
    const int k1 = t >> 3, k2 = t & 7;
    dft8<true>(v);
#pragma unroll
    for (int tp = 0; tp < 8; tp++) scr[slot(k1, tp, k2)] = v[tp];
}

CBS_HD void inv_p2(cplx v[8], cplx *scr, const Twiddles &tw, int t)
{
    const int k1 = t >> 3, tp = t & 7;
    v[0] = scr[slot(k1, tp, 0)];
#pragma unroll
    for (int k2 = 1; k2 < 8; k2++) v[k2] = cmul_conj(scr[slot(k1, tp, k2)], tw.t2[k2]);
    dft8<true>(v);
#pragma unroll
    for (int mp = 0; mp < 8; mp++) scr[slot(k1, tp, mp)] = v[mp];
}

CBS_HD void inv_p1(cplx v[8], const cplx *scr, const Twiddles &tw, int t)
{
    const double cr[8] = CBS_CM_RE, ci[8] = CBS_CM_IM;
    const int a = t & 7, b = t >> 3;
#pragma unroll
    for (int k1 = 0; k1 < 8; k1++) v[k1] = cmul_conj(scr[slot(k1, a, b)], tw.t1[k1]);
    dft8<true>(v);
#pragma unroll
    for (int m = 1; m < 8; m++) v[m] = cmul_conj(v[m], cplx{cr[m], ci[m]});
}

// ---------------------------------------------------------------------------------------------
// Shuffle-exchange variant ("x").  ncu (profiles/r01_final_ncu_full.csv) shows the FFT kernels bound by the
// shared-memory data pipe (64 % of peak, vs 40 % FP64): a transpose through shared memory moves every
// value twice (STS + LDS).  The transpose between passes 2 and 3 only exchanges values among the 8 lanes
// that share k1 = t >> 3, so it is done with 7 rounds of width-8 warp shuffles instead (each value moves
// once, no barrier).  Round r moves register r of lane a to lane (a + r) & 7; for the register indices to
// be compile-time constants the pass-2 outputs must sit in rotated order (register r = output (a + r) & 7)
// and the pass-3 inputs arrive in the order tp = (b - r) & 7.  Both rotations are free:
//   * a rotation of DFT outputs = a modulation of its inputs, folded into the pass-1 twiddle table
//     (t1x[t][k1] = t1[t][k1] * W8^((t>>3)*(t&7))); the pass-2 twiddles are stored rotated (t2x);
//   * a reversed+rotated input order of pass 3 = the conjugate-direction DFT-8 followed by a per-lane phase
//     W8^(b*k3) on the spectrum.  The phase is NOT applied: the forward transform yields conj(phi) * X,
//     the pointwise products with TRUE key spectra yield conj(phi) * OUT, and the mirrored inverse
//     consumes exactly conj(phi) * OUT.  Key material therefore keeps the layout and values of the plain
//     transform (keys are converted with fwd_p1..p3 above).
// The exchange itself is a template on the lane-exchange functor so tests/cpu_emul executes the same
// phase code with an emulated shuffle.
CBS_HD void load_twiddles_x(Twiddles &tw, const double *table, int t) { load_twiddles(tw, table + kTwiddleXOffset, t); }

// pass 2 of the forward transform: on return v[r] = Z[k1][k2 = (a + r) & 7][tp = a], a = t & 7
CBS_HD void fwd_p2x(cplx v[8], const cplx *scr, const Twiddles &tw, int t)
{
    const int k1 = t >> 3, tp = t & 7;
#pragma unroll
    for (int mp = 0; mp < 8; mp++) v[mp] = scr[slot(k1, tp, mp)];
    dft8<false>(v);
#pragma unroll
    for (int r = 0; r < 8; r++) v[r] = cmul(v[r], tw.t2[r]);
}
// [exchange fwd: v[r] <- lane (a - r) & 7's v[r], r = 1..7]  then pass 3:
CBS_HD void fwd_p3x(cplx v[8]) { dft8<true>(v); }

// inverse: pass 3, [exchange inv: v[r] <- lane (a + r) & 7's v[r]], pass 2 into the transpose tile
CBS_HD void inv_p3x(cplx v[8]) { dft8<false>(v); }
CBS_HD void inv_p2x(cplx v[8], cplx *scr, const Twiddles &tw, int t)
{
    const int k1 = t >> 3, tp = t & 7;
#pragma unroll
    for (int r = 0; r < 8; r++) v[r] = cmul_conj(v[r], tw.t2[r]);
    dft8<true>(v);
#pragma unroll
    for (int mp = 0; mp < 8; mp++) scr[slot(k1, tp, mp)] = v[mp];
}

#ifdef __CUDACC__
// width-8 lane exchange of registers 1..7 (28 SHFL.IDX); dir = -1 forward, +1 inverse
template <int DIR>
__device__ __forceinline__ void exchange8(cplx v[8], int a)
{
#pragma unroll
    for (int r = 1; r < 8; r++) {
        const int src = (a + DIR * r) & 7;
        v[r].x = __shfl_sync(0xffffffffu, v[r].x, src, 8);
        v[r].y = __shfl_sync(0xffffffffu, v[r].y, src, 8);
    }
}
#endif

// ---------------------------------------------------------------------------------------------
// integer <-> double helpers

// signed balanced digits, finest level first (tfhe SignedDecomposer; SURVEY.md Appendix A).
// state after closest_representable, already shifted down to base_log*level bits.
CBS_HD uint64_t decomp_init(uint64_t x, int base_log, int level)
{
    const int nr = 64 - base_log * level;
    return (x >> nr) + ((x >> (nr - 1)) & 1ull);
}
CBS_HD int32_t decomp_next(uint64_t &st, int base_log)
{
    const uint64_t mask = (1ull << base_log) - 1ull;
    uint64_t res = st & mask;
    st >>= base_log;
    uint64_t carry = (((res - 1ull) | st) & res) >> (base_log - 1);
    st += carry;
    return (int32_t)(uint32_t)(res - (carry << base_log));
}

// tfhe SignedDecomposer(base_log 23, level 1) digit of a 64-bit word from its high 32 bits alone:
//   s = ((hi >> 8) + 1) >> 1, digit = s - (s > 2^22 ? 2^23 : 0)  ==  (((int32)(hi - 0x100)) >> 9) + 1
CBS_HD int32_t digit_b23_l1_hi(uint32_t hi) { return (((int32_t)(hi - 0x100u)) >> 9) + 1; }

// exact int32 -> double without the conversion pipe (|x| < 2^31)
CBS_HD double i32_to_double(int32_t x)
{
#ifdef __CUDA_ARCH__
    return __hiloint2double(0x43300000, (int)((uint32_t)x ^ 0x80000000u)) - 4503601774854144.0;  // 2^52 + 2^31
#else
    return (double)x;
#endif
}

// Inverse-FFT output -> torus word.  `r` already carries the 2^64 scale (folded into the key's
// Fourier data), so: reduce modulo 2^64 to the nearest multiple (magic add, exact), then one
// round-to-nearest conversion.  Same value as tfhe's from_torus(frac) * 2^64 rounding, except at
// r = 2^63 mod 2^65: the tie of the reduction goes to the even multiple, f = +2^63, and the
// conversion saturates to 2^63 - 1 where tfhe gives 2^63 (one unit of 2^-64, DESIGN.md section 2;
// the exact fix costs 123 instructions per blind-rotation step).  The host branch does the same.
CBS_HD uint64_t torus_from_scaled(double r)
{
    const double M = 124615124604835863084731911901282304.0;  // 1.5 * 2^116: ulp = 2^64
    double k = (r + M) - M;
    double f = r - k;  // in [-2^63, 2^63], exact
#ifdef __CUDA_ARCH__
    return (uint64_t)__double2ll_rn(f);
#else
    if (f >= 9223372036854775808.0) return 0x7FFFFFFFFFFFFFFFull;
    double rr = __builtin_nearbyint(f);
    return (uint64_t)(int64_t)rr;
#endif
}

// u64 torus word -> double "as signed integer" (tfhe forward_as_torus without the 2^-64)
CBS_HD double torus_to_double(uint64_t x) { return (double)(int64_t)x; }

}  // namespace cbs
