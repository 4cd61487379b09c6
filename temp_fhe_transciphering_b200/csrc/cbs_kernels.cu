// cbs_kernels.cu — hand-written sm_100a kernels of the circuit-bootstrapping AES transciphering path.
//
// Each kernel states the reference routine it replaces (paths relative to
// /root/reference/submission/).  Work decomposition common to the FFT kernels: a GROUP of 64
// threads (2 warps) owns one GLWE ciphertext / accumulator; the ciphertext lives in shared memory
// as u64, polynomials are transformed with the 3-pass radix-8 FP64 FFT of fft512.cuh, Fourier-domain
// key material is streamed from L2/HBM with coalesced 16-byte loads (512 B per warp instruction) and
// the pointwise multiply-accumulate, inverse transform and torus rounding never leave registers.
// Groups synchronise with named barriers (bar.sync id, 64), never with __syncthreads, so the groups
// of a CTA drift freely and hide each other's shared-memory and barrier latency.
#include "cbs_kernels.cuh"
#include "chacha20.h"
#include "digits.cuh"
#include "fft512.cuh"
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <mutex>

namespace cbs {

// ------------------------------------------------------------------------------------------------
// group plumbing
struct Group {
    int t;       // thread index inside the group, 0..63
    int bar;     // named barrier id (1..15)
    cplx *scr0;  // two 8 KB transpose tiles used alternately: no WAR barrier between transforms
    cplx *scr1;
    int flip;
};

__device__ __forceinline__ void group_sync(int bar) { asm volatile("bar.sync %0, 64;" ::"r"(bar) : "memory"); }

__device__ __forceinline__ void fwd_fft(cplx v[8], Group &g, const Twiddles &tw)
{
    cplx *s = g.flip ? g.scr1 : g.scr0;
    g.flip ^= 1;
    fwd_p1(v, s, tw, g.t);
    group_sync(g.bar);
    fwd_p2(v, s, tw, g.t);
    group_sync(g.bar);
    fwd_p3(v, s, g.t);
}

__device__ __forceinline__ void inv_fft(cplx v[8], Group &g, const Twiddles &tw)
{
    cplx *s = g.flip ? g.scr1 : g.scr0;
    g.flip ^= 1;
    inv_p3(v, s, g.t);
    group_sync(g.bar);
    inv_p2(v, s, tw, g.t);
    group_sync(g.bar);
    inv_p1(v, s, tw, g.t);
}

// coefficient e (0..2047) of the negacyclic extension of p: p[e] for e < N, -p[e-N] otherwise
__device__ __forceinline__ uint64_t neg_read(const uint64_t *p, int e)
{
    uint64_t x = p[e & 1023];
    return (e & 1024) ? (0ull - x) : x;
}

__device__ __forceinline__ cplx ldg_cplx(const double *p)
{
    double2 d = __ldg(reinterpret_cast<const double2 *>(p));
    return cplx{d.x, d.y};
}

// out[c][k3] += v[k3] * key_c[k3*64 + t]   for c < NOUT; key polys are consecutive Fourier polys
template <int NOUT>
__device__ __forceinline__ void mul_acc(cplx (&out)[NOUT][8], const cplx v[8], const double *key, int t)
{
#pragma unroll
    for (int c = 0; c < NOUT; c++) {
#pragma unroll
        for (int k3 = 0; k3 < 8; k3++) {
            cplx w = ldg_cplx(key + (size_t)c * kFourierPolyDoubles + (size_t)(k3 * 64 + t) * 2);
            cfma(out[c][k3], v[k3], w);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K0: standard -> Fourier conversion (tfhe convert_standard_*_to_fourier; call sites
// src/bin/server_encrypted_aes_decryption.rs:646-687; split limbs
// cbs_lib/src/fourier_glwe_keyswitch.rs:188-199)
constexpr int kConvGroups = 4;
__global__ void __launch_bounds__(64 * kConvGroups) k_std_to_fourier(const uint64_t *__restrict__ in,
                                                                      double *__restrict__ out, int npoly, int mode,
                                                                      int split, const double *__restrict__ twtab)
{
    __shared__ cplx scr[kConvGroups][512];
    Group g;
    g.t = threadIdx.x & 63;
    const int gi = threadIdx.x >> 6;
    g.bar = 1 + gi;
    g.scr0 = g.scr1 = scr[gi];
    g.flip = 0;
    const int poly = blockIdx.x * kConvGroups + gi;
    if (poly >= npoly) return;
    Twiddles tw;
    load_twiddles(tw, twtab, g.t);
    const uint64_t *p = in + (size_t)poly * 1024;
    cplx v[8];
#pragma unroll
    for (int m = 0; m < 8; m++) {
        uint64_t lo = p[g.t + 64 * m], hi = p[g.t + 64 * m + 512];
        if (mode == 1) {
            lo = (lo << (64 - split)) >> (64 - split);
            hi = (hi << (64 - split)) >> (64 - split);
        } else if (mode == 2) {
            lo >>= split;
            hi >>= split;
        }
        v[m] = cplx{torus_to_double(lo), torus_to_double(hi)};
    }
    fwd_fft(v, g, tw);
    double *o = out + (size_t)poly * kFourierPolyDoubles;
#pragma unroll
    for (int k3 = 0; k3 < 8; k3++) {
        double2 w = make_double2(v[k3].x * (1.0 / 512.0), v[k3].y * (1.0 / 512.0));
        *reinterpret_cast<double2 *>(o + (size_t)(k3 * 64 + g.t) * 2) = w;
    }
}

void launch_std_to_fourier(const uint64_t *in, double *out, int npoly, int mode, int split, const double *tw,
                           cudaStream_t s)
{
    if (npoly <= 0) return;
    k_std_to_fourier<<<(npoly + kConvGroups - 1) / kConvGroups, 64 * kConvGroups, 0, s>>>(in, out, npoly, mode, split, tw);
}

// ------------------------------------------------------------------------------------------------
// 128-point transform for the keyswitch ring N' = 256 as two register passes over shared memory:
//   A : radix 8 over the stride-16 points n = j + 16 m of a thread j < 16, twiddle W128^(j k), output y_k[j]
//   BC: radix 16 over the 16 contiguous values y_k[0..15] of a thread k < 8 (two DFT-8 + one butterfly level)
// X[k + 8 g] = sum_j W16^(j g) W128^(j k) sum_m x[j + 16 m] W8^(m k) ends up at position ks_pos(k, g); the inverse mirrors
// it (unnormalised; the key carries the 1/128).  Positions are XOR-swizzled inside each block of 16 so that both passes
// read and write shared memory without bank conflicts; data and key use the same order, so pointwise products do not care.
// (Round 1 ran seven radix-2 shared-memory stages: 14 CTA barriers per keyswitch, shared-memory pipe 65 % with 3.1 M bank
// conflicts, 42 us per 512 ciphertexts.)  tw128 layout: [128] twist exp(i*pi*j/256), then [64] w = exp(-2*pi*i*j/128).
constexpr int kKsThreads = 256;
constexpr int kKsCt = 2;  // ciphertexts per CTA: they share every key value fetched from L2

__device__ __forceinline__ int ks_pos(int k, int j) { return 16 * k + (j ^ k); }
__device__ __forceinline__ cplx ks_w128(const cplx *w, int e)  // exp(-2*pi*i*e/128), 0 <= e < 128
{
    const cplx r = w[e & 63];
    return (e & 64) ? cplx{-r.x, -r.y} : r;
}
__device__ __forceinline__ void ks_fwd_a(cplx v[8], cplx *F, int j, const cplx *w)
{
    dft8<false>(v);
    F[ks_pos(0, j)] = v[0];
#pragma unroll
    for (int k = 1; k < 8; k++) F[ks_pos(k, j)] = cmul(v[k], ks_w128(w, j * k));
}
__device__ __forceinline__ void ks_fwd_bc(cplx *F, int k, const cplx *w)
{
    cplx e[8], o[8];
#pragma unroll
    for (int a = 0; a < 8; a++) {
        e[a] = F[ks_pos(k, 2 * a)];
        o[a] = F[ks_pos(k, 2 * a + 1)];
    }
    dft8<false>(e);
    dft8<false>(o);
#pragma unroll
    for (int g = 0; g < 8; g++) {
        const cplx t = g ? cmul(o[g], w[8 * g]) : o[0];
        F[ks_pos(k, g)] = cadd(e[g], t);
        F[ks_pos(k, g + 8)] = csub(e[g], t);
    }
}
__device__ __forceinline__ void ks_inv_bc(cplx *F, int k, const cplx *w)
{
    cplx e[8], o[8];
#pragma unroll
    for (int g = 0; g < 8; g++) {
        const cplx z0 = F[ks_pos(k, g)], z1 = F[ks_pos(k, g + 8)];
        e[g] = cadd(z0, z1);
        o[g] = g ? cmul_conj(csub(z0, z1), w[8 * g]) : csub(z0, z1);
    }
    dft8<true>(e);
    dft8<true>(o);
#pragma unroll
    for (int a = 0; a < 8; a++) {
        F[ks_pos(k, 2 * a)] = e[a];
        F[ks_pos(k, 2 * a + 1)] = o[a];
    }
}
__device__ __forceinline__ void ks_inv_a(cplx v[8], const cplx *F, int j, const cplx *w)
{
    v[0] = F[ks_pos(0, j)];
#pragma unroll
    for (int k = 1; k < 8; k++) v[k] = cmul_conj(F[ks_pos(k, j)], ks_w128(w, j * k));
    dft8<true>(v);  // v[m] = 128 x[j + 16 m]
}

// key polynomial -> Fourier, in the position order of the passes above, scaled by 1/128
__global__ void __launch_bounds__(128) k_ksk_to_fourier(const uint64_t *__restrict__ in, double *__restrict__ out, int npoly,
                                                         const double *__restrict__ tw128)
{
    __shared__ __align__(16) cplx data[128];
    __shared__ __align__(16) cplx w[64];
    const int poly = blockIdx.x;
    if (poly >= npoly) return;
    for (int i = threadIdx.x; i < 64; i += 128) w[i] = cplx{tw128[256 + 2 * i], tw128[256 + 2 * i + 1]};
    __syncthreads();
    const uint64_t *p = in + (size_t)poly * 256;
    if (threadIdx.x < 16) {
        const int j = threadIdx.x;
        cplx v[8];
#pragma unroll
        for (int m = 0; m < 8; m++) {
            const int n = j + 16 * m;
            v[m] = cmul(cplx{torus_to_double(p[n]), torus_to_double(p[n + 128])}, cplx{tw128[2 * n], tw128[2 * n + 1]});
        }
        ks_fwd_a(v, data, j, w);
    }
    __syncthreads();
    if (threadIdx.x < 8) ks_fwd_bc(data, threadIdx.x, w);
    __syncthreads();
    const int q = threadIdx.x;
    out[((size_t)poly * 128 + q) * 2] = data[q].x * (1.0 / 128.0);
    out[((size_t)poly * 128 + q) * 2 + 1] = data[q].y * (1.0 / 128.0);
}

void launch_ksk_to_fourier(const uint64_t *in, double *out, int npoly, const double *tw128, cudaStream_t s)
{
    k_ksk_to_fourier<<<npoly, 128, 0, s>>>(in, out, npoly, tw128);
}

// ------------------------------------------------------------------------------------------------
// K2: keyswitch_lwe_ciphertext_by_glwe_keyswitch, cbs_lib/src/fourier_glwe_keyswitch.rs:344-379
// (convert_lwe_to_glwe_const glwe_conv.rs:12-44 -> keyswitch_glwe_ciphertext :213-342, Vanilla FFT,
// B = 2^4, l = 3, ring N' = 256 -> sample extract 0).  Two ciphertexts per CTA, 3 CTA barriers per keyswitch:
//   1. thread (ciphertext, input poly i, j): loads its 16 coefficients of the const-embedded input, decomposes them,
//      and runs pass A of the three digit polynomials straight from registers;
//   2. pass BC of the 48 digit polynomials (384 sixteen-point jobs);
//   3. thread (ciphertext, position): the 24 x 4 products against the Fourier key - every key value fetched from L2
//      serves both ciphertexts of the CTA (round 1: one ciphertext per CTA, 196 KB of key per ciphertext);
//   4. inverse passes of the 8 output polynomials, untwist, torus rounding, sample extraction.
constexpr int kKsSmemBytes = (kKsCt * 24 * 128 + 128 + 64) * (int)sizeof(cplx);

__global__ void __launch_bounds__(kKsThreads) k_lwe_keyswitch(const uint64_t *__restrict__ in,
                                                               uint64_t *__restrict__ out, int count,
                                                               const double *__restrict__ ksk_f,
                                                               const double *__restrict__ tw128)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cplx *F = reinterpret_cast<cplx *>(smem_raw);  // [ciphertext][24][128]
    cplx *twist = F + kKsCt * 24 * 128;
    cplx *w = twist + 128;
    const int ct0 = blockIdx.x * kKsCt;
    for (int i = threadIdx.x; i < 128; i += kKsThreads) twist[i] = cplx{tw128[2 * i], tw128[2 * i + 1]};
    for (int i = threadIdx.x; i < 64; i += kKsThreads) w[i] = cplx{tw128[256 + 2 * i], tw128[256 + 2 * i + 1]};
    __syncthreads();
    // 1. digits of the const-embedded input (g[0] = a[0], g[n] = -a[256 - n]), folded + twisted, pass A
    {
        const int c = threadIdx.x >> 7, i = (threadIdx.x >> 4) & 7, j = threadIdx.x & 15;
        if (ct0 + c < count) {
            const uint64_t *a = in + (size_t)(ct0 + c) * kLweBig + i * 256;
            uint64_t sl[8], sh[8];
#pragma unroll
            for (int m = 0; m < 8; m++) {
                const int n = j + 16 * m;
                const uint64_t lo = (n == 0) ? a[0] : (0ull - a[256 - n]);
                const uint64_t hi = 0ull - a[128 - n];  // coefficient n + 128
                sl[m] = decomp_init(lo, 4, 3);
                sh[m] = decomp_init(hi, 4, 3);
            }
#pragma unroll
            for (int tt = 0; tt < 3; tt++) {
                cplx v[8];
#pragma unroll
                for (int m = 0; m < 8; m++) {
                    const double dl = (double)decomp_next(sl[m], 4), dh = (double)decomp_next(sh[m], 4);
                    v[m] = cmul(cplx{dl, dh}, twist[j + 16 * m]);
                }
                ks_fwd_a(v, F + (c * 24 + i * 3 + tt) * 128, j, w);
            }
        }
    }
    __syncthreads();
    // 2. pass BC of every digit polynomial
    for (int id = threadIdx.x; id < kKsCt * 24 * 8; id += kKsThreads) {
        const int poly = id >> 3, k = id & 7;
        if (ct0 + poly / 24 < count) ks_fwd_bc(F + poly * 128, k, w);
    }
    __syncthreads();
    // 3. products: thread (ciphertext c, position q), 4 output polynomials
    cplx acc[4];
    {
        const int c = threadIdx.x >> 7, q = threadIdx.x & 127;
#pragma unroll
        for (int o = 0; o < 4; o++) acc[o] = cplx{0.0, 0.0};
        if (ct0 + c < count) {
            const cplx *Fc = F + c * 24 * 128 + q;
#pragma unroll 2
            for (int i = 0; i < 8; i++) {  // 24 key loads (L2) in flight per thread
#pragma unroll
                for (int tt = 0; tt < 3; tt++) {
                    const int lev = 2 - tt;
                    const cplx f = Fc[(i * 3 + tt) * 128];
                    const double *kp = ksk_f + ((size_t)((i * 3 + lev) * 4) * 128 + q) * 2;
#pragma unroll
                    for (int o = 0; o < 4; o++) cfma(acc[o], f, ldg_cplx(kp + (size_t)o * 256));
                }
            }
        }
    }
    __syncthreads();
    {
        const int c = threadIdx.x >> 7, q = threadIdx.x & 127;
#pragma unroll
        for (int o = 0; o < 4; o++) F[(c * 24 + o) * 128 + q] = acc[o];  // output polynomial o of ciphertext c
    }
    __syncthreads();
    // 4. inverse passes, untwist, round to the torus, sample-extract coefficient 0
    if (threadIdx.x < kKsCt * 4 * 8) {
        const int c = threadIdx.x >> 5, o = (threadIdx.x >> 3) & 3, k = threadIdx.x & 7;
        if (ct0 + c < count) ks_inv_bc(F + (c * 24 + o) * 128, k, w);
    }
    __syncthreads();
    if (threadIdx.x < kKsCt * 4 * 16) {
        const int c = threadIdx.x >> 6, o = (threadIdx.x >> 4) & 3, j = threadIdx.x & 15;
        if (ct0 + c < count) {
            cplx v[8];
            ks_inv_a(v, F + (c * 24 + o) * 128, j, w);
            uint64_t *dst = out + (size_t)(ct0 + c) * kLweSmall;
#pragma unroll
            for (int m = 0; m < 8; m++) {
                const int n = j + 16 * m;
                const cplx z = cmul_conj(v[m], twist[n]);
                const uint64_t lo = torus_from_scaled(z.x), hi = torus_from_scaled(z.y);
                if (o < 3) {
                    // lwe[o*256 + x] = m[0] for x = 0, -m[256 - x] otherwise
                    if (n == 0) dst[o * 256] = lo;
                    else dst[o * 256 + 256 - n] = 0ull - lo;
                    dst[o * 256 + 128 - n] = 0ull - hi;
                } else if (n == 0) {
                    dst[kLweN] = lo + in[(size_t)(ct0 + c) * kLweBig + kBigN];
                }
            }
        }
    }
}

void launch_lwe_keyswitch(const DeviceKeys &K, const uint64_t *in, uint64_t *out, int count, cudaStream_t s)
{
    if (count <= 0) return;
    static bool attr_done[64] = {false};
    int attr_dev = 0;
    cudaGetDevice(&attr_dev);
    bool &attr = attr_done[attr_dev & 63];
    if (!attr) {
        cudaFuncSetAttribute(k_lwe_keyswitch, cudaFuncAttributeMaxDynamicSharedMemorySize, kKsSmemBytes);
        attr = true;
    }
    k_lwe_keyswitch<<<(count + kKsCt - 1) / kKsCt, kKsThreads, kKsSmemBytes, s>>>(in, out, count, K.ksk_f, K.tw128);
}

// ------------------------------------------------------------------------------------------------
// K1: blind rotation.  Accumulator construction cbs_lib/src/ggsw_conv.rs:250-268 and
// gen_blind_rotate_local_assign cbs_lib/src/pbs.rs:70-161 (fast_pbs_modulus_switch with
// LutCountLog(3); polynomial_wrapping_monic_monomial_mul_and_subtract utils.rs:503-568; tfhe
// add_external_product_assign with B = 2^23, l = 1).
//
// One group per LWE ciphertext, kBrGroups groups per CTA, 1 CTA per SM.  Per step:
//   3 x [rotate-subtract + decompose + forward FFT]  ->  9 pointwise MACs against BSK_i  ->
//   3 x [inverse FFT + torus rounding + accumulate].
constexpr int kBrGroups = 4;

__device__ __forceinline__ int modswitch_dev(uint64_t x)
{
    // ((x >> (64 - log2N - 2 + 3)) + 1) >> 1 << 3   (N = 1024, log_lut_count = 3)
    uint64_t y = x >> 55;
    y = (y + 1) >> 1;
    return (int)(y << 3);
}

// ---- key tiles through a bulk-copy (TMA) ring ------------------------------------------------------------
// Used by the blind rotation, the trace, the scheme switch and the LUT ladders.  Described for the blind
// rotation: the 4 groups of a CTA consume the same BSK tiles (BSK_i row r = 3 Fourier polys = 24,576 B) in the
// same order, so each tile is fetched ONCE per CTA with a bulk asynchronous copy (cp.async.bulk, the
// 1-D TMA path: SASS UBLKCP) into a 2-deep shared-memory ring guarded by full/empty mbarriers, while
// the groups are still busy with the forward FFT that precedes its use.  This removes the exposed
// L2 latency of 72 dependent 16-byte loads per thread per step (ncu r01: long_scoreboard was the top
// stall) and cuts L2->SM key traffic 4x.  Thread 0 of group 0 is the producer; every consumer thread
// releases a tile with one mbarrier arrive after its last read, so no extra group barrier is needed.
constexpr int kBrTileBytes = 3 * 512 * 16;  // 24,576
constexpr int kBrRing = 2;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, int parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ bool mbar_test(uint64_t *bar, int parity)
{
    uint32_t ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.shared::cta.b64 st, [%0];\n}\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_tile(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n}\n" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---- v3: TMA-staged + instruction diet --------------------------------------------------------------
// ncu r01 (profiles/r01_blind_rotate_ncu_full.csv) showed the FFT core itself sustains 74 % of the FP64
// peak at this occupancy (tools/bench_fft) while the whole kernel reached 28 %: the time goes to the
// glue between transforms.  Changes relative to k_blind_rotate_tma:
//   * accumulator stored as PAIRS (coef[j], coef[j+512]) so the folded FFT input point, its rotated
//     partner and the read-modify-write of the update are single 128-bit shared accesses;
//   * l = 1, B = 2^23 digit computed from the high word only (5 integer ops instead of the generic
//     multi-level decomposer);
//   * the BSK tile reads are software-pipelined against the multiply-accumulate (next column's 8 values
//     are in flight while the current column's 32 DFMAs issue), the first column prefetched before the
//     last forward pass.
// (Tried and rejected on B200: pass-2 twiddles in a shared table, 13.3 vs 12.4 ms; three polynomials in
//  flight per group with 3 groups per CTA, 18.5 ms: occupancy beats per-thread ILP here.)
struct __align__(16) u64x2 {
    uint64_t lo, hi;
};

__device__ __forceinline__ void fwd_p2_s(cplx v[8], cplx *scr, const cplx *t2s, int t)
{
    const int k1 = t >> 3, tp = t & 7;
#pragma unroll
    for (int mp = 0; mp < 8; mp++) v[mp] = scr[slot(k1, tp, mp)];
    dft8<false>(v);
    scr[slot(k1, tp, 0)] = v[0];
#pragma unroll
    for (int k2 = 1; k2 < 8; k2++) scr[slot(k1, tp, k2)] = cmul(v[k2], t2s[k2 * 8]);
}
__device__ __forceinline__ void inv_p2_s(cplx v[8], cplx *scr, const cplx *t2s, int t)
{
    const int k1 = t >> 3, tp = t & 7;
    v[0] = scr[slot(k1, tp, 0)];
#pragma unroll
    for (int k2 = 1; k2 < 8; k2++) v[k2] = cmul_conj(scr[slot(k1, tp, k2)], t2s[k2 * 8]);
    dft8<true>(v);
#pragma unroll
    for (int mp = 0; mp < 8; mp++) scr[slot(k1, tp, mp)] = v[mp];
}

// inverse transform with the pass-2 twiddles in shared memory (t2s = table[k2*8 + t'] + (t & 7))
__device__ __forceinline__ void inv_fft_s(cplx v[8], Group &g, const Twiddles &tw, const cplx *t2s)
{
    cplx *s = g.flip ? g.scr1 : g.scr0;
    g.flip ^= 1;
    inv_p3(v, s, g.t);
    group_sync(g.bar);
    inv_p2_s(v, s, t2s, g.t);
    group_sync(g.bar);
    inv_p1(v, s, tw, g.t);
}
// shuffle-exchange variant with the rotated pass-2 twiddles in shared memory (t2xs = table[r*8 + a] + (t & 7))
__device__ __forceinline__ void fwd_p2x_s(cplx v[8], const cplx *scr, const cplx *t2xs, int t)
{
    const int k1 = t >> 3, tp = t & 7;
#pragma unroll
    for (int mp = 0; mp < 8; mp++) v[mp] = scr[slot(k1, tp, mp)];
    dft8<false>(v);
#pragma unroll
    for (int r = 0; r < 8; r++) v[r] = cmul(v[r], t2xs[r * 8]);
}
__device__ __forceinline__ void inv_p2x_s(cplx v[8], cplx *scr, const cplx *t2xs, int t)
{
    const int k1 = t >> 3, tp = t & 7;
#pragma unroll
    for (int r = 0; r < 8; r++) v[r] = cmul_conj(v[r], t2xs[r * 8]);
    dft8<true>(v);
#pragma unroll
    for (int mp = 0; mp < 8; mp++) scr[slot(k1, tp, mp)] = v[mp];
}
__device__ __forceinline__ void fill_t2x_table(cplx *t2tab, const double *twtab, int tid)
{
    if (tid < 64) {
        const int a = tid >> 3, r = tid & 7;
        const double *x = twtab + kTwiddleXOffset;
        t2tab[r * 8 + a] = cplx{x[(512 + a * 8 + r) * 2], x[(512 + a * 8 + r) * 2 + 1]};
    }
}
// fill a 64-entry shared table with the pass-2 twiddles transposed to [k2][t'] (conflict-free reads)
__device__ __forceinline__ void fill_t2_table(cplx *t2tab, const double *twtab, int tid)
{
    if (tid < 64) {
        const int tp = tid >> 3, k2 = tid & 7;
        t2tab[k2 * 8 + tp] = cplx{twtab[(512 + tp * 8 + k2) * 2], twtab[(512 + tp * 8 + k2) * 2 + 1]};
    }
}

// ---- v4: the production blind rotation = v3 (TMA ring, paired accumulator, shuffle-exchange transforms) with the per-thread
// twiddles in TENSOR MEMORY.  v3 kept the 16 complex pass-1 / pass-2 twiddles of a thread in 64 of its 246 registers.
// Blackwell's tensor memory (256 KB per SM, idle in an FP64 kernel) is addressable per lane with tcgen05.ld/st (SASS
// LDTM/STTM): every thread parks its twiddles there once and fetches four at a time right before the multiply
// (tools/bench_tmem.cu: 360-470 B/clk/SM, 22-35 cycles, no interference with the shared-memory pipe).  ptxas spends the
// freed registers on deeper load/FMA scheduling: 5.53 instead of 5.80 ms per wave of 592 ciphertexts (-4.8 %), FP64 pipe
// 62 % of a step.  (More groups per SM at the 168-register cap of a 320/384-thread CTA lose: profiles/r02_brbench_variants.txt.)
// The pass-2 <-> pass-3 transposes of all six transforms go through width-8 warp shuffles (fft512.cuh, shuffle-exchange
// variant) instead of shared memory: 432 fewer shared-memory wavefronts per step and ciphertext and 6 instead of 12 group
// barriers per step.  The BSK stays in the plain transform's layout.
__device__ __forceinline__ void tmem_alloc_cols(uint32_t *slot, int cols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cols(uint32_t addr, int cols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_ld_c4(uint32_t taddr, cplx *w)
{
    asm volatile(
        "{\n\t.reg .b32 t<16>;\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {t0,t1,t2,t3,t4,t5,t6,t7,t8,t9,t10,t11,t12,t13,t14,t15}, [%8];\n\t"
        "tcgen05.wait::ld.sync.aligned;\n\t"
        "mov.b64 %0, {t0,t1};\n\tmov.b64 %1, {t2,t3};\n\tmov.b64 %2, {t4,t5};\n\tmov.b64 %3, {t6,t7};\n\t"
        "mov.b64 %4, {t8,t9};\n\tmov.b64 %5, {t10,t11};\n\tmov.b64 %6, {t12,t13};\n\tmov.b64 %7, {t14,t15};\n\t}"
        : "=d"(w[0].x), "=d"(w[0].y), "=d"(w[1].x), "=d"(w[1].y), "=d"(w[2].x), "=d"(w[2].y), "=d"(w[3].x), "=d"(w[3].y)
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st_c4(uint32_t taddr, const cplx *w)
{
    asm volatile(
        "{\n\t.reg .b32 t<16>;\n\t"
        "mov.b64 {t0,t1}, %1;\n\tmov.b64 {t2,t3}, %2;\n\tmov.b64 {t4,t5}, %3;\n\tmov.b64 {t6,t7}, %4;\n\t"
        "mov.b64 {t8,t9}, %5;\n\tmov.b64 {t10,t11}, %6;\n\tmov.b64 {t12,t13}, %7;\n\tmov.b64 {t14,t15}, %8;\n\t"
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {t0,t1,t2,t3,t4,t5,t6,t7,t8,t9,t10,t11,t12,t13,t14,t15};\n\t}" ::"r"(taddr),
        "d"(w[0].x), "d"(w[0].y), "d"(w[1].x), "d"(w[1].y), "d"(w[2].x), "d"(w[2].y), "d"(w[3].x), "d"(w[3].y)
        : "memory");
}
// tm = this thread's 64 tensor-memory columns: t1x[0..7] at [0, 32), t2x[0..7] at [32, 64)
__device__ __forceinline__ void fwd_p1_tm(cplx v[8], cplx *scr, uint32_t tm, int t)
{
    const double cr[8] = CBS_CM_RE, ci[8] = CBS_CM_IM;
#pragma unroll
    for (int m = 1; m < 8; m++) v[m] = cmul(v[m], cplx{cr[m], ci[m]});
    dft8<false>(v);
    const int a = t & 7, b = t >> 3;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        cplx w[4];
        tmem_ld_c4(tm + 16 * h, w);
#pragma unroll
        for (int k = 0; k < 4; k++) scr[slot(4 * h + k, a, b)] = cmul(v[4 * h + k], w[k]);
    }
}
__device__ __forceinline__ void fwd_p2x_tm(cplx v[8], const cplx *scr, uint32_t tm, int t)
{
    const int k1 = t >> 3, tp = t & 7;
#pragma unroll
    for (int mp = 0; mp < 8; mp++) v[mp] = scr[slot(k1, tp, mp)];
    dft8<false>(v);
#pragma unroll
    for (int h = 0; h < 2; h++) {
        cplx w[4];
        tmem_ld_c4(tm + 32 + 16 * h, w);
#pragma unroll
        for (int k = 0; k < 4; k++) v[4 * h + k] = cmul(v[4 * h + k], w[k]);
    }
}
__device__ __forceinline__ void inv_p2x_tm(cplx v[8], cplx *scr, uint32_t tm, int t)
{
    const int k1 = t >> 3, tp = t & 7;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        cplx w[4];
        tmem_ld_c4(tm + 32 + 16 * h, w);
#pragma unroll
        for (int k = 0; k < 4; k++) v[4 * h + k] = cmul_conj(v[4 * h + k], w[k]);
    }
    dft8<true>(v);
#pragma unroll
    for (int mp = 0; mp < 8; mp++) scr[slot(k1, tp, mp)] = v[mp];
}
__device__ __forceinline__ void inv_p1_tm(cplx v[8], const cplx *scr, uint32_t tm, int t)
{
    const double cr[8] = CBS_CM_RE, ci[8] = CBS_CM_IM;
    const int a = t & 7, b = t >> 3;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        cplx w[4];
        tmem_ld_c4(tm + 16 * h, w);
#pragma unroll
        for (int k = 0; k < 4; k++) v[4 * h + k] = cmul_conj(scr[slot(4 * h + k, a, b)], w[k]);
    }
    dft8<true>(v);
#pragma unroll
    for (int m = 1; m < 8; m++) v[m] = cmul_conj(v[m], cplx{cr[m], ci[m]});
}

constexpr int kBr4GroupSmem = kGlweWords * 8 + 2 * 8192;   // accumulator 24 KB + 2 transpose tiles
constexpr int kBr4RingOff = kBrGroups * kBr4GroupSmem;
constexpr int kBr4BarOff = kBr4RingOff + kBrRing * kBrTileBytes;
constexpr int kBr4RotOff = kBr4BarOff + 64;                  // 2 x 2 mbarriers + tensor-memory slot
constexpr int kBr4SmemBytes = kBr4RotOff + kBrGroups * kLweN * 2;

__global__ void __launch_bounds__(64 * kBrGroups, 1) k_blind_rotate_v4(const uint64_t *__restrict__ lwe, uint64_t *__restrict__ acc_out,
                                                                        int count, const double *__restrict__ bsk_f,
                                                                        const double *__restrict__ twtab)
{
    constexpr int G = kBrGroups;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int gi = threadIdx.x >> 6, warp = threadIdx.x >> 5;
    const int ct = blockIdx.x * G + gi;
    unsigned char *ring = smem_raw + kBr4RingOff;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + kBr4BarOff);
    uint64_t *empty = full + kBrRing;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(empty + kBrRing);
    const int active_groups = min(G, count - blockIdx.x * G);
    if (threadIdx.x == 0) {
        for (int b = 0; b < kBrRing; b++) {
            mbar_init(full + b, 1);
            mbar_init(empty + b, 64 * active_groups);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc_cols(tmem_slot, 256);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tm = *tmem_slot + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)(64 * (warp >> 2));
    const int t = threadIdx.x & 63;
    {
        Twiddles tw;
        load_twiddles_x(tw, twtab, t);
        tmem_st_c4(tm, tw.t1);
        tmem_st_c4(tm + 16, tw.t1 + 4);
        tmem_st_c4(tm + 32, tw.t2);
        tmem_st_c4(tm + 48, tw.t2 + 4);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    if (ct < count) {
        const bool producer = (threadIdx.x == 0);
        const char *bsk_bytes = reinterpret_cast<const char *>(bsk_f);
        constexpr int kTiles = kLweN * 3;
        if (producer)
            for (int b = 0; b < kBrRing; b++) tma_load_tile(ring + b * kBrTileBytes, bsk_bytes + (size_t)b * kBrTileBytes, kBrTileBytes, full + b);
        __syncwarp();
        unsigned char *base = smem_raw + (size_t)gi * kBr4GroupSmem;
        u64x2 *acc = reinterpret_cast<u64x2 *>(base);  // [3][512] pairs (coef j, coef j + 512)
        const int bar = 1 + gi;
        cplx *scr0 = reinterpret_cast<cplx *>(base + kGlweWords * 8);
        cplx *scr1 = scr0 + 512;  // two tiles used alternately: no write-after-read barrier between transforms
        int flip = 0;
        const uint64_t *a = lwe + (size_t)ct * kLweSmall;
        // all 768 mod-switched rotation amounts up front: no global-load latency inside the step loop
        uint16_t *rot = reinterpret_cast<uint16_t *>(smem_raw + kBr4RotOff) + gi * kLweN;
        for (int q = t; q < kLweN; q += 64) rot[q] = (uint16_t)(modswitch_dev(a[q]) & 2047);
        {
            const int bt = modswitch_dev(a[kLweN]);
            for (int jj = t; jj < 512; jj += 64) {
                acc[jj] = u64x2{0, 0};
                acc[512 + jj] = u64x2{0, 0};
                u64x2 b;
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int j = jj + 512 * h;
                    const int e = (j + bt) & 2047;
                    const int i = e & 1023;
                    uint64_t val = 1ull << (61 - 2 * (i & 7));
                    const bool neg = (i < 512) != ((e & 1024) != 0);
                    (h ? b.hi : b.lo) = neg ? (0ull - val) : val;
                }
                acc[1024 + jj] = b;
            }
        }
        group_sync(bar);
        int tile = 0;
#pragma unroll 1
        for (int i = 0; i < kLweN; i++) {
            const int d = rot[i];
            const bool skip = (d == 0);
            cplx out[3][8];
#pragma unroll
            for (int c = 0; c < 3; c++)
#pragma unroll
                for (int k = 0; k < 8; k++) out[c][k] = cplx{0.0, 0.0};
#pragma unroll 1
            for (int r = 0; r < 3; r++, tile++) {
                const int buf = tile % kBrRing;
                const int use = tile / kBrRing;
                if (producer && tile >= 1 && tile - 1 + kBrRing < kTiles) {
                    const int pb = (tile - 1) % kBrRing, puse = (tile - 1) / kBrRing;
                    mbar_wait(empty + pb, puse & 1);
                    tma_load_tile(ring + pb * kBrTileBytes, bsk_bytes + (size_t)(tile - 1 + kBrRing) * kBrTileBytes, kBrTileBytes, full + pb);
                }
                __syncwarp();
                if (!skip) {
                    cplx v[8];
                    const u64x2 *p = acc + r * 512;
#pragma unroll
                    for (int m = 0; m < 8; m++) {
                        const int jj = t + 64 * m;
                        const int e0 = (jj - d) & 2047;
                        const uint4 src = reinterpret_cast<const uint4 *>(p)[e0 & 511];
                        const uint4 own = reinterpret_cast<const uint4 *>(p)[jj];
                        const bool sw = (e0 & 512) != 0;
                        const uint32_t ml = (uint32_t)((int32_t)(e0 << 21) >> 31);
                        const uint32_t mh = (uint32_t)((int32_t)((e0 ^ (e0 << 1)) << 21) >> 31);
                        const uint32_t rll = sw ? src.z : src.x, rlh = sw ? src.w : src.y;
                        const uint32_t rhl = sw ? src.x : src.z, rhh = sw ? src.y : src.w;
                        v[m] = cplx{digit_b23_l1_double(hi_condneg_sub(rll, rlh, ml, own.x, own.y)),
                                    digit_b23_l1_double(hi_condneg_sub(rhl, rhh, mh, own.z, own.w))};
                    }
                    cplx *s = flip ? scr1 : scr0;
                    flip ^= 1;
                    fwd_p1_tm(v, s, tm, t);
                    group_sync(bar);
                    fwd_p2x_tm(v, s, tm, t);
                    exchange8<-1>(v, t & 7);
                    const cplx *key = reinterpret_cast<const cplx *>(ring + buf * kBrTileBytes) + t;
                    mbar_wait(full + buf, use & 1);
                    cplx kc[8], kn[8];  // tile reads software-pipelined against the multiply-accumulate
#pragma unroll
                    for (int k3 = 0; k3 < 8; k3++) kc[k3] = key[k3 * 64];  // column 0, overlaps the last pass
                    fwd_p3x(v);
#pragma unroll
                    for (int c = 0; c < 3; c++) {
                        if (c < 2) {
#pragma unroll
                            for (int k3 = 0; k3 < 8; k3++) kn[k3] = key[(c + 1) * 512 + k3 * 64];
                        }
#pragma unroll
                        for (int k3 = 0; k3 < 8; k3++) cfma(out[c][k3], v[k3], kc[k3]);
#pragma unroll
                        for (int k3 = 0; k3 < 8; k3++) kc[k3] = kn[k3];
                    }
                } else {
                    mbar_wait(full + buf, use & 1);
                }
                mbar_arrive(empty + buf);
            }
            if (skip) continue;
#pragma unroll
            for (int c = 0; c < 3; c++) {
                cplx *s = flip ? scr1 : scr0;
                flip ^= 1;
                inv_p3x(out[c]);
                exchange8<1>(out[c], t & 7);
                inv_p2x_tm(out[c], s, tm, t);
                group_sync(bar);
                inv_p1_tm(out[c], s, tm, t);
                u64x2 *p = acc + c * 512;
#pragma unroll
                for (int m = 0; m < 8; m++) {
                    u64x2 w = p[t + 64 * m];
                    w.lo += torus_from_scaled(out[c][m].x);
                    w.hi += torus_from_scaled(out[c][m].y);
                    p[t + 64 * m] = w;
                }
            }
        }
        group_sync(bar);
        uint64_t *o = acc_out + (size_t)ct * kGlweWords;
        for (int w = t; w < 3 * 512; w += 64) {
            const u64x2 x = acc[w];
            const int c = w >> 9, jj = w & 511;
            o[c * 1024 + jj] = x.lo;
            o[c * 1024 + jj + 512] = x.hi;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) tmem_dealloc_cols(*tmem_slot, 256);
}

// Other decompositions measured on B200 and rejected (tools/brbench.py, 1024 ciphertexts):
//   * one polynomial per 64-thread sub-group, three sub-groups per ciphertext, spectra exchanged through
//     the transpose tiles (per-step latency 15.9 k -> 9.3 k cycles, but only 2 ciphertexts fit per SM):
//     14.2 ms vs 12.4 ms;
//   * five groups per CTA with a single transpose tile: ptxas caps 320 threads at 168 registers, 472 B of
//     spills: 23.6 ms;
//   * three polynomials in flight per group with 3 groups per CTA (ILP instead of occupancy): 18.5 ms;
//   * polynomials 0,1 and columns 0,1 transformed as pairs between the same barriers (2x ILP, same
//     occupancy): 13.7 ms, 136 B of spills;
//   * pass-2 twiddles in a shared table: 13.3 ms; balancing the last wave with 3-group CTAs: -2 % only,
//     because a group's step is a latency chain that does not speed up when its neighbours leave.
// Session 3 of round 2 (all parity-green on B200, code in git history at fbc3b6c, numbers in profiles/r02_brbench_variants.txt):
//   * the ACCUMULATOR in tensor memory (every thread owns its 24 coefficient pairs in 96 columns, update = LDTM/add/STTM, the
//     build stages the polynomial through a transient 8 KB tile): 16 instead of 40 KB of shared memory per ciphertext, so
//     SIX groups per SM (12 warps, 168 registers) and a 3-row key ring fit: 8.30 ms per wave of 888 = 9.34 us per
//     ciphertext, EXACTLY v4's 5.53 ms per 592; the same kernel at 4 groups 5.73 ms (252 registers) / 6.33 ms (compiled at
//     the 168-register cap): 8 -> 12 warps buy +14 %, the register cap costs 10 %, the staging barrier 4 %;
//   * BSK tiles shared memory -> tensor memory with tcgen05.cp (SASS UTCCP, tools/test_utccp.cu) and key reads with
//     tcgen05.ld: 7.1-7.2 ms per 592 (tensor-memory read bandwidth, 98 KB per tile and CTA);
//   * the thread's own accumulator coefficients mirrored in tensor memory (-16 % shared-memory wavefronts): 5.61 ms;
//   * the build of polynomial r + 1 software-pipelined into the products / pass 2 of polynomial r: 5.97 / 6.12 ms with the
//     rolled loop (one wasted build per step), 7.1 / 6.1 ms unrolled (80 KB of code: stall_no_instruction 0.49 per issue);
//   * polynomials 0,1 and columns 0,1 transformed as pairs (twiddles fetched once for both): 5.61 ms.
// Why none of them moves the needle (tools/bench_rf.cu, bench_issue.cu, bench_fp64ops.cu, bench_dft8.cu; DESIGN.md section 4):
// the kernel is bound by REGISTER-FILE READ BANDWIDTH.  A scheduler fetches two 32-bit register operands per cycle: DADD/DMUL
// with two fresh 64-bit sources issue every 2 cycles (the nominal FP64 rate), a DFMA with three every 3.06 cycles, a 3-source
// LOP3/IMAD every 2; DADD + LOP3 pairs take 3.6 cycles and not 2.  ncu shows 0.53 (8 warps) and 0.56 (12 warps) instructions per
// cycle and scheduler and the same 55.7 % FP64-pipe utilisation at both occupancies, and 96 extra instructions per step of
// ANY kind (LOP3 inside the products, LOP3 or DFMA inside the build) cost +1.9 ... +2.5 % each.  tools/sass_rf_model.py counts
// 10,555 register source words per warp and step (lower bound 5,278 cycles against 3,924 of FP64-pipe time and 7,050 measured).
// Per-step cycle budget of a group before the twiddles moved to tensor memory (clock64 probes, round 1): build 4.2 k, forward passes 3.3 k, pass 3 + MAC 2.8 k,
// inverse 4.2 k, torus + update 1.5 k, tile wait 0.5 k.
// Round 2, all parity-green on B200 and all slower (code in git history, commit 1d4... "Blind rotation experiments";
// numbers in profiles/r02_brbench_variants.txt, ncu summaries profiles/r02_br_*_ncu.txt, DESIGN.md section 5):
//   * twiddles in TENSOR MEMORY (tcgen05.ld/st, SASS LDTM/STTM; tools/bench_tmem.cu: 360-470 B/clk/SM next to an
//     unaffected shared-memory pipe) so that 5 or 6 groups fit the 168-register cap of a 320/384-thread CTA, one
//     transpose tile per group and a ring of single-polynomial tiles: 10.3 ms per wave of 888 (6 groups) against
//     5.8 ms per wave of 592 - the ring is one BSK row deep at 6 groups (227 KB of shared memory), so every group
//     waits for the slowest one three times per step (15 % of all samples on the tile wait);
//   * a one-warp 512-point transform (16 points per thread, shuffles only, tables in tensor memory) with a TEAM of
//     three warps per ciphertext exchanging spectra through tensor memory: shared-memory pipe 58 -> 47 %, no transpose
//     tiles, 5-row ring - but the three warps of a team share a scheduler (tensor-memory lane quarter = warp % 4 =
//     scheduler) and run in lock step: 6.7 ms per 592;
//   * the same transform with one warp per ciphertext (8 free-running warps per SM, output columns accumulated through
//     tensor memory): 130 KB of code (stall_no_instruction 0.77 per issue) and a 4-tile ring: 18.1 ms per 1184.

// ---- low-latency blind rotation for small batches -------------------------------------------------------------
// k_blind_rotate_v4 keeps one ciphertext per 64-thread group, so a step is a serial chain of 3 builds, 6 transforms and
// 9 products (~15.9 k cycles, 5.8 ms per blind rotation) however few ciphertexts there are.  The toy instance (128
// ciphertexts per round), the upper levels of the max tree and most layers of the inner-product circuit are far below
// one wave (592), so for <= 2 ciphertexts per SM a TEAM of 192 threads owns one ciphertext: sub-group r builds and
// transforms polynomial r, the three spectra meet in an 8 KB-per-polynomial exchange tile, sub-group c accumulates and
// inverse-transforms output column c and updates accumulator polynomial c (which only it reads in the next build).  The
// chain per step is 1 build + 2 transforms + 3 products.  Two teams per CTA share a 3-slot TMA ring holding the three
// BSK row tiles of the current step; the refill for step i + 1 is issued at the top of that step.
constexpr int kLlTeams = 2;
constexpr int kLlTeamThreads = 192;
constexpr int kLlTeamSmem = kGlweWords * 8 + 3 * 8192 + 3 * 8192;  // accumulator 24 KB + 3 transpose tiles + 3 exchange tiles = 72 KB
constexpr int kLlRing = 3;
constexpr int kLlSmemBytes = kLlTeams * kLlTeamSmem + kLlRing * kBrTileBytes + 64 + kLlTeams * kLweN * 2;

__device__ __forceinline__ void named_sync(int bar, int nthreads)
{
    asm volatile("bar.sync %0, %1;" ::"r"(bar), "r"(nthreads) : "memory");
}

__global__ void __launch_bounds__(kLlTeamThreads * kLlTeams, 1) k_blind_rotate_ll(const uint64_t *__restrict__ lwe,
                                                                                    uint64_t *__restrict__ acc_out, int count,
                                                                                    const double *__restrict__ bsk_f,
                                                                                    const double *__restrict__ twtab, int teams)
{
    // `teams` (1 or 2) ciphertexts per CTA: up to one ciphertext per SM the second team stays idle and a blind
    // rotation takes 2.3 ms instead of 3.2 ms (the two teams of a CTA share the shared-memory pipe)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int team = threadIdx.x / kLlTeamThreads;
    const int u = threadIdx.x - team * kLlTeamThreads;
    const int sub = u >> 6, t = u & 63;
    const int ct = (team < teams) ? blockIdx.x * teams + team : count;
    unsigned char *ring = smem_raw + (size_t)kLlTeams * kLlTeamSmem;
    uint64_t *full = reinterpret_cast<uint64_t *>(ring + kLlRing * kBrTileBytes);
    uint64_t *empty = full + kLlRing;
    const int active_teams = min(teams, count - blockIdx.x * teams);
    if (threadIdx.x == 0) {
        for (int b = 0; b < kLlRing; b++) {
            mbar_init(full + b, 1);
            mbar_init(empty + b, kLlTeamThreads * active_teams);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (ct >= count) return;
    const bool producer = (threadIdx.x == 0);
    const char *bsk_bytes = reinterpret_cast<const char *>(bsk_f);
    if (producer)
        for (int b = 0; b < kLlRing; b++) tma_load_tile(ring + b * kBrTileBytes, bsk_bytes + (size_t)b * kBrTileBytes, kBrTileBytes, full + b);
    __syncwarp();

    unsigned char *base = smem_raw + (size_t)team * kLlTeamSmem;
    u64x2 *acc = reinterpret_cast<u64x2 *>(base);                                     // [3][512] pairs (coef j, coef j + 512)
    cplx *scr = reinterpret_cast<cplx *>(base + kGlweWords * 8 + sub * 8192);         // this sub-group's transpose tile
    cplx *X = reinterpret_cast<cplx *>(base + kGlweWords * 8 + 3 * 8192);             // [3][512] spectra, slot-major
    const int tbar = 1 + team * 4, sbar = 2 + team * 4 + sub;
    const uint64_t *a = lwe + (size_t)ct * kLweSmall;
    uint16_t *rot = reinterpret_cast<uint16_t *>(ring + kLlRing * kBrTileBytes + 64) + team * kLweN;
    for (int q = u; q < kLweN; q += kLlTeamThreads) rot[q] = (uint16_t)(modswitch_dev(a[q]) & 2047);
    u64x2 *p = acc + sub * 512;  // the polynomial this sub-group owns
    {
        const int bt = modswitch_dev(a[kLweN]);
        for (int jj = t; jj < 512; jj += 64) {
            u64x2 b{0, 0};
            if (sub == 2) {
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int j = jj + 512 * h;
                    const int e = (j + bt) & 2047;
                    const int i = e & 1023;
                    uint64_t val = 1ull << (61 - 2 * (i & 7));
                    const bool neg = (i < 512) != ((e & 1024) != 0);
                    (h ? b.hi : b.lo) = neg ? (0ull - val) : val;
                }
            }
            p[jj] = b;
        }
    }
    named_sync(tbar, kLlTeamThreads);
    Twiddles tw;
    load_twiddles_x(tw, twtab, t);

#pragma unroll 1
    for (int i = 0; i < kLweN; i++) {
        const int d = rot[i];
        if (producer && i >= 1) {
#pragma unroll 1
            for (int b = 0; b < kLlRing; b++) {
                mbar_wait(empty + b, (i - 1) & 1);
                tma_load_tile(ring + b * kBrTileBytes, bsk_bytes + (size_t)(i * 3 + b) * kBrTileBytes, kBrTileBytes, full + b);
            }
        }
        __syncwarp();  // the producer lane rejoins its warp before the next (aligned) named barrier
        if (d == 0) {  // trivial rotation: the product is exactly zero, only the ring bookkeeping remains
#pragma unroll 1
            for (int b = 0; b < kLlRing; b++) {
                mbar_wait(full + b, i & 1);
                mbar_arrive(empty + b);
            }
            continue;
        }
        cplx v[8];
#pragma unroll
        for (int m = 0; m < 8; m++) {
            const int jj = t + 64 * m;
            const int e0 = (jj - d) & 2047;
            const uint4 src = reinterpret_cast<const uint4 *>(p)[e0 & 511];
            const uint4 own = reinterpret_cast<const uint4 *>(p)[jj];
            const bool sw = (e0 & 512) != 0;
            const uint32_t ml = (uint32_t)((int32_t)(e0 << 21) >> 31);
            const uint32_t mh = (uint32_t)((int32_t)((e0 ^ (e0 << 1)) << 21) >> 31);
            const uint32_t rll = sw ? src.z : src.x, rlh = sw ? src.w : src.y;
            const uint32_t rhl = sw ? src.x : src.z, rhh = sw ? src.y : src.w;
            v[m] = cplx{digit_b23_l1_double(hi_condneg_sub(rll, rlh, ml, own.x, own.y)),
                        digit_b23_l1_double(hi_condneg_sub(rhl, rhh, mh, own.z, own.w))};
        }
        fwd_p1(v, scr, tw, t);
        named_sync(sbar, 64);
        fwd_p2x(v, scr, tw, t);
        exchange8<-1>(v, t & 7);
        fwd_p3x(v);
        named_sync(tbar, kLlTeamThreads);  // every sub-group has finished reading the previous step's spectra
#pragma unroll
        for (int k3 = 0; k3 < 8; k3++) X[sub * 512 + k3 * 64 + t] = v[k3];
        named_sync(tbar, kLlTeamThreads);
        cplx out[8];
#pragma unroll
        for (int k3 = 0; k3 < 8; k3++) out[k3] = cplx{0.0, 0.0};
#pragma unroll
        for (int r = 0; r < 3; r++) {
            mbar_wait(full + r, i & 1);
            const cplx *key = reinterpret_cast<const cplx *>(ring + r * kBrTileBytes) + sub * 512 + t;
            const cplx *S = X + r * 512 + t;
            if (r == sub) {  // own spectrum: still in registers (sub-group uniform branch; 3.33 -> 3.17 ms)
#pragma unroll
                for (int k3 = 0; k3 < 8; k3++) cfma(out[k3], v[k3], key[k3 * 64]);
            } else {
#pragma unroll
                for (int k3 = 0; k3 < 8; k3++) cfma(out[k3], S[k3 * 64], key[k3 * 64]);
            }
            mbar_arrive(empty + r);
        }
        inv_p3x(out);
        exchange8<1>(out, t & 7);
        inv_p2x(out, scr, tw, t);
        named_sync(sbar, 64);
        inv_p1(out, scr, tw, t);
#pragma unroll
        for (int m = 0; m < 8; m++) {
            u64x2 w = p[t + 64 * m];
            w.lo += torus_from_scaled(out[m].x);
            w.hi += torus_from_scaled(out[m].y);
            p[t + 64 * m] = w;
        }
        named_sync(sbar, 64);  // polynomial `sub` is complete before the next build's rotated reads
    }
    uint64_t *o = acc_out + (size_t)ct * kGlweWords + sub * 1024;
    for (int w = t; w < 512; w += 64) {
        const u64x2 x = p[w];
        o[w] = x.lo;
        o[w + 512] = x.hi;
    }
}

void launch_blind_rotate(const DeviceKeys &K, const uint64_t *lwe, uint64_t *acc, int count, cudaStream_t s)
{
    if (count <= 0) return;
    // per-device state, initialised once per device (the stage executables call this from one host thread per GPU)
    static std::once_flag once[64];
    static int sm_count[64];
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    std::call_once(once[dev], [&] {
        cudaFuncSetAttribute(k_blind_rotate_ll, cudaFuncAttributeMaxDynamicSharedMemorySize, kLlSmemBytes);
        cudaFuncSetAttribute(k_blind_rotate_v4, cudaFuncAttributeMaxDynamicSharedMemorySize, kBr4SmemBytes);
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        sm_count[dev] = n > 0 ? n : 1;
    });
    const int sms = sm_count[dev];
    // CBS_BR_LOWLAT: 0 = never use the team kernel, 1 = for small batches and small tails (default), 2 = always
    static const int ll_mode = [] {
        const char *e = getenv("CBS_BR_LOWLAT");
        return e ? atoi(e) : 1;
    }();
    auto launch_team = [&](const uint64_t *in, uint64_t *out, int n) {
        const int teams = n <= sms ? 1 : kLlTeams;
        k_blind_rotate_ll<<<(n + teams - 1) / teams, kLlTeamThreads * kLlTeams, kLlSmemBytes, s>>>(in, out, n, K.bsk_f, K.tw, teams);
    };
    // small batches (at most kLlTeams ciphertexts per SM): the 192-thread-team kernel, 2.4x shorter per blind rotation
    if (ll_mode == 2 || (ll_mode == 1 && count <= kLlTeams * sms)) {
        launch_team(lwe, acc, count);
        return;
    }
    // a last partial wave of at most two ciphertexts per SM also goes to the team kernel (3.2 / 2.4 ms instead of 5.8 ms)
    const int wave = sms * kBrGroups, rem = count % wave;
    int head = count;
    if (ll_mode == 1 && count > wave && rem > 0 && rem <= kLlTeams * sms) head = count - rem;
    k_blind_rotate_v4<<<(head + kBrGroups - 1) / kBrGroups, 64 * kBrGroups, kBr4SmemBytes, s>>>(lwe, acc, head, K.bsk_f, K.tw);
    if (head < count) launch_team(lwe + (size_t)head * kLweSmall, acc + (size_t)head * kGlweWords, count - head);
}

// ------------------------------------------------------------------------------------------------
// a2: cbs_lib/src/ggsw_conv.rs:302-314 — X^-k, + 2^(log_scale-1), sample extract 0,
// lwe_preprocessing_assign (mod_switch.rs:52-74 == >> 10), convert_lwe_to_glwe_const.
// extract-then-embed only negates coefficients j >= 1 around the logical shift, so level k is:
//   mask[c][0] = m[0] >> 10,  mask[c][j] = -((-m[j]) >> 10)  with m = acc.mask[c] * X^-k,
//   body = [(acc.body[k] + 2^(63-2(k+1))) >> 10, 0, 0, ...].
__device__ __forceinline__ uint64_t glev_pre_word(const uint64_t *acc, int lvl, int p, int j)
{
    if (p < 2) {
        const uint64_t x = neg_read(acc + p * 1024, (j + lvl) & 2047);
        return (j == 0) ? (x >> 10) : (0ull - ((0ull - x) >> 10));
    }
    if (j != 0) return 0;
    return (acc[2048 + lvl] + (1ull << (63 - 2 * (lvl + 1)))) >> 10;
}

__global__ void k_glev_from_acc(const uint64_t *__restrict__ acc, uint64_t *__restrict__ glev, int count)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)count * kGlevWords) return;
    const int ct = (int)(idx / kGlevWords);
    const int rem = (int)(idx % kGlevWords);
    const int lvl = rem / kGlweWords, w = rem % kGlweWords;
    glev[idx] = glev_pre_word(acc + (size_t)ct * kGlweWords, lvl, w >> 10, w & 1023);
}

void launch_glev_from_acc(const uint64_t *acc, uint64_t *glev, int count, cudaStream_t s)
{
    if (count <= 0) return;
    const size_t total = (size_t)count * kGlevWords;
    k_glev_from_acc<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(acc, glev, count);
}

// ------------------------------------------------------------------------------------------------
// K4: trace_assign, cbs_lib/src/automorphism.rs:195-233: 10 x [X -> X^kappa (utils.rs:475-490),
// keyswitch_glwe_ciphertext with Split(41) two-limb FFT (fourier_glwe_keyswitch.rs:213-342), add].
__constant__ int c_kappa_inv[10];  // kappa^-1 mod 2048 for kappa = (1024 >> s) + 1

// ---- trace: both key limbs in one pass, two cooperating 64-thread sub-groups per GLWE -------------------
// The Split(41) keyswitch needs Sum_F F x K_lo and Sum_F F x K_hi over the same six digit spectra F.
// Holding both accumulator sets in one thread (192 registers) is impossible, so k_trace ran two
// passes and recomputed the six forward FFTs (18 FFTs per step; the first version).  Here sub-group A accumulates the lo
// limb and sub-group B the hi limb; A transforms the digits of mask polynomial 0, B those of mask
// polynomial 1, and each spectrum is handed to the partner through an 8 KB shared tile written and read
// in the owner's register-slot order (no transpose, conflict-free).  12 FFTs per step, 8 warps per SM
// (was 18 FFTs at 6 warps), and the second GLWE copy (`nxt`) is gone: all permuted reads of a step
// happen before its first write.
constexpr int kTr2Glwe = 2;                                              // GLWEs per CTA (4 sub-groups, 256 threads)

__device__ __forceinline__ void unit_sync(int bar) { asm volatile("bar.sync %0, 128;" ::"r"(bar) : "memory"); }

// coefficient e (0..2047) of the negacyclic extension, pair layout: A = (coef[q], coef[q+512]), q = e & 511
__device__ __forceinline__ uint64_t pair_pick(const u64x2 &A, int h)
{
    uint64_t x = (h & 1) ? A.hi : A.lo;
    return (h & 2) ? (0ull - x) : x;
}

// ---- automorphism-key tiles staged through a TMA ring -------------------------------------------------
// ncu r01 (profiles/r01_final_ncu_full.csv) on v2: long-scoreboard (48 dependent 16-byte key loads from L2
// per thread per digit level) was the top stall at 31 % of warp time.  The four key tiles of a digit
// level - (input poly i, limb) in {0,1}^2, 24,576 B each - are now fetched once per CTA with
// cp.async.bulk into four single-slot lanes guarded by full/empty mbarriers and shared by the two GLWE
// units of the CTA; the request for level n+1 is issued right after level n is released, one whole
// transform before its use.  Shared memory is found by single-buffering the spectrum exchange (one
// extra 128-thread barrier per level) and using one transpose tile per sub-group (the unit barriers
// already order every tile reuse).
constexpr int kTr3UnitSmem = kGlweWords * 8 + 2 * 8192 + 2 * 8192;  // cur 24 KB + 2 tiles + exchange = 56 KB
constexpr int kTr3SmemBytes = kTr2Glwe * kTr3UnitSmem + 4 * kBrTileBytes + 1024 + 64;

// Transforms are the shuffle-exchange ones (fft512.cuh "x"): one shared-memory transpose and one sub-group barrier per
// transform instead of two; both sub-groups produce spectra with the same per-lane phase, so the exchange tile and
// the (plain-layout) key tiles are used unchanged.
__global__ void __launch_bounds__(128 * kTr2Glwe, 1) k_trace_v3(const uint64_t *__restrict__ in,
                                                                 uint64_t *__restrict__ out, int count, int from_acc,
                                                                 const double *__restrict__ auto_f,
                                                                 const double *__restrict__ twtab)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int gl = threadIdx.x >> 7;
    const int sub = (threadIdx.x >> 6) & 1;
    const int t = threadIdx.x & 63;
    const int idx = blockIdx.x * kTr2Glwe + gl;
    unsigned char *ring = smem_raw + (size_t)kTr2Glwe * kTr3UnitSmem;  // lane (i, limb) at (limb*2 + i) * 24,576
    uint64_t *full = reinterpret_cast<uint64_t *>(ring + 4 * kBrTileBytes + 1024);
    uint64_t *empty = full + 4;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(empty + 4);
    const int warp = threadIdx.x >> 5;
    const int active_units = min(kTr2Glwe, count - blockIdx.x * kTr2Glwe);
    if (threadIdx.x == 0) {
        for (int b = 0; b < 4; b++) {
            mbar_init(full + b, 1);
            mbar_init(empty + b, 64 * active_units);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc_cols(tmem_slot, 128);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // the 16 complex twiddles of a thread live in tensor memory (see k_blind_rotate_v4): 64 columns per warp, the two warps
    // of a lane quarter side by side
    const uint32_t tm = *tmem_slot + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)(64 * (warp >> 2));
    {
        Twiddles tw;
        load_twiddles_x(tw, twtab, t);
        tmem_st_c4(tm, tw.t1);
        tmem_st_c4(tm + 16, tw.t1 + 4);
        tmem_st_c4(tm + 32, tw.t2);
        tmem_st_c4(tm + 48, tw.t2 + 4);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    if (idx < count) {
        const bool producer = (threadIdx.x == 0);
        const char *key_bytes = reinterpret_cast<const char *>(auto_f);
        // tile of use n = s*3 + tt (level lev = 2 - tt), lane (i, sp): Fourier polys [s][i][sp][lev][0..2]
        auto tile_src = [&](int n, int i, int sp) {
            const int s = n / 3, lev = 2 - (n % 3);
            return key_bytes + (size_t)((((s * 2 + i) * 2 + sp) * 3 + lev) * 3) * kFourierPolyDoubles * 8;
        };
        // refill of the four ring lanes for use n: `early` only takes the lanes every consumer has already released
        // (non-blocking test right after a level's products), the regular call one barrier into the next transform
        // blocks for the rest.  issued = bit mask of the lanes already requested for the pending use.
        int issued = 0;
        auto produce = [&](int n, bool early) {
            if (n >= 30) return;
    #pragma unroll
            for (int L = 0; L < 4; L++) {
                if (issued & (1 << L)) continue;
                if (n > 0) {
                    if (early) {
                        if (!mbar_test(empty + L, (n - 1) & 1)) continue;
                    } else {
                        mbar_wait(empty + L, (n - 1) & 1);
                    }
                }
                tma_load_tile(ring + L * kBrTileBytes, tile_src(n, L & 1, L >> 1), kBrTileBytes, full + L);
                issued |= 1 << L;
            }
            if (!early) issued = 0;
        };
        if (producer) produce(0, false);
        __syncwarp();  // the producer lane rejoins its warp before the next (aligned) named barrier
        int want = -1;  // next ring refill the producer owes (issued one barrier into the following transform)

        unsigned char *base = smem_raw + (size_t)gl * kTr3UnitSmem;
        u64x2 *cur = reinterpret_cast<u64x2 *>(base);
        cplx *scr = reinterpret_cast<cplx *>(base + kGlweWords * 8 + sub * 8192);
        cplx *X = reinterpret_cast<cplx *>(base + kGlweWords * 8 + 16384);  // [sub 2][512]
        const int sbar = 1 + gl * 2 + sub;
        const int ubar = 5 + gl;
        {
            const int u = threadIdx.x & 127;
            if (from_acc) {
                const uint64_t *acc = in + (size_t)(idx / kCbsLevel) * kGlweWords;
                const int lvl = idx % kCbsLevel;
                // unrolled: the 16 loads of a thread are in flight together and the polynomial index is a constant per iteration
#pragma unroll
                for (int it = 0; it < 12; it++) {
                    const int w = u + 128 * it;
                    const int p = it >> 2, jj = w & 511;
                    cur[w] = u64x2{glev_pre_word(acc, lvl, p, jj), glev_pre_word(acc, lvl, p, jj + 512)};
                }
            } else {
                const uint64_t *src = in + (size_t)idx * kGlweWords;
#pragma unroll
                for (int it = 0; it < 12; it++) {
                    const int w = u + 128 * it;
                    const int p = it >> 2, jj = w & 511;
                    cur[w] = u64x2{src[p * 1024 + jj], src[p * 1024 + jj + 512]};
                }
            }
        }
        unit_sync(ubar);

    #pragma unroll 1
        for (int s = 0; s < 10; s++) {
            const int kinv = c_kappa_inv[s];
            uint64_t pk[16];
            {
                const u64x2 *p = cur + sub * 512;
    #pragma unroll
                for (int m = 0; m < 8; m++) {
                    const int jj = t + 64 * m;
                    const int e = (jj * kinv) & 2047;
                    const u64x2 A = p[e & 511];
                    const int h = e >> 9;
                    pk[2 * m] = pack_digits<13, 3, uint64_t>(pair_pick(A, h));
                    pk[2 * m + 1] = pack_digits<13, 3, uint64_t>(pair_pick(A, (h + kinv) & 3));
                }
            }
            u64x2 nb[4];
    #pragma unroll
            for (int q = 0; q < 4; q++) {
                const int jj = t + 64 * (4 * sub + q);
                const int e = (jj * kinv) & 2047;
                const u64x2 A = cur[1024 + (e & 511)];
                const int h = e >> 9;
                const u64x2 own = cur[1024 + jj];
                nb[q] = u64x2{own.lo + pair_pick(A, h), own.hi + pair_pick(A, (h + kinv) & 3)};
            }
            unit_sync(ubar);
    #pragma unroll
            for (int q = 0; q < 4; q++) cur[1024 + t + 64 * (4 * sub + q)] = nb[q];

            cplx acc[3][8];
    #pragma unroll
            for (int c = 0; c < 3; c++)
    #pragma unroll
                for (int k = 0; k < 8; k++) acc[c][k] = cplx{0.0, 0.0};
    #pragma unroll 1
            for (int tt = 0; tt < 3; tt++) {
                const int n = s * 3 + tt;
                cplx v[8];
    #pragma unroll
                for (int m = 0; m < 8; m++)
                    v[m] = cplx{i32_to_double(unpack_digit<13, uint64_t>(pk[2 * m], tt)),
                                i32_to_double(unpack_digit<13, uint64_t>(pk[2 * m + 1], tt))};
                fwd_p1_tm(v, scr, tm, t);
                group_sync(sbar);
                if (producer && want >= 0) {
                    produce(want, false);
                    want = -1;
                }
                __syncwarp();  // the producer lane rejoins its warp before the next (aligned) named barrier
                fwd_p2x_tm(v, scr, tm, t);
                exchange8<-1>(v, t & 7);
                fwd_p3x(v);
                cplx *Xw = X + sub * 512 + t;
                const cplx *Xr = X + (1 - sub) * 512 + t;
    #pragma unroll
                for (int k3 = 0; k3 < 8; k3++) Xw[k3 * 64] = v[k3];
                unit_sync(ubar);
                // own spectrum x key(i = sub, limb = sub), partner spectrum x key(i = 1 - sub, limb = sub)
                const int Lown = sub * 2 + sub, Loth = sub * 2 + (1 - sub);
                mbar_wait(full + Lown, n & 1);
                {
                    const cplx *key = reinterpret_cast<const cplx *>(ring + Lown * kBrTileBytes) + t;
    #pragma unroll
                    for (int c = 0; c < 3; c++)
    #pragma unroll
                        for (int k3 = 0; k3 < 8; k3++) cfma(acc[c][k3], v[k3], key[c * 512 + k3 * 64]);
                }
                mbar_arrive(empty + Lown);
                mbar_wait(full + Loth, n & 1);
                {
                    const cplx *key = reinterpret_cast<const cplx *>(ring + Loth * kBrTileBytes) + t;
    #pragma unroll
                    for (int k3 = 0; k3 < 8; k3++) {
                        const cplx o = Xr[k3 * 64];
    #pragma unroll
                        for (int c = 0; c < 3; c++) cfma(acc[c][k3], o, key[c * 512 + k3 * 64]);
                    }
                }
                mbar_arrive(empty + Loth);
                want = n + 1;
                unit_sync(ubar);  // partner finished reading the exchange tile before it is rewritten
                if (producer) produce(want, true);  // lanes both units have released are refilled right away
                __syncwarp();
            }
            const int shift = sub ? 41 : 0;
    #pragma unroll
            for (int c = 0; c < 3; c++) {
                inv_p3x(acc[c]);
                exchange8<1>(acc[c], t & 7);
                if (producer && want >= 0) {
                    produce(want, false);
                    want = -1;
                }
                __syncwarp();
                inv_p2x_tm(acc[c], scr, tm, t);
                group_sync(sbar);
                inv_p1_tm(acc[c], scr, tm, t);
                u64x2 *p = cur + c * 512;
                if (sub == 0) {
    #pragma unroll
                    for (int m = 0; m < 8; m++) {
                        u64x2 w = p[t + 64 * m];
                        w.lo += torus_from_scaled(acc[c][m].x);
                        w.hi += torus_from_scaled(acc[c][m].y);
                        p[t + 64 * m] = w;
                    }
                }
                unit_sync(ubar);
                if (sub == 1) {
    #pragma unroll
                    for (int m = 0; m < 8; m++) {
                        u64x2 w = p[t + 64 * m];
                        w.lo += torus_from_scaled(acc[c][m].x) << shift;
                        w.hi += torus_from_scaled(acc[c][m].y) << shift;
                        p[t + 64 * m] = w;
                    }
                }
            }
            unit_sync(ubar);
        }
        uint64_t *dst = out + (size_t)idx * kGlweWords;
        for (int w = threadIdx.x & 127; w < 3 * 512; w += 128) {
            const u64x2 x = cur[w];
            const int c = w >> 9, jj = w & 511;
            dst[c * 1024 + jj] = x.lo;
            dst[c * 1024 + jj + 512] = x.hi;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) tmem_dealloc_cols(*tmem_slot, 128);
}

// Round 2, measured and rejected (code in git history, "trace v4"): one 64-thread group per GLWE with the six keyswitch
// accumulators in TENSOR MEMORY (tcgen05.ld/st, one round trip per accumulator and input polynomial, the three digit
// spectra resident in registers, key tiles regrouped per (in poly, limb, column) as three 8 KB bulk copies on one
// mbarrier): no exchange tile, no cross-group barrier, 4 GLWEs per CTA - parity-green, and the same throughput per SM as
// this kernel (0.243 ms per wave of 592 GLWEs against 2 x 0.116 ms per wave of 296; profiles/r02_brbench_variants.txt).
// Like the blind rotation the trace is not limited by its barriers but by three co-limiting pipes (FP64 35 %, shared
// memory 59 %, issue 39 %) at 8 warps per SM, which the register file (255 per thread) and shared memory pin.
// Session 3: THREE units per CTA (12 warps at 168 registers; the exchange tile aliased onto the transpose tiles with one
// more sub-group barrier per level, the packed digits of a step parked in tensor memory, 124 B of spills): parity-green,
// trace + scheme switch of 512 ciphertexts 1.88 ms against 1.80 ms (2.12 ms without the digits in tensor memory); the
// aliasing alone costs 0.5 % at two units (profiles/r02_brbench_variants.txt).  More resident warps do not help here either.

// ------------------------------------------------------------------------------------------------
// LWE-to-GLWE packing (Chen-Dai-Kim-Song 2020, cbs_lib glwe_conv.rs pack_lwes): big LWE i -> coefficient i % 1024 of
// GLWE i / 1024, through a tree of automorphism keyswitches, one launch per level L = 1..10 covering every group.
// Item t < s = 1024 >> L of a group is
//   q[t] = (e + X^s o) + keyswitch(auto[10 - L], (e - X^s o)(X^kappa)),   kappa = 2^L + 1,  e = p[t],  o = p[t + s],
// the keyswitch being one step of k_trace_v3 (the same Split(41) two-limb products, key ring and transforms) with the X^s
// multiply-add/subtract fused into the load.  Level 1 reads the LWE rows: p[j] = const_embed(lwe_j >> 10) (glev_pre_word's
// arithmetic).  A group of c inputs has min(c, s) non-zero items at level L and only those run: a zero item stays exactly
// zero (its digits, spectra and products are 0), and an o past the previous level's min(c, 2s) items is read as zero.
// Levels 2..9 work in place on ws [group][gs][3072]: item t reads slots t and t + s and writes slot t, and no other item
// touches either.  Every CTA of a launch reads the same 295 KB key, which stays in L2.  The keyswitch is written out here
// rather than shared with k_trace_v3 through an inline helper: ptxas then schedules the trace differently.
__device__ __forceinline__ uint64_t pack_in_word(const uint64_t *item, bool lwe, int p, int j)
{
    if (!lwe) return item[p * 1024 + j];
    if (p == 2) return j == 0 ? item[2048] >> 10 : 0;
    return j == 0 ? item[p * 1024] >> 10 : 0ull - (item[p * 1024 + 1024 - j] >> 10);
}

__global__ void __launch_bounds__(128 * kTr2Glwe, 1) k_pack_level(const uint64_t *src, uint64_t *dst, int count, int level,
                                                                   int gs, const double *__restrict__ auto_f,
                                                                   const double *__restrict__ twtab)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int gl = threadIdx.x >> 7;
    const int sub = (threadIdx.x >> 6) & 1;
    const int t = threadIdx.x & 63;
    const int stride = 1024 >> level;
    const int items = (count >> 10) * stride + min(count & 1023, stride);
    const int idx = blockIdx.x * kTr2Glwe + gl;
    unsigned char *ring = smem_raw + (size_t)kTr2Glwe * kTr3UnitSmem;
    uint64_t *full = reinterpret_cast<uint64_t *>(ring + 4 * kBrTileBytes + 1024);
    uint64_t *empty = full + 4;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(empty + 4);
    const int warp = threadIdx.x >> 5;
    const int active_units = min(kTr2Glwe, items - blockIdx.x * kTr2Glwe);
    if (threadIdx.x == 0) {
        for (int b = 0; b < 4; b++) {
            mbar_init(full + b, 1);
            mbar_init(empty + b, 64 * active_units);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc_cols(tmem_slot, 128);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tm = *tmem_slot + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)(64 * (warp >> 2));
    {
        Twiddles tw;
        load_twiddles_x(tw, twtab, t);
        tmem_st_c4(tm, tw.t1);
        tmem_st_c4(tm + 16, tw.t1 + 4);
        tmem_st_c4(tm + 32, tw.t2);
        tmem_st_c4(tm + 48, tw.t2 + 4);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    if (idx < items) {
        const int g = idx / stride, it = idx % stride;
        const int nprev = min(min(1024, count - g * 1024), 2 * stride);  // non-zero items of the previous level
        const bool lwe = (level == 1);
        const size_t item_words = lwe ? kLweBig : kGlweWords;
        const uint64_t *e_src = src + (lwe ? (size_t)(g * 1024 + it) : (size_t)g * gs + it) * item_words;
        const uint64_t *o_src = (it + stride < nprev) ? e_src + (size_t)stride * item_words : nullptr;
        uint64_t *dptr = dst + ((size_t)g * (level == 10 ? 1 : gs) + it) * kGlweWords;
        const int ks = 10 - level;  // automorphism key X -> X^((1024 >> ks) + 1)

        const bool producer = (threadIdx.x == 0);
        const char *key_bytes = reinterpret_cast<const char *>(auto_f);
        // tile of use n (digit level lev = 2 - n), lane (i, sp): Fourier polys [ks][i][sp][lev][0..2]; ring as k_trace_v3
        auto tile_src = [&](int n, int i, int sp) {
            return key_bytes + (size_t)((((ks * 2 + i) * 2 + sp) * 3 + (2 - n)) * 3) * kFourierPolyDoubles * 8;
        };
        int issued = 0;
        auto produce = [&](int n, bool early) {
            if (n >= 3) return;
    #pragma unroll
            for (int L = 0; L < 4; L++) {
                if (issued & (1 << L)) continue;
                if (n > 0) {
                    if (early) {
                        if (!mbar_test(empty + L, (n - 1) & 1)) continue;
                    } else {
                        mbar_wait(empty + L, (n - 1) & 1);
                    }
                }
                tma_load_tile(ring + L * kBrTileBytes, tile_src(n, L & 1, L >> 1), kBrTileBytes, full + L);
                issued |= 1 << L;
            }
            if (!early) issued = 0;
        };
        if (producer) produce(0, false);
        __syncwarp();
        int want = -1;

        unsigned char *base = smem_raw + (size_t)gl * kTr3UnitSmem;
        u64x2 *cur = reinterpret_cast<u64x2 *>(base);
        cplx *scr = reinterpret_cast<cplx *>(base + kGlweWords * 8 + sub * 8192);
        cplx *X = reinterpret_cast<cplx *>(base + kGlweWords * 8 + 16384);
        const int sbar = 1 + gl * 2 + sub;
        const int ubar = 5 + gl;
        const int u = threadIdx.x & 127;
        // cur = e - X^s o (the keyswitch input), sum = e + X^s o (kept in registers until the input has been read)
        u64x2 sum[12];
#pragma unroll
        for (int k = 0; k < 12; k++) {
            const int w = u + 128 * k;
            const int p = k >> 2, jj = w & 511;
            uint64_t ev[2], xo[2];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int j = jj + 512 * h, js = j - stride;
                ev[h] = pack_in_word(e_src, lwe, p, j);
                xo[h] = !o_src ? 0ull : js >= 0 ? pack_in_word(o_src, lwe, p, js) : 0ull - pack_in_word(o_src, lwe, p, js + 1024);
            }
            cur[w] = u64x2{ev[0] - xo[0], ev[1] - xo[1]};
            sum[k] = u64x2{ev[0] + xo[0], ev[1] + xo[1]};
        }
        unit_sync(ubar);

        const int kinv = c_kappa_inv[ks];
        uint64_t pk[16];
        {
            const u64x2 *p = cur + sub * 512;
    #pragma unroll
            for (int m = 0; m < 8; m++) {
                const int jj = t + 64 * m;
                const int e = (jj * kinv) & 2047;
                const u64x2 A = p[e & 511];
                const int h = e >> 9;
                pk[2 * m] = pack_digits<13, 3, uint64_t>(pair_pick(A, h));
                pk[2 * m + 1] = pack_digits<13, 3, uint64_t>(pair_pick(A, (h + kinv) & 3));
            }
        }
        u64x2 pb[4];  // body of the automorphism image, pairs u + 128 q
    #pragma unroll
        for (int q = 0; q < 4; q++) {
            const int e = ((u + 128 * q) * kinv) & 2047;
            const u64x2 A = cur[1024 + (e & 511)];
            const int h = e >> 9;
            pb[q] = u64x2{pair_pick(A, h), pair_pick(A, (h + kinv) & 3)};
        }
        unit_sync(ubar);
    #pragma unroll
        for (int k = 0; k < 12; k++) {
            u64x2 x = sum[k];
            if (k >= 8) {
                x.lo += pb[k - 8].lo;
                x.hi += pb[k - 8].hi;
            }
            cur[u + 128 * k] = x;
        }

        cplx acc[3][8];
    #pragma unroll
        for (int c = 0; c < 3; c++)
    #pragma unroll
            for (int k = 0; k < 8; k++) acc[c][k] = cplx{0.0, 0.0};
    #pragma unroll 1
        for (int n = 0; n < 3; n++) {
            cplx v[8];
    #pragma unroll
            for (int m = 0; m < 8; m++)
                v[m] = cplx{i32_to_double(unpack_digit<13, uint64_t>(pk[2 * m], n)),
                            i32_to_double(unpack_digit<13, uint64_t>(pk[2 * m + 1], n))};
            fwd_p1_tm(v, scr, tm, t);
            group_sync(sbar);
            if (producer && want >= 0) {
                produce(want, false);
                want = -1;
            }
            __syncwarp();
            fwd_p2x_tm(v, scr, tm, t);
            exchange8<-1>(v, t & 7);
            fwd_p3x(v);
            cplx *Xw = X + sub * 512 + t;
            const cplx *Xr = X + (1 - sub) * 512 + t;
    #pragma unroll
            for (int k3 = 0; k3 < 8; k3++) Xw[k3 * 64] = v[k3];
            unit_sync(ubar);
            const int Lown = sub * 2 + sub, Loth = sub * 2 + (1 - sub);
            mbar_wait(full + Lown, n & 1);
            {
                const cplx *key = reinterpret_cast<const cplx *>(ring + Lown * kBrTileBytes) + t;
    #pragma unroll
                for (int c = 0; c < 3; c++)
    #pragma unroll
                    for (int k3 = 0; k3 < 8; k3++) cfma(acc[c][k3], v[k3], key[c * 512 + k3 * 64]);
            }
            mbar_arrive(empty + Lown);
            mbar_wait(full + Loth, n & 1);
            {
                const cplx *key = reinterpret_cast<const cplx *>(ring + Loth * kBrTileBytes) + t;
    #pragma unroll
                for (int k3 = 0; k3 < 8; k3++) {
                    const cplx o = Xr[k3 * 64];
    #pragma unroll
                    for (int c = 0; c < 3; c++) cfma(acc[c][k3], o, key[c * 512 + k3 * 64]);
                }
            }
            mbar_arrive(empty + Loth);
            want = n + 1;
            unit_sync(ubar);
            if (producer) produce(want, true);
            __syncwarp();
        }
        const int shift = sub ? 41 : 0;
    #pragma unroll
        for (int c = 0; c < 3; c++) {
            inv_p3x(acc[c]);
            exchange8<1>(acc[c], t & 7);
            if (producer && want >= 0) {
                produce(want, false);
                want = -1;
            }
            __syncwarp();
            inv_p2x_tm(acc[c], scr, tm, t);
            group_sync(sbar);
            inv_p1_tm(acc[c], scr, tm, t);
            u64x2 *p = cur + c * 512;
            if (sub == 0) {
    #pragma unroll
                for (int m = 0; m < 8; m++) {
                    u64x2 w = p[t + 64 * m];
                    w.lo += torus_from_scaled(acc[c][m].x);
                    w.hi += torus_from_scaled(acc[c][m].y);
                    p[t + 64 * m] = w;
                }
            }
            unit_sync(ubar);
            if (sub == 1) {
    #pragma unroll
                for (int m = 0; m < 8; m++) {
                    u64x2 w = p[t + 64 * m];
                    w.lo += torus_from_scaled(acc[c][m].x) << shift;
                    w.hi += torus_from_scaled(acc[c][m].y) << shift;
                    p[t + 64 * m] = w;
                }
            }
        }
        unit_sync(ubar);
        for (int w = u; w < 3 * 512; w += 128) {
            const u64x2 x = cur[w];
            const int c = w >> 9, jj = w & 511;
            dptr[c * 1024 + jj] = x.lo;
            dptr[c * 1024 + jj + 512] = x.hi;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) tmem_dealloc_cols(*tmem_slot, 128);
}

// once per device: the automorphism inverses of the trace and packing kernels, and their shared-memory opt-in
static void auto_kernels_init()
{
    static bool init_done[64] = {false};
    int init_dev = 0;
    cudaGetDevice(&init_dev);
    bool &init = init_done[init_dev & 63];
    if (init) return;
    int kinv[10];
    for (int i = 0; i < 10; i++) {
        const int kappa = (1024 >> i) + 1;
        int x = 1;
        for (int c = 1; c < 2048; c += 2)
            if ((c * kappa) % 2048 == 1) x = c;
        kinv[i] = x;
    }
    cudaMemcpyToSymbol(c_kappa_inv, kinv, sizeof(kinv));
    cudaFuncSetAttribute(k_trace_v3, cudaFuncAttributeMaxDynamicSharedMemorySize, kTr3SmemBytes);
    cudaFuncSetAttribute(k_pack_level, cudaFuncAttributeMaxDynamicSharedMemorySize, kTr3SmemBytes);
    init = true;
}

void launch_trace(const DeviceKeys &K, const uint64_t *in, uint64_t *out, int count, int from_acc, cudaStream_t s)
{
    if (count <= 0) return;
    auto_kernels_init();
    k_trace_v3<<<(count + kTr2Glwe - 1) / kTr2Glwe, 128 * kTr2Glwe, kTr3SmemBytes, s>>>(in, out, count, from_acc, K.auto_f, K.tw);
}

void launch_pack_lwes(const DeviceKeys &K, const uint64_t *in, uint64_t *ws, uint64_t *out, int count, cudaStream_t s)
{
    if (count <= 0) return;
    auto_kernels_init();
    const int gs = std::min(count, 512);
    for (int level = 1; level <= 10; level++) {
        const int st = 1024 >> level;
        const int items = (count >> 10) * st + std::min(count & 1023, st);
        k_pack_level<<<(items + kTr2Glwe - 1) / kTr2Glwe, 128 * kTr2Glwe, kTr3SmemBytes, s>>>(
            level == 1 ? in : ws, level == 10 ? out : ws, count, level, gs, K.auto_f, K.tw);
    }
}

// ------------------------------------------------------------------------------------------------
// K5: switch_scheme cbs_lib/src/ggsw_conv.rs:163-193 (2 external products with the scheme-switching
// key, B = 2^17, l = 2, per GLEV level) fused with tfhe convert_standard_ggsw_ciphertext_to_fourier
// (call sites server_encrypted_aes_decryption.rs:430-436): every finished row is rounded to the
// torus exactly like the reference and immediately forward-transformed from registers.
constexpr int kSsGroups = 4;
constexpr int kSsGroupSmem = kGlweWords * 8 + 2 * 512 * 16;  // 40 KB
constexpr int kSsSmemBytes = kSsGroups * kSsGroupSmem;

__device__ __forceinline__ void emit_row_poly(const uint64_t lo[8], const uint64_t hi[8], uint64_t *std_dst,
                                              double *f_dst, Group &g, const Twiddles &tw)
{
    const int t = g.t;
    if (std_dst) {
#pragma unroll
        for (int m = 0; m < 8; m++) {
            std_dst[t + 64 * m] = lo[m];
            std_dst[t + 64 * m + 512] = hi[m];
        }
    }
    if (f_dst) {
        cplx v[8];
#pragma unroll
        for (int m = 0; m < 8; m++) v[m] = cplx{torus_to_double(lo[m]), torus_to_double(hi[m])};
        fwd_fft(v, g, tw);
#pragma unroll
        for (int k3 = 0; k3 < 8; k3++)
            *reinterpret_cast<double2 *>(f_dst + (size_t)(k3 * 64 + t) * 2) =
                make_double2(v[k3].x * (1.0 / 512.0), v[k3].y * (1.0 / 512.0));
    }
}

// the 12 scheme-switching-key row tiles go through the 2-deep TMA ring shared by the CTA's groups
constexpr int kSs2SmemBytes = kSsSmemBytes + kBrRing * kBrTileBytes + 64;
__global__ void __launch_bounds__(64 * kSsGroups, 1) k_scheme_switch_v2(const uint64_t *__restrict__ glev,
                                                                      uint64_t *__restrict__ ggsw_std,
                                                                      double *__restrict__ ggsw_f, int count,
                                                                      const double *__restrict__ ss_f,
                                                                      const double *__restrict__ twtab)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int gi = threadIdx.x >> 6;
    const int idx = blockIdx.x * kSsGroups + gi;  // (ciphertext, level)
    // scheme-switching key row tiles (i, level, row) = 3 Fourier polys, shared by the groups of the CTA
    unsigned char *ring = smem_raw + (size_t)kSsGroups * kSsGroupSmem;
    uint64_t *full = reinterpret_cast<uint64_t *>(ring + kBrRing * kBrTileBytes);
    uint64_t *empty = full + kBrRing;
    const int active_groups = min(kSsGroups, count * kCbsLevel - blockIdx.x * kSsGroups);
    if (threadIdx.x == 0) {
        for (int b = 0; b < kBrRing; b++) {
            mbar_init(full + b, 1);
            mbar_init(empty + b, 64 * active_groups);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (idx >= count * kCbsLevel) return;
    const bool producer = (threadIdx.x == 0);
    constexpr int kTiles = 12;  // (i 2) x (row 3) x (digit 2), consumption order
    auto tile_src = [&](int k) {
        const int i = k / 6, r = (k % 6) / 2, lev = 1 - (k % 2);
        return reinterpret_cast<const char *>(ss_f) + (size_t)(((i * 2 + lev) * 3 + r) * 3) * kFourierPolyDoubles * 8;
    };
    if (producer)
        for (int b = 0; b < kBrRing; b++) tma_load_tile(ring + b * kBrTileBytes, tile_src(b), kBrTileBytes, full + b);
    __syncwarp();  // the producer lane rejoins its warp before the next (aligned) named barrier
    int tile = 0;
    unsigned char *base = smem_raw + (size_t)gi * kSsGroupSmem;
    uint64_t *gl = reinterpret_cast<uint64_t *>(base);
    Group g;
    g.t = threadIdx.x & 63;
    g.bar = 1 + gi;
    g.scr0 = reinterpret_cast<cplx *>(base + kGlweWords * 8);
    g.scr1 = g.scr0 + 512;
    g.flip = 0;
    const int t = g.t;
    const uint64_t *src = glev + (size_t)idx * kGlweWords;
    {
        // all 24 16-byte loads of a thread in flight at once: the rolled 8-byte loop left 21 % of the kernel's samples on this
        // prologue (ncu r02, long scoreboard) - a CTA only lives for ~55 us
        const ulonglong2 *src2 = reinterpret_cast<const ulonglong2 *>(src);
        ulonglong2 *gl2 = reinterpret_cast<ulonglong2 *>(gl);
        ulonglong2 buf[kGlweWords / 128];
#pragma unroll
        for (int q = 0; q < kGlweWords / 128; q++) buf[q] = src2[t + 64 * q];
#pragma unroll
        for (int q = 0; q < kGlweWords / 128; q++) gl2[t + 64 * q] = buf[q];
    }
    Twiddles tw;
    load_twiddles(tw, twtab, g.t);
    group_sync(g.bar);
    // GGSW layout [level][row][poly]; idx = ct*7 + level
    uint64_t *std_base = ggsw_std ? ggsw_std + (size_t)idx * 3 * kGlweWords : nullptr;
    double *f_base = ggsw_f ? ggsw_f + (size_t)idx * 9 * kFourierPolyDoubles : nullptr;

#pragma unroll 1
    for (int i = 0; i < 2; i++) {
        cplx acc[3][8];
#pragma unroll
        for (int c = 0; c < 3; c++)
#pragma unroll
            for (int k = 0; k < 8; k++) acc[c][k] = cplx{0.0, 0.0};
#pragma unroll 1
        for (int r = 0; r < 3; r++) {
            uint64_t pk[16];
#pragma unroll
            for (int m = 0; m < 8; m++) {
                pk[2 * m] = pack_digits<17, 2, uint64_t>(gl[r * 1024 + t + 64 * m]);
                pk[2 * m + 1] = pack_digits<17, 2, uint64_t>(gl[r * 1024 + t + 64 * m + 512]);
            }
#pragma unroll 1
            for (int tt = 0; tt < 2; tt++, tile++) {
                const int buf = tile % kBrRing, use = tile / kBrRing;
                if (producer && tile >= 1 && tile - 1 + kBrRing < kTiles) {
                    const int pb = (tile - 1) % kBrRing, puse = (tile - 1) / kBrRing;
                    mbar_wait(empty + pb, puse & 1);
                    tma_load_tile(ring + pb * kBrTileBytes, tile_src(tile - 1 + kBrRing), kBrTileBytes, full + pb);
                }
                __syncwarp();  // the producer lane rejoins its warp before the next (aligned) named barrier
                cplx v[8];
#pragma unroll
                for (int m = 0; m < 8; m++)
                    v[m] = cplx{i32_to_double(unpack_digit<17, uint64_t>(pk[2 * m], tt)),
                                i32_to_double(unpack_digit<17, uint64_t>(pk[2 * m + 1], tt))};
                fwd_fft(v, g, tw);
                mbar_wait(full + buf, use & 1);
                const cplx *key = reinterpret_cast<const cplx *>(ring + buf * kBrTileBytes) + t;
#pragma unroll
                for (int c = 0; c < 3; c++)
#pragma unroll
                    for (int k3 = 0; k3 < 8; k3++) cfma(acc[c][k3], v[k3], key[c * 512 + k3 * 64]);
                mbar_arrive(empty + buf);
            }
        }
#pragma unroll
        for (int c = 0; c < 3; c++) {
            inv_fft(acc[c], g, tw);
            uint64_t lo[8], hi[8];
#pragma unroll
            for (int m = 0; m < 8; m++) {
                lo[m] = torus_from_scaled(acc[c][m].x);
                hi[m] = torus_from_scaled(acc[c][m].y);
            }
            emit_row_poly(lo, hi, std_base ? std_base + (size_t)(i * 3 + c) * 1024 : nullptr,
                          f_base ? f_base + (size_t)(i * 3 + c) * kFourierPolyDoubles : nullptr, g, tw);
        }
    }
    // row k = the GLEV level itself (ggsw_conv.rs:191)
#pragma unroll 1
    for (int c = 0; c < 3; c++) {
        uint64_t lo[8], hi[8];
#pragma unroll
        for (int m = 0; m < 8; m++) {
            lo[m] = gl[c * 1024 + t + 64 * m];
            hi[m] = gl[c * 1024 + t + 64 * m + 512];
        }
        emit_row_poly(lo, hi, std_base ? std_base + (size_t)(6 + c) * 1024 : nullptr,
                      f_base ? f_base + (size_t)(6 + c) * kFourierPolyDoubles : nullptr, g, tw);
    }
}

void launch_scheme_switch(const DeviceKeys &K, const uint64_t *glev, uint64_t *ggsw_std, double *ggsw_f, int count,
                          cudaStream_t s)
{
    if (count <= 0) return;
    static bool attr_done[64] = {false};
    int attr_dev = 0;
    cudaGetDevice(&attr_dev);
    bool &attr = attr_done[attr_dev & 63];
    if (!attr) {
        cudaFuncSetAttribute(k_scheme_switch_v2, cudaFuncAttributeMaxDynamicSharedMemorySize, kSs2SmemBytes);
        attr = true;
    }
    const int groups = count * kCbsLevel;
    k_scheme_switch_v2<<<(groups + kSsGroups - 1) / kSsGroups, 64 * kSsGroups, kSs2SmemBytes, s>>>(glev, ggsw_std, ggsw_f, count, K.ss_f, K.tw);
}

void launch_ggsw_to_fourier(const DeviceKeys &K, const uint64_t *ggsw_std, double *ggsw_f, int count, cudaStream_t s)
{
    launch_std_to_fourier(ggsw_std, ggsw_f, count * kCbsLevel * 9, 0, 0, K.tw, s);
}

// ------------------------------------------------------------------------------------------------
// K6: evaluate_8_to_8_cipher_lut, src/bin/server_encrypted_aes_decryption.rs:550-588 (== evaluate_8_to_8_lut
// cbs_lib/src/aes_he.rs:791-832): per accumulator 8 x [acc*X^(-2^i) - acc ; add_external_product_assign
// with GGSW bit i, B = 2^2, l = 7], then 4 sample extractions at 0, 256, 512, 768.
constexpr int kLutGroups = 4;
constexpr int kLutGroupSmem = kGlweWords * 8 + 2 * 512 * 16;  // 40 KB
constexpr int kLutSmemBytes = kLutGroups * kLutGroupSmem;

// acc += ggsw (x) (src_a - src_b) where the difference is formed per coefficient by `coef`
template <typename CoefFn>
__device__ __forceinline__ void cbs_external_product(cplx (&out)[3][8], const double *ggsw, Group &g,
                                                     const Twiddles &tw, CoefFn coef)
{
    const int t = g.t;
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
        for (int k = 0; k < 8; k++) out[c][k] = cplx{0.0, 0.0};
#pragma unroll 1
    for (int r = 0; r < 3; r++) {
        uint32_t pk[16];
#pragma unroll
        for (int m = 0; m < 8; m++) {
            pk[2 * m] = pack_digits<2, 7, uint32_t>(coef(r, t + 64 * m));
            pk[2 * m + 1] = pack_digits<2, 7, uint32_t>(coef(r, t + 64 * m + 512));
        }
#pragma unroll 1
        for (int tt = 0; tt < 7; tt++) {
            const int lev = 6 - tt;
            cplx v[8];
#pragma unroll
            for (int m = 0; m < 8; m++)
                v[m] = cplx{i32_to_double(unpack_digit<2, uint32_t>(pk[2 * m], tt)),
                            i32_to_double(unpack_digit<2, uint32_t>(pk[2 * m + 1], tt))};
            fwd_fft(v, g, tw);
            mul_acc<3>(out, v, ggsw + (size_t)((lev * 3 + r) * 3) * kFourierPolyDoubles, t);
        }
    }
}

// ---- LUT ladder with gathered selectors (inner-product circuit, host/ip_plan.h) ---------------------------
// Same ladder as k_lut8_v2 (below), but the 8 selector GGSWs of a job are picked by index (sel[job][i], -1 = the
// selector is the constant 0: the CMux is the identity and is skipped), so one circuit-bootstrapped bit can
// feed several ladders and ladders may have fewer than 8 inputs.
__global__ void __launch_bounds__(64 * kLutGroups, 1) k_lut8_gather(const double *__restrict__ ggsw_f,
                                                                     const int *__restrict__ sel,
                                                                     const uint64_t *__restrict__ luts,
                                                                     const int *__restrict__ lut_index,
                                                                     const int *__restrict__ out_index,
                                                                     uint64_t *__restrict__ out, int njobs,
                                                                     const double *__restrict__ twtab)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int gi = threadIdx.x >> 6;
    const int job = blockIdx.x * kLutGroups + gi;
    if (job >= njobs) return;
    unsigned char *base = smem_raw + (size_t)gi * kLutGroupSmem;
    uint64_t *acc = reinterpret_cast<uint64_t *>(base);
    Group g;
    g.t = threadIdx.x & 63;
    g.bar = 1 + gi;
    g.scr0 = reinterpret_cast<cplx *>(base + kGlweWords * 8);
    g.scr1 = g.scr0 + 512;
    g.flip = 0;
    Twiddles tw;
    load_twiddles(tw, twtab, g.t);
    const int t = g.t;
    const uint64_t *src = luts + (size_t)lut_index[job] * kGlweWords;
    for (int w = t; w < kGlweWords; w += 64) acc[w] = src[w];
    group_sync(g.bar);
#pragma unroll 1
    for (int i = 0; i < 8; i++) {
        const int which = sel[job * 8 + i];
        if (which < 0) continue;
        const int d = 1 << i;
        cplx o[3][8];
        cbs_external_product(o, ggsw_f + (size_t)which * kGgswWords, g, tw, [&](int r, int j) {
            return neg_read(acc + r * 1024, (j + d) & 2047) - acc[r * 1024 + j];  // acc * X^-d - acc
        });
#pragma unroll
        for (int c = 0; c < 3; c++) {
            inv_fft(o[c], g, tw);
#pragma unroll
            for (int m = 0; m < 8; m++) {
                acc[c * 1024 + t + 64 * m] += torus_from_scaled(o[c][m].x);
                acc[c * 1024 + t + 64 * m + 512] += torus_from_scaled(o[c][m].y);
            }
        }
    }
    group_sync(g.bar);
    for (int q = 0; q < 4; q++) {
        const int T = 256 * q;
        uint64_t *o = out + (size_t)(out_index[job] + q) * kLweBig;
        for (int w = t; w < 2048; w += 64) {
            const int c = w >> 10, j = w & 1023;
            const uint64_t *mp = acc + c * 1024;
            o[w] = (j <= T) ? mp[T - j] : (0ull - mp[1024 + T - j]);
        }
        if (t == 0) o[2048] = acc[2048 + T];
    }
}

void launch_lut8_gather(const DeviceKeys &K, const double *ggsw_f, const int *sel, const uint64_t *luts, const int *lut_index,
                        const int *out_index, uint64_t *out, int njobs, cudaStream_t s)
{
    if (njobs <= 0) return;
    static bool attr_done[64] = {false};
    int attr_dev = 0;
    cudaGetDevice(&attr_dev);
    if (!attr_done[attr_dev & 63]) {
        cudaFuncSetAttribute(k_lut8_gather, cudaFuncAttributeMaxDynamicSharedMemorySize, kLutSmemBytes);
        attr_done[attr_dev & 63] = true;
    }
    k_lut8_gather<<<(njobs + kLutGroups - 1) / kLutGroups, 64 * kLutGroups, kLutSmemBytes, s>>>(ggsw_f, sel, luts, lut_index,
                                                                                                 out_index, out, njobs, K.tw);
}

// rows[i] = pool[idx[i]] (LWE(2048) ciphertexts); idx < 0 gives the trivial encryption of 0
__global__ void k_gather_lwe(const uint64_t *__restrict__ pool, const int *__restrict__ idx, uint64_t *__restrict__ rows)
{
    const int i = blockIdx.x;
    const int src = idx[i];
    uint64_t *o = rows + (size_t)i * kLweBig;
    if (src < 0) {
        for (int w = threadIdx.x; w < kLweBig; w += blockDim.x) o[w] = 0;
    } else {
        const uint64_t *p = pool + (size_t)src * kLweBig;
        for (int w = threadIdx.x; w < kLweBig; w += blockDim.x) o[w] = p[w];
    }
}

void launch_gather_lwe(const uint64_t *pool, const int *idx, uint64_t *rows, int count, cudaStream_t s)
{
    if (count <= 0) return;
    k_gather_lwe<<<count, 256, 0, s>>>(pool, idx, rows);
}

// pool[dst] = pool[a] + pool[b] for LWE(2048) ciphertexts (XOR of the encrypted bits at delta 2^63), triples (dst, a, b)
__global__ void k_lwe_add_rows(uint64_t *__restrict__ pool, const int *__restrict__ triples)
{
    const int dst = triples[3 * blockIdx.x], a = triples[3 * blockIdx.x + 1], b = triples[3 * blockIdx.x + 2];
    const uint64_t *pa = pool + (size_t)a * kLweBig, *pb = pool + (size_t)b * kLweBig;
    uint64_t *o = pool + (size_t)dst * kLweBig;
    for (int w = threadIdx.x; w < kLweBig; w += blockDim.x) o[w] = pa[w] + pb[w];
}

void launch_lwe_add_rows(uint64_t *pool, const int *triples, int count, cudaStream_t s)
{
    if (count <= 0) return;
    k_lwe_add_rows<<<count, 256, 0, s>>>(pool, triples);
}

// pool[dst] = fresh LWE(2048) encryption of the bit whose circuit bootstrap left glev[pos]: 2 x the level-1 GLEV
// ciphertext (bit * 2^62 in the constant coefficient after the trace), sample-extracted at degree 0; pairs (pos, dst)
__global__ void k_glev_to_lwe(const uint64_t *__restrict__ glev, const int *__restrict__ pairs, uint64_t *__restrict__ pool)
{
    const int pos = pairs[2 * blockIdx.x], dst = pairs[2 * blockIdx.x + 1];
    const uint64_t *g = glev + (size_t)pos * kGlevWords;
    uint64_t *o = pool + (size_t)dst * kLweBig;
    for (int w = threadIdx.x; w < 2048; w += blockDim.x) {
        const int c = w >> 10, j = w & 1023;
        const uint64_t x = (j == 0) ? g[c * 1024] : (0ull - g[c * 1024 + 1024 - j]);
        o[w] = x << 1;
    }
    if (threadIdx.x == 0) o[2048] = g[2048] << 1;
}

void launch_glev_to_lwe(const uint64_t *glev, const int *pairs, uint64_t *pool, int count, cudaStream_t s)
{
    if (count <= 0) return;
    k_glev_to_lwe<<<count, 256, 0, s>>>(glev, pairs, pool);
}

// ---- LUT ladder v2: GGSW row tiles staged through the same 2-deep TMA ring as the blind rotation --------
// All groups of a CTA evaluate accumulators of the SAME byte, i.e. against the same 8 GGSW bits, so each
// (level, row) tile of 3 Fourier polynomials is fetched once per CTA.  `groups` = jobs per CTA must divide
// accs_per_byte (8 -> 4, 6 -> 3, 2 -> 2).  *masks_nonzero == 0: the LUT accumulators are trivial GLWE (zero mask),
// as every keyed LUT of rounds 8..1 and 0 is (src/data_struct.rs:145-151,258-263): the first CMux then has
// zero digits for both mask polynomials and 14 of its 21 forward transforms are skipped.
constexpr int kLut2GroupSmem = kGlweWords * 8 + 2 * 512 * 16;  // 40 KB
constexpr int kLut2SmemBytes = kLutGroups * kLut2GroupSmem + kBrRing * kBrTileBytes + 1024 + 64;

__global__ void __launch_bounds__(64 * kLutGroups, 1) k_lut8_v2(const double *__restrict__ ggsw_f,
                                                                 const uint64_t *__restrict__ luts,
                                                                 const int *__restrict__ lut_index,
                                                                 const int *__restrict__ out_index,
                                                                 uint64_t *__restrict__ out, int njobs, int accs_per_byte,
                                                                 const double *__restrict__ twtab, int groups,
                                                                 const int *__restrict__ masks_nonzero)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // trivial accumulators: found by k_masks_nonzero right after the key upload (device flag)
    const int trivial = masks_nonzero != nullptr && *masks_nonzero == 0;
    const int gi = threadIdx.x >> 6;
    const int job = (gi < groups) ? blockIdx.x * groups + gi : njobs;
    unsigned char *ring = smem_raw + (size_t)kLutGroups * kLut2GroupSmem;
    cplx *t2tab = reinterpret_cast<cplx *>(ring + kBrRing * kBrTileBytes);
    uint64_t *full = reinterpret_cast<uint64_t *>(ring + kBrRing * kBrTileBytes + 1024);
    uint64_t *empty = full + kBrRing;
    const int active_groups = min(groups, njobs - blockIdx.x * groups);
    fill_t2_table(t2tab, twtab, threadIdx.x);
    if (threadIdx.x == 0) {
        for (int b = 0; b < kBrRing; b++) {
            mbar_init(full + b, 1);
            mbar_init(empty + b, 64 * active_groups);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (job >= njobs) return;
    const bool producer = (threadIdx.x == 0);
    const char *bits = reinterpret_cast<const char *>(ggsw_f + (size_t)((blockIdx.x * groups) / accs_per_byte) * 8 * kGgswWords);
    constexpr int kTiles = 8 * 21;
    // tile k = (bit i, row r, digit tt): level 6 - tt, Fourier polys [i][lev][r][0..2]
    auto tile_src = [&](int k) {
        const int i = k / 21, r = (k % 21) / 7, lev = 6 - (k % 7);
        return bits + ((size_t)i * kGgswWords + (size_t)((lev * 3 + r) * 3) * kFourierPolyDoubles) * 8;
    };
    if (producer)
        for (int b = 0; b < kBrRing; b++) tma_load_tile(ring + b * kBrTileBytes, tile_src(b), kBrTileBytes, full + b);
    __syncwarp();  // the producer lane rejoins its warp before the next (aligned) named barrier

    unsigned char *base = smem_raw + (size_t)gi * kLut2GroupSmem;
    uint64_t *acc = reinterpret_cast<uint64_t *>(base);
    Group g;
    g.t = threadIdx.x & 63;
    g.bar = 1 + gi;
    g.scr0 = reinterpret_cast<cplx *>(base + kGlweWords * 8);
    g.scr1 = g.scr0 + 512;
    g.flip = 0;
    const int t = g.t;
    const cplx *t2s = t2tab + (t & 7);
    Twiddles tw;
    load_twiddles(tw, twtab, t);
    const uint64_t *src = luts + (size_t)lut_index[job] * kGlweWords;
    for (int w = t; w < kGlweWords; w += 64) acc[w] = src[w];
    group_sync(g.bar);

    int tile = 0;
#pragma unroll 1
    for (int i = 0; i < 8; i++) {
        const int d = 1 << i;
        cplx o[3][8];
#pragma unroll
        for (int c = 0; c < 3; c++)
#pragma unroll
            for (int k = 0; k < 8; k++) o[c][k] = cplx{0.0, 0.0};
#pragma unroll 1
        for (int r = 0; r < 3; r++) {
            const bool zero = trivial && i == 0 && r < 2;  // trivial LUT: mask polynomials are exactly zero
            uint32_t pk[16];
            if (!zero) {
                const uint64_t *p = acc + r * 1024;
#pragma unroll
                for (int m = 0; m < 8; m++) {
                    const int j = t + 64 * m;
                    pk[2 * m] = pack_digits<2, 7, uint32_t>(neg_read(p, (j + d) & 2047) - p[j]);  // acc * X^-d - acc
                    pk[2 * m + 1] = pack_digits<2, 7, uint32_t>(neg_read(p, (j + 512 + d) & 2047) - p[j + 512]);
                }
            }
#pragma unroll 1
            for (int tt = 0; tt < 7; tt++, tile++) {
                const int buf = tile % kBrRing, use = tile / kBrRing;
                if (producer && tile >= 1 && tile - 1 + kBrRing < kTiles) {
                    const int pb = (tile - 1) % kBrRing, puse = (tile - 1) / kBrRing;
                    mbar_wait(empty + pb, puse & 1);
                    tma_load_tile(ring + pb * kBrTileBytes, tile_src(tile - 1 + kBrRing), kBrTileBytes, full + pb);
                }
                __syncwarp();  // the producer lane rejoins its warp before the next (aligned) named barrier
                if (!zero) {
                    cplx v[8];
#pragma unroll
                    for (int m = 0; m < 8; m++)
                        v[m] = cplx{i32_to_double(unpack_digit<2, uint32_t>(pk[2 * m], tt)),
                                    i32_to_double(unpack_digit<2, uint32_t>(pk[2 * m + 1], tt))};
                    cplx *s = g.flip ? g.scr1 : g.scr0;
                    g.flip ^= 1;
                    fwd_p1(v, s, tw, t);
                    group_sync(g.bar);
                    fwd_p2_s(v, s, t2s, t);
                    group_sync(g.bar);
                    mbar_wait(full + buf, use & 1);
                    const cplx *key = reinterpret_cast<const cplx *>(ring + buf * kBrTileBytes) + t;
                    cplx kc[8];
#pragma unroll
                    for (int k3 = 0; k3 < 8; k3++) kc[k3] = key[k3 * 64];
                    fwd_p3(v, s, t);
#pragma unroll
                    for (int k3 = 0; k3 < 8; k3++) cfma(o[0][k3], v[k3], kc[k3]);
#pragma unroll
                    for (int c = 1; c < 3; c++)
#pragma unroll
                        for (int k3 = 0; k3 < 8; k3++) cfma(o[c][k3], v[k3], key[c * 512 + k3 * 64]);
                } else {
                    mbar_wait(full + buf, use & 1);
                }
                mbar_arrive(empty + buf);
            }
        }
#pragma unroll
        for (int c = 0; c < 3; c++) {
            inv_fft_s(o[c], g, tw, t2s);
#pragma unroll
            for (int m = 0; m < 8; m++) {
                acc[c * 1024 + t + 64 * m] += torus_from_scaled(o[c][m].x);
                acc[c * 1024 + t + 64 * m + 512] += torus_from_scaled(o[c][m].y);
            }
        }
    }
    group_sync(g.bar);
    for (int q = 0; q < 4; q++) {
        const int T = 256 * q;
        uint64_t *dst = out + (size_t)(out_index[job] + q) * kLweBig;
        for (int w = t; w < 2048; w += 64) {
            const int c = w >> 10, j = w & 1023;
            const uint64_t *mp = acc + c * 1024;
            dst[w] = (j <= T) ? mp[T - j] : (0ull - mp[1024 + T - j]);
        }
        if (t == 0) dst[2048] = acc[2048 + T];
    }
}

// flag |= 1 if any mask word (first two polynomials) of the `count` GLWE accumulators at `luts` is non-zero.  Replaces a host
// scan of up to 17 MB per key upload that sat on the critical path of every end-to-end call.
__global__ void __launch_bounds__(256) k_masks_nonzero(const uint64_t *__restrict__ luts, int count, int *__restrict__ flag)
{
    uint64_t acc = 0;
    for (int g = blockIdx.x; g < count; g += gridDim.x) {
        const uint64_t *m = luts + (size_t)g * kGlweWords;
        for (int j = threadIdx.x; j < 2048; j += 256) acc |= m[j];
    }
    if (__syncthreads_or(acc != 0) && threadIdx.x == 0) atomicOr(flag, 1);
}

void launch_masks_nonzero(const uint64_t *luts, int count, int *flag, cudaStream_t s)
{
    if (count <= 0) return;
    k_masks_nonzero<<<count < 592 ? count : 592, 256, 0, s>>>(luts, count, flag);
}

// Mask polynomials of a seeded transciphering key (include/cbs_b200.h): CTA g = GLWE g of the direction's AllRdKeys order,
// thread t = ChaCha20 block t of its mask (words 8t .. 8t + 7), written as four 16-byte stores.  The first nfirst GLWE go to
// `first`, the next 8 nfirst to `mid`, the rest to `last`.
__global__ void __launch_bounds__(256) k_expand_lut_masks(LutMaskSeed seed, uint32_t dir, int nfirst, uint64_t *__restrict__ first,
                                                          uint64_t *__restrict__ mid, uint64_t *__restrict__ last)
{
    const int g = blockIdx.x, t = threadIdx.x;
    uint64_t w[8];
    cbs_chacha::mask_block(seed.w, dir, (uint32_t)g, (uint32_t)t, w);
    uint64_t *glwe = g < nfirst ? first + (size_t)g * kGlweWords
                     : g < 9 * nfirst ? mid + (size_t)(g - nfirst) * kGlweWords
                                      : last + (size_t)(g - 9 * nfirst) * kGlweWords;
    ulonglong2 *dst = reinterpret_cast<ulonglong2 *>(glwe + 8 * t);
#pragma unroll
    for (int i = 0; i < 4; i++) dst[i] = make_ulonglong2(w[2 * i], w[2 * i + 1]);
}

void launch_expand_lut_masks(const LutMaskSeed &seed, int dir, int nfirst, int nglwe, uint64_t *first, uint64_t *mid,
                             uint64_t *last, cudaStream_t s)
{
    if (nglwe <= 0) return;
    k_expand_lut_masks<<<nglwe, cbs_chacha::kMaskBlocksPerGlwe, 0, s>>>(seed, (uint32_t)dir, nfirst, first, mid, last);
}

int launch_lut8(const DeviceKeys &K, const double *ggsw_f, const uint64_t *luts, const int *lut_index,
                const int *out_index, uint64_t *out, int njobs, int accs_per_byte, const int *masks_nonzero, cudaStream_t s)
{
    if (njobs <= 0) return 0;
    // a ragged tail would read another byte's selectors
    if (njobs % accs_per_byte != 0) return -1;
    static bool attr_done[64] = {false};
    int attr_dev = 0;
    cudaGetDevice(&attr_dev);
    bool &attr = attr_done[attr_dev & 63];
    if (!attr) {
        cudaFuncSetAttribute(k_lut8_v2, cudaFuncAttributeMaxDynamicSharedMemorySize, kLut2SmemBytes);
        attr = true;
    }
    // `groups` jobs per CTA must all belong to the same byte: the largest divisor of accs_per_byte that fits a CTA
    int groups = 1;
    for (int gsz = kLutGroups; gsz >= 1; gsz--)
        if (accs_per_byte % gsz == 0) {
            groups = gsz;
            break;
        }
    k_lut8_v2<<<njobs / groups, 64 * kLutGroups, kLut2SmemBytes, s>>>(ggsw_f, luts, lut_index, out_index, out, njobs, accs_per_byte, K.tw,
                                                                      groups, masks_nonzero);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// a8: known_rotate_keyed_lut, cbs_lib/src/aes_he.rs:64-93 (rounds 10 + 9: the AES ciphertext byte is
// public, so the keyed LUT is "rotated" by plain sample extraction at lut_idx*256 + byte).
// t4 layout [4 mult][nblocks][128][2049]; k10_9 layout [4][16][2][3072]; ct = raw AES ciphertext bytes.
// slot != nullptr: luts is a key-slot pool [S][nmult][16][2] and block blk reads slot slot[blk].
__global__ void k_known_rotate(const uint8_t *__restrict__ ct, const uint64_t *__restrict__ luts,
                               uint64_t *__restrict__ tm, int nblocks, int inv_shift, const int *__restrict__ slot)
{
    const int lweid = blockIdx.x;  // (m, blk, i)
    const int i = lweid % 128, blk = (lweid / 128) % nblocks, m = lweid / (128 * nblocks);
    const int byte = i >> 3, bit = i & 7;
    // inverse direction: cleartext inv_shift_rows of the AES ciphertext first
    // (server_encrypted_aes_decryption.rs:89-91,590-597); forward direction: SubBytes precedes ShiftRows
    const int row = byte & 3, col = byte >> 2;
    const int src = inv_shift ? 4 * ((col - row + 4) & 3) + row : byte;
    const int T = (bit & 3) * 256 + ct[blk * 16 + src];
    if (slot) luts += (size_t)slot[blk] * (gridDim.x / (128 * nblocks)) * 32 * kGlweWords;
    const uint64_t *glwe = luts + (size_t)((m * 16 + byte) * 2 + (bit >> 2)) * kGlweWords;
    uint64_t *o = tm + (size_t)lweid * kLweBig;
    for (int w = threadIdx.x; w < 2048; w += blockDim.x) {
        const int c = w >> 10, j = w & 1023;
        const uint64_t *mp = glwe + c * 1024;
        o[w] = (j <= T) ? mp[T - j] : (0ull - mp[1024 + T - j]);
    }
    if (threadIdx.x == 0) o[2048] = glwe[2048 + T];
}

void launch_known_rotate(const uint8_t *ct, const uint64_t *luts, uint64_t *tm, int nblocks, int nmult, int inv_shift,
                         const int *slot, cudaStream_t s)
{
    if (nblocks <= 0) return;
    k_known_rotate<<<nmult * nblocks * 128, 256, 0, s>>>(ct, luts, tm, nblocks, inv_shift, slot);
}

// Key-slot LUT index tables of one lane part of nb blocks (block b under slot slot[b] of a pool [S][...]): the middle rounds'
// job (blk, byte, m, a) -> slot * 8 nmult 32 + (m 16 + byte) 2 + a (GLWE from the round's base in mid [S][8][nmult][16][2]),
// the last round's job (blk, byte, a) -> slot * 32 + byte 2 + a, in the job order of the single-key tables; CTA 0 also writes
// *flag = OR of slot_flags[slot[b]] (non-zero: some block's LUTs have a non-zero mask, so no block takes the first-CMux
// shortcut of trivial LUTs).
__global__ void __launch_bounds__(256) k_slot_lut_index(const int *__restrict__ slot, int nb, int nmult,
                                                        const int *__restrict__ slot_flags, int *__restrict__ lut_mid,
                                                        int *__restrict__ lut_last, int *__restrict__ flag)
{
    const int n = nb * 16 * nmult * 2;
    for (int job = blockIdx.x * blockDim.x + threadIdx.x; job < n; job += gridDim.x * blockDim.x) {
        const int a = job & 1, m = (job >> 1) % nmult, bb = job / (2 * nmult);  // bb = blk * 16 + byte
        const int s = slot[bb >> 4], byte = bb & 15;
        lut_mid[job] = s * 8 * nmult * 32 + (m * 16 + byte) * 2 + a;
        if (m == 0) lut_last[bb * 2 + a] = s * 32 + byte * 2 + a;
    }
    if (blockIdx.x == 0) {
        int any = 0;
        for (int b = threadIdx.x; b < nb; b += blockDim.x) any |= slot_flags[slot[b]];
        any = __syncthreads_or(any != 0);
        if (threadIdx.x == 0) *flag = any != 0;
    }
}

void launch_slot_lut_index(const int *slot, int nb, int nmult, const int *slot_flags, int *lut_mid, int *lut_last, int *flag,
                           cudaStream_t s)
{
    if (nb <= 0) return;
    const int n = nb * 16 * nmult * 2, blocks = (n + 255) / 256;
    k_slot_lut_index<<<blocks < 148 ? blocks : 148, 256, 0, s>>>(slot, nb, nmult, slot_flags, lut_mid, lut_last, flag);
}

// forward linear layer: he_shift_rows (cbs_lib/src/aes_he.rs:348-366) on the x1, x2, x3 lists followed by
// he_mix_columns_precomp (aes_he.rs:441-474), fused into one gather-add.  t3 = [3 (x1,x2,x3)][nblocks][128][2049].
__global__ void k_fwd_linear(const uint64_t *__restrict__ t3, uint64_t *__restrict__ st, int nblocks)
{
    const int lweid = blockIdx.x;
    const int bit = lweid & 7, byte = (lweid >> 3) & 15, blk = lweid >> 7;
    const int row = byte & 3, col = byte >> 2;
    const size_t mult = (size_t)nblocks * 128 * kLweBig;
    // shifted(r, c) = t(r, (r + c) % 4)
    auto src = [&](int m, int r) {
        r &= 3;
        return t3 + (size_t)m * mult + ((size_t)blk * 128 + (size_t)(4 * ((r + col) & 3) + r) * 8 + bit) * kLweBig;
    };
    const uint64_t *p2 = src(1, row), *p3 = src(2, row + 1), *pa = src(0, row + 2), *pb = src(0, row + 3);
    uint64_t *o = st + (size_t)lweid * kLweBig;
    for (int w = threadIdx.x; w < kLweBig; w += blockDim.x) o[w] = p2[w] + p3[w] + pa[w] + pb[w];
}

void launch_fwd_linear(const uint64_t *t3, uint64_t *st, int nblocks, cudaStream_t s)
{
    if (nblocks <= 0) return;
    k_fwd_linear<<<nblocks * 128, 256, 0, s>>>(t3, st, nblocks);
}

// CTR finish: last-round ShiftRows as a permutation, XOR with the public AES-CTR ciphertext bits
// (adding bit * 2^63 to the body), and the MSB-first bit order of result.bin.
__global__ void k_ctr_finish(const uint64_t *__restrict__ in, const uint8_t *__restrict__ ct, uint64_t *__restrict__ out)
{
    const int lweid = blockIdx.x;  // destination (blk, byte, msb-first position)
    const int pos = lweid & 7, byte = (lweid >> 3) & 15, blk = lweid >> 7;
    const int b = 7 - pos;
    const int row = byte & 3, col = byte >> 2;
    const int sbyte = 4 * ((row + col) & 3) + row;
    const uint64_t *p = in + ((size_t)blk * 128 + sbyte * 8 + b) * kLweBig;
    uint64_t *o = out + (size_t)lweid * kLweBig;
    for (int w = threadIdx.x; w < 2048; w += blockDim.x) o[w] = p[w];
    if (threadIdx.x == 0) o[2048] = p[2048] + ((uint64_t)((ct[blk * 16 + byte] >> b) & 1) << 63);
}

void launch_ctr_finish(const uint64_t *in, const uint8_t *ct, uint64_t *out, int nblocks, cudaStream_t s)
{
    if (nblocks <= 0) return;
    k_ctr_finish<<<nblocks * 128, 256, 0, s>>>(in, ct, out);
}

// a9: he_inv_mix_columns_precomp + he_inv_shift_rows, src/bin/server_encrypted_aes_decryption.rs:195-265,
// fused into one gather-add (LWE addition = XOR at delta = 2^63).  byte index = 4*col + row.
__global__ void k_inv_linear(const uint64_t *__restrict__ t4, uint64_t *__restrict__ st, int nblocks)
{
    const int lweid = blockIdx.x;  // (blk, byte, bit)
    const int bit = lweid & 7, byte = (lweid >> 3) & 15, blk = lweid >> 7;
    const int row = byte & 3, col = byte >> 2;
    const int scol = (4 - row + col) & 3;  // inv shift rows source column (row 0: identity)
    const size_t mult = (size_t)nblocks * 128 * kLweBig;
    auto src = [&](int m, int r) {
        return t4 + (size_t)m * mult + ((size_t)blk * 128 + (size_t)(4 * scol + (r & 3)) * 8 + bit) * kLweBig;
    };
    const uint64_t *p14 = src(3, row), *p11 = src(1, row + 1), *p13 = src(2, row + 2), *p9 = src(0, row + 3);
    uint64_t *o = st + (size_t)lweid * kLweBig;
    for (int w = threadIdx.x; w < kLweBig; w += blockDim.x) o[w] = p14[w] + p11[w] + p13[w] + p9[w];
}

void launch_inv_linear(const uint64_t *t4, uint64_t *st, int nblocks, cudaStream_t s)
{
    if (nblocks <= 0) return;
    k_inv_linear<<<nblocks * 128, 256, 0, s>>>(t4, st, nblocks);
}

// final reversal of the 8 LWE inside every byte (server_encrypted_aes_decryption.rs:182-189)
__global__ void k_reverse_bits(const uint64_t *__restrict__ in, uint64_t *__restrict__ out)
{
    const int lweid = blockIdx.x;
    const int srcid = (lweid & ~7) | (7 - (lweid & 7));
    const uint64_t *p = in + (size_t)srcid * kLweBig;
    uint64_t *o = out + (size_t)lweid * kLweBig;
    for (int w = threadIdx.x; w < kLweBig; w += blockDim.x) o[w] = p[w];
}

void launch_reverse_bits(const uint64_t *in, uint64_t *out, int nblocks, cudaStream_t s)
{
    if (nblocks <= 0) return;
    k_reverse_bits<<<nblocks * 128, 256, 0, s>>>(in, out);
}

// ------------------------------------------------------------------------------------------------
// a10: max_of_two, src/bin/server_encrypted_compute.rs:34-98.  One group per (pair, output bit j):
//   e <- lwe_a[j] (const-embedded);  for i = 15..0 (LSB -> MSB):
//     m0 = e + Gb[i] (x) (A - e);  m1 = B + Gb[i] (x) (e - B);  e = m0 + Ga[i] (x) (m1 - m0)
//   with A = embed(lwe_b[j]), B = embed(lwe_a[j]) (the reference's naming is crossed, :78-79).
// Differences from the reference, all deliberate (DESIGN.md): e starts from operand a's bit instead
// of carrying the previous output bit's e, so output bits are independent (parallel) and a == b
// yields the right value instead of a stale one; and the data operands A, B are not the const-embedded input
// LWEs but FRESH encryptions of the same bits taken from the circuit bootstrap that is run anyway for the selector
// GGSWs: 2 x (level-1 GLEV ciphertext, which encrypts bit * 2^62 after the trace).  With the raw LWEs the data
// noise is carried from one max_of_two to the next and grows with the depth of the reduction (measured 2^58.5
// after 3 levels, 2^60.2 after 9: the 512-value maximum of the medium instance came out wrong); refreshed
// operands make every level's output noise independent of the levels below.
constexpr int kMaxGroups = 2;
constexpr int kMaxGroupSmem = 3 * kGlweWords * 8 + 2 * 512 * 16;  // e, m0, m1 + tiles = 88 KB
constexpr int kMaxSmemBytes = kMaxGroups * kMaxGroupSmem;

// operand GLWEs of the ladder: op[i] = 2 * glev[i][level 1]  (bit * 2^63 in the constant coefficient)
__global__ void k_glev_to_operand(const uint64_t *__restrict__ glev, uint64_t *__restrict__ op)
{
    const uint64_t *src = glev + (size_t)blockIdx.x * kGlevWords;
    uint64_t *dst = op + (size_t)blockIdx.x * kGlweWords;
    for (int w = threadIdx.x; w < kGlweWords; w += blockDim.x) dst[w] = src[w] << 1;
}

void launch_glev_to_operand(const uint64_t *glev, uint64_t *op, int count, cudaStream_t s)
{
    if (count <= 0) return;
    k_glev_to_operand<<<count, 256, 0, s>>>(glev, op);
}

__global__ void __launch_bounds__(64 * kMaxGroups, 1) k_max_ladder(const double *__restrict__ ggsw_f,
                                                                    const uint64_t *__restrict__ op,
                                                                    const int *__restrict__ a_idx,
                                                                    const int *__restrict__ b_idx,
                                                                    uint64_t *__restrict__ out, int npairs,
                                                                    const double *__restrict__ twtab)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int gi = threadIdx.x >> 6;
    const int idx = blockIdx.x * kMaxGroups + gi;  // (pair, j)
    if (idx >= npairs * 16) return;
    const int pair = idx >> 4, jbit = idx & 15;
    unsigned char *base = smem_raw + (size_t)gi * kMaxGroupSmem;
    uint64_t *e = reinterpret_cast<uint64_t *>(base);
    uint64_t *m0 = e + kGlweWords, *m1 = m0 + kGlweWords;
    Group g;
    g.t = threadIdx.x & 63;
    g.bar = 1 + gi;
    g.scr0 = reinterpret_cast<cplx *>(base + 3 * kGlweWords * 8);
    g.scr1 = g.scr0 + 512;
    g.flip = 0;
    Twiddles tw;
    load_twiddles(tw, twtab, g.t);
    const int t = g.t;
    const int va = a_idx[pair], vb = b_idx[pair];
    const uint64_t *la = op + ((size_t)va * 16 + jbit) * kGlweWords;  // operand a, bit j  -> "B"
    const uint64_t *lb = op + ((size_t)vb * 16 + jbit) * kGlweWords;  // operand b, bit j  -> "A"
    for (int w = t; w < kGlweWords; w += 64) e[w] = la[w];
    group_sync(g.bar);
    cplx o[3][8];
#pragma unroll 1
    for (int i = 15; i >= 0; i--) {
        const double *Ga = ggsw_f + ((size_t)va * 16 + i) * kGgswWords;
        const double *Gb = ggsw_f + ((size_t)vb * 16 + i) * kGgswWords;
        // m0 = e + Gb (x) (A - e)
        cbs_external_product(o, Gb, g, tw, [&](int r, int j) { return lb[r * 1024 + j] - e[r * 1024 + j]; });
#pragma unroll
        for (int c = 0; c < 3; c++) {
            inv_fft(o[c], g, tw);
#pragma unroll
            for (int m = 0; m < 8; m++) {
                const int j = c * 1024 + t + 64 * m;
                m0[j] = e[j] + torus_from_scaled(o[c][m].x);
                m0[j + 512] = e[j + 512] + torus_from_scaled(o[c][m].y);
            }
        }
        // m1 = B + Gb (x) (e - B)
        cbs_external_product(o, Gb, g, tw, [&](int r, int j) { return e[r * 1024 + j] - la[r * 1024 + j]; });
#pragma unroll
        for (int c = 0; c < 3; c++) {
            inv_fft(o[c], g, tw);
#pragma unroll
            for (int m = 0; m < 8; m++) {
                const int j = t + 64 * m;
                m1[c * 1024 + j] = la[c * 1024 + j] + torus_from_scaled(o[c][m].x);
                m1[c * 1024 + j + 512] = la[c * 1024 + j + 512] + torus_from_scaled(o[c][m].y);
            }
        }
        // e = m0 + Ga (x) (m1 - m0)   (only own coefficients are touched: no cross-thread hazard)
        cbs_external_product(o, Ga, g, tw, [&](int r, int j) { return m1[r * 1024 + j] - m0[r * 1024 + j]; });
#pragma unroll
        for (int c = 0; c < 3; c++) {
            inv_fft(o[c], g, tw);
#pragma unroll
            for (int m = 0; m < 8; m++) {
                const int j = c * 1024 + t + 64 * m;
                e[j] = m0[j] + torus_from_scaled(o[c][m].x);
                e[j + 512] = m0[j + 512] + torus_from_scaled(o[c][m].y);
            }
        }
    }
    group_sync(g.bar);
    // extract_lwe_sample_from_glwe_ciphertext(e, 0)
    uint64_t *dst = out + (size_t)idx * kLweBig;
    for (int w = t; w < 2048; w += 64) {
        const int c = w >> 10, j = w & 1023;
        dst[w] = (j == 0) ? e[c * 1024] : (0ull - e[c * 1024 + 1024 - j]);
    }
    if (t == 0) dst[2048] = e[2048];
}

void launch_max_ladder(const DeviceKeys &K, const double *ggsw_f, const uint64_t *op, const int *a_idx,
                       const int *b_idx, uint64_t *out, int npairs, cudaStream_t s)
{
    if (npairs <= 0) return;
    static bool attr_done[64] = {false};
    int attr_dev = 0;
    cudaGetDevice(&attr_dev);
    bool &attr = attr_done[attr_dev & 63];
    if (!attr) {
        cudaFuncSetAttribute(k_max_ladder, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmemBytes);
        attr = true;
    }
    const int groups = npairs * 16;
    k_max_ladder<<<(groups + kMaxGroups - 1) / kMaxGroups, 64 * kMaxGroups, kMaxSmemBytes, s>>>(ggsw_f, op, a_idx, b_idx,
                                                                                                  out, npairs, K.tw);
}

// ------------------------------------------------------------------------------------------------
// FP64 FMA peak probe (roofline denominator: MEASURED_PEAKS.json has no FP64 figure; SURVEY.md 8(d)
// asks for it to be measured in the same run).  16 independent DFMA chains per thread.
__global__ void __launch_bounds__(256) k_fp64_peak(double *out, int iters)
{
    double a[16];
#pragma unroll
    for (int i = 0; i < 16; i++) a[i] = 1.0 + 1e-9 * (threadIdx.x + i);
    const double m = 1.0000001, c = 1e-7;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 16; i++) a[i] = fma(a[i], m, c);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) s += a[i];
    if (s == 123.456) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

void launch_fp64_peak(double *scratch, int blocks, int iters, cudaStream_t s)
{
    k_fp64_peak<<<blocks, 256, 0, s>>>(scratch, iters);
}

}  // namespace cbs
