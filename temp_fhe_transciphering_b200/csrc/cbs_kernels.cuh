// cbs_kernels.cuh — launch wrappers of the sm_100a kernels (implemented in cbs_kernels.cu).
//
// All pointers are DEVICE pointers.  Layouts:
//   LWE(n)        [n mask][body] u64
//   GLWE          [3][1024] u64 (2 mask polys, body)
//   GLEV          [7][3][1024] u64
//   GGSW std      [7 level][3 row][3 poly][1024] u64                  (level 1 = coarsest first)
//   Fourier poly  [8 slot k3][64 thread u] complex double ("slot-major", see fft512.cuh),
//                 value = DFT bin (u>>3) + 8*(u&7) + 64*k3 of the twisted fold, times 1/512,
//                 coefficients taken as signed integers (so inverse transforms land in 2^64 units)
//   BSK Fourier   [768][3 row][3 col] Fourier polys
//   auto Fourier  [10][2 in][2 split][3 level][3 col] Fourier polys
//   ss Fourier    [2][2 level][3 row][3 col] Fourier polys
//   GGSW Fourier  [7 level][3 row][3 col] Fourier polys
//   KSK Fourier   [8 in][3 level][4 col][128] complex (radix-2 order of the 128-point transform)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cbs {

constexpr int kLweN = 768;
constexpr int kLweSmall = kLweN + 1;   // 769
constexpr int kBigN = 2048;
constexpr int kLweBig = kBigN + 1;     // 2049
constexpr int kGlweWords = 3 * 1024;   // 3072
constexpr int kCbsLevel = 7;
constexpr int kGlevWords = kCbsLevel * kGlweWords;       // 21504
constexpr int kGgswWords = kCbsLevel * 3 * kGlweWords;   // 64512 (u64 std, or doubles in Fourier)
constexpr int kFourierPolyDoubles = 1024;                // 512 complex

struct DeviceKeys {
    const double *tw;       // twiddle table (fft512.cuh)
    const double *tw128;    // twiddles of the 128-point transform (keyswitch ring N' = 256)
    const double *bsk_f;    // 768*9 Fourier polys
    const double *auto_f;   // 10*2*2*3*3 Fourier polys
    const double *ss_f;     // 2*2*3*3 Fourier polys
    const double *ksk_f;    // 8*3*4*128 complex
};

// generic std -> Fourier conversion of `npoly` polynomials (N = 1024).
// mode 0: whole word; mode 1: low `split` bits; mode 2: word >> split.
void launch_std_to_fourier(const uint64_t *in, double *out, int npoly, int mode, int split, const double *tw,
                           cudaStream_t s);
// KSK (N' = 256) std -> Fourier
void launch_ksk_to_fourier(const uint64_t *in, double *out, int npoly, const double *tw128, cudaStream_t s);

// a6  LWE(2048) -> LWE(768)
void launch_lwe_keyswitch(const DeviceKeys &K, const uint64_t *in, uint64_t *out, int count, cudaStream_t s);
// a1  blind rotation of the multi-LUT CBS accumulator
void launch_blind_rotate(const DeviceKeys &K, const uint64_t *lwe, uint64_t *acc, int count, cudaStream_t s);
// a2  acc -> 7 pre-trace GLWE (exposed separately for parity tests; the production path fuses it)
void launch_glev_from_acc(const uint64_t *acc, uint64_t *glev, int count, cudaStream_t s);
// a3  trace on `count` GLWE.  from_acc = 1: `in` is acc[count/7][3072] and a2 is fused in.
void launch_trace(const DeviceKeys &K, const uint64_t *in, uint64_t *out, int count, int from_acc, cudaStream_t s);
// LWE-to-GLWE packing: in[count][2049] big LWE -> out[ceil(count/1024)][3072], coefficient i % 1024 of GLWE i / 1024
//     decrypts to bit i; 10 launches (one per tree level), ws[ceil(count/1024)][min(count, 512)][3072] holds the levels
void launch_pack_lwes(const DeviceKeys &K, const uint64_t *in, uint64_t *ws, uint64_t *out, int count, cudaStream_t s);
// a4 + a5  glev[count][7][3072] -> ggsw std (nullable) and ggsw Fourier (nullable)
void launch_scheme_switch(const DeviceKeys &K, const uint64_t *glev, uint64_t *ggsw_std, double *ggsw_f, int count,
                          cudaStream_t s);
// a5 alone: GGSW std -> Fourier
void launch_ggsw_to_fourier(const DeviceKeys &K, const uint64_t *ggsw_std, double *ggsw_f, int count, cudaStream_t s);

// a7  8-bit LUT ladders.  job j: GGSW bits ggsw_f[(j / accs_per_byte) * 8 .. +8], accumulator
//     lut[lut_index[j]] (GLWE), outputs 4 LWE(2048) written to out[out_index[j] + {0,1,2,3}].
//     *masks_nonzero == 0 (launch_masks_nonzero) marks every accumulator as a trivial GLWE (zero mask polynomials);
//     nullptr = not known.  Returns non-zero, launching nothing, if njobs is not a multiple of accs_per_byte.
int launch_lut8(const DeviceKeys &K, const double *ggsw_f, const uint64_t *luts, const int *lut_index,
                const int *out_index, uint64_t *out, int njobs, int accs_per_byte, const int *masks_nonzero, cudaStream_t s);
// *flag |= 1 if any mask word of the `count` GLWE accumulators at `luts` is non-zero (device-side "are these LUTs trivial?")
void launch_masks_nonzero(const uint64_t *luts, int count, int *flag, cudaStream_t s);
// mask polynomials (words 0..2047) of the nglwe LUT GLWE of a seeded transciphering key of direction dir from its 32-byte
//     mask seed (chacha20.h mask_block): GLWE g < nfirst at first[g], then mid[g - nfirst], then last[g - 9 nfirst]; the body
//     words are left as they are
struct LutMaskSeed {
    uint32_t w[8];  // the seed as 8 little-endian words
};
void launch_expand_lut_masks(const LutMaskSeed &seed, int dir, int nfirst, int nglwe, uint64_t *first, uint64_t *mid,
                             uint64_t *last, cudaStream_t s);

// a7 with gathered selectors (inner-product circuit): job j runs the ladder over the GGSWs ggsw_f[sel[j*8 + i]]
//     (i = 0..7, -1 = constant-0 selector) on accumulator luts[lut_index[j]], 4 LWE(2048) out at out[out_index[j] + q]
void launch_lut8_gather(const DeviceKeys &K, const double *ggsw_f, const int *sel, const uint64_t *luts, const int *lut_index,
                        const int *out_index, uint64_t *out, int njobs, cudaStream_t s);
// rows[i] = pool[idx[i]] for LWE(2048) ciphertexts (idx < 0: trivial zero)
void launch_gather_lwe(const uint64_t *pool, const int *idx, uint64_t *rows, int count, cudaStream_t s);

// circuit plumbing (host/ip_plan.h): pool[dst] = pool[a] + pool[b] for triples (dst, a, b) of LWE(2048) rows
void launch_lwe_add_rows(uint64_t *pool, const int *triples, int count, cudaStream_t s);
// pool[dst] = fresh LWE(2048) of the bit bootstrapped into glev[pos] (2 x level-1 GLEV, sample 0), pairs (pos, dst)
void launch_glev_to_lwe(const uint64_t *glev, const int *pairs, uint64_t *pool, int count, cudaStream_t s);

// a8  rounds 10+9: sample extraction from the encrypted keyed LUTs (ct = raw AES ciphertext bytes; the cleartext inv_shift_rows is applied inside)
//     luts = [nmult][16][2] GLWE, tm = [nmult][nblocks][128][2049]; inv_shift = 1 for the inverse direction.
//     slot = nullptr: one key; else a device [nblocks] slot table, luts a key-slot pool [S][nmult][16][2] and block b reads
//     the LUTs of slot slot[b]
void launch_known_rotate(const uint8_t *ct, const uint64_t *luts, uint64_t *tm, int nblocks, int nmult, int inv_shift,
                         const int *slot, cudaStream_t s);
// key-slot LUT index tables of nb blocks under slots slot[nb] (device): lut_mid[nb*16*nmult*2] for the middle rounds (GLWE
//     indices into mid + round * nmult*32 of a pool mid [S][8][nmult][16][2]), lut_last[nb*16*2] into last [S][16][2], both in
//     the job order of the single-key tables; *flag = OR of slot_flags[slot[b]] (the k_lut8_v2 trivial-LUT flag of the blocks)
void launch_slot_lut_index(const int *slot, int nb, int nmult, const int *slot_flags, int *lut_mid, int *lut_last, int *flag,
                           cudaStream_t s);
// forward direction (CTR): ShiftRows + MixColumns-precomp over t3 = [3 (x1,x2,x3)][nblocks][128][2049]
void launch_fwd_linear(const uint64_t *t3, uint64_t *st, int nblocks, cudaStream_t s);
// last-round ShiftRows permutation + XOR with the public ciphertext bits + MSB-first order
void launch_ctr_finish(const uint64_t *in, const uint8_t *ct, uint64_t *out, int nblocks, cudaStream_t s);
// a9  st = InvShiftRows(InvMixColumns-precomp(t9, t11, t13, t14)), t4 = [4][nblocks][128][2049]
void launch_inv_linear(const uint64_t *t4, uint64_t *st, int nblocks, cudaStream_t s);
// final per-byte bit reversal (LSB-first -> MSB-first)
void launch_reverse_bits(const uint64_t *in, uint64_t *out, int nblocks, cudaStream_t s);

// a10 CMux ladder of max_of_two for `npairs` independent pairs of 16-bit values.
//     ggsw_f: Fourier GGSW of every value's 16 bits (MSB first); a_idx/b_idx: value indices;
//     op: the values' bits as fresh GLWE operands [nvalues][16][3072] (launch_glev_to_operand); out[npairs][16][2049].
void launch_max_ladder(const DeviceKeys &K, const double *ggsw_f, const uint64_t *op, const int *a_idx,
                       const int *b_idx, uint64_t *out, int npairs, cudaStream_t s);
// op[i] = 2 * glev[i][level 1]: a fresh GLWE encryption of bit i at 2^63 from its circuit bootstrap's GLEV
void launch_glev_to_operand(const uint64_t *glev, uint64_t *op, int count, cudaStream_t s);

// FP64 FMA throughput probe: blocks x 256 threads x iters x 16 FMAs
void launch_fp64_peak(double *scratch, int blocks, int iters, cudaStream_t s);

}  // namespace cbs
