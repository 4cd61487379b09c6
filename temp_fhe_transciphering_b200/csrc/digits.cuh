// digits.cuh — device-only integer glue between the u64 torus words and the FP64 transforms: the packed signed digits of
// the multi-level decompositions and the one-level B = 2^23 digit of the blind rotation.  Kept apart from
// cbs_kernels.cu so that tests/device_helpers.cu checks the very same code on the device.
#pragma once
#include "fft512.cuh"

namespace cbs {

// all LEVEL digits of x packed W = BASE_LOG+1 bits each, finest level in the low bits
template <int BASE_LOG, int LEVEL, typename PackT>
__device__ __forceinline__ PackT pack_digits(uint64_t x)
{
    constexpr int W = BASE_LOG + 1;
    uint64_t st = decomp_init(x, BASE_LOG, LEVEL);
    PackT p = 0;
#pragma unroll
    for (int tt = 0; tt < LEVEL; tt++) {
        int32_t d = decomp_next(st, BASE_LOG);
        p |= (PackT)((uint32_t)d & ((1u << W) - 1u)) << (tt * W);
    }
    return p;
}
template <int BASE_LOG, typename PackT>
__device__ __forceinline__ int32_t unpack_digit(PackT p, int tt)
{
    constexpr int W = BASE_LOG + 1;
    uint32_t raw = (uint32_t)(p >> (tt * W)) & ((1u << W) - 1u);
    return (int32_t)(raw << (32 - W)) >> (32 - W);
}

// tfhe SignedDecomposer(23, 1) digit (closest representable, balanced, in (-2^22, 2^22]) from the high word of x only,
// directly as a double.  With hi = x >> 32:
//   s = ((hi >> 8) + 1) >> 1,  digit = s - (s > 2^22 ? 2^23 : 0)   ==   (((int32)(hi - 0x100)) >> 9) + 1
// (digit_b23_l1_hi in fft512.cuh); digit + 2^31 is the low word of the magic number 2^52 + 2^31 + digit, so the
// conversion is three integer instructions and one DADD.
__device__ __forceinline__ double digit_b23_l1_double(uint32_t hi)
{
    const uint32_t lo = (uint32_t)(((int32_t)(hi - 0x100u)) >> 9) + 0x80000001u;
    return __hiloint2double(0x43300000, (int)lo) - 4503601774854144.0;
}
// high word of ((X ^ M) - M) - O for the 64-bit X = (xh:xl), O = (oh:ol) and M = (m:m), m = 0 or ~0:
// the conditional negation of X folded into the subtraction of the own coefficient
__device__ __forceinline__ uint32_t hi_condneg_sub(uint32_t xl, uint32_t xh, uint32_t m, uint32_t ol, uint32_t oh)
{
    uint32_t hi;
    asm("{\n\t.reg .u32 a, b;\n\t"
        "xor.b32 a, %1, %3;\n\t"
        "xor.b32 b, %2, %3;\n\t"
        "sub.cc.u32 a, a, %3;\n\t"
        "subc.u32 b, b, %3;\n\t"
        "sub.cc.u32 a, a, %4;\n\t"
        "subc.u32 %0, b, %5;\n\t}"
        : "=r"(hi)
        : "r"(xl), "r"(xh), "r"(m), "r"(ol), "r"(oh));
    return hi;
}

}  // namespace cbs
