// chacha20.h — the RFC 8439 ChaCha20 block function and the mask stream of the seeded transciphering keys
// (include/cbs_b200.h, "Seeded transciphering keys").  One definition for the host (keyset.cpp: the key generator's
// Rng, the seeded generators and cbs_*trans_key_seeded_expand) and the device (k_expand_lut_masks), so both expand
// a seed to the same words.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define CBS_HD __host__ __device__ __forceinline__
#define CBS_UNROLL _Pragma("unroll")
#else
#define CBS_HD inline
#define CBS_UNROLL
#endif

namespace cbs_chacha {

CBS_HD uint32_t rotl32(uint32_t x, int k) { return (x << k) | (x >> (32 - k)); }

// out = the 16 words of the block for input words `in` (constants, key, counter, nonce), after the feed-forward
CBS_HD void block(const uint32_t in[16], uint32_t out[16])
{
    uint32_t x[16];
    CBS_UNROLL
    for (int i = 0; i < 16; i++) x[i] = in[i];
#define CBS_QR(a, b, c, d)                                                                       \
    x[a] += x[b], x[d] = rotl32(x[d] ^ x[a], 16), x[c] += x[d], x[b] = rotl32(x[b] ^ x[c], 12), \
        x[a] += x[b], x[d] = rotl32(x[d] ^ x[a], 8), x[c] += x[d], x[b] = rotl32(x[b] ^ x[c], 7)
    CBS_UNROLL
    for (int r = 0; r < 10; r++) {
        CBS_QR(0, 4, 8, 12);
        CBS_QR(1, 5, 9, 13);
        CBS_QR(2, 6, 10, 14);
        CBS_QR(3, 7, 11, 15);
        CBS_QR(0, 5, 10, 15);
        CBS_QR(1, 6, 11, 12);
        CBS_QR(2, 7, 8, 13);
        CBS_QR(3, 4, 9, 14);
    }
#undef CBS_QR
    CBS_UNROLL
    for (int i = 0; i < 16; i++) out[i] = x[i] + in[i];
}

constexpr uint32_t kMaskTag = 0x6b73616d;  // "mask" (little-endian), nonce word 3 of every mask block
constexpr int kMaskBlocksPerGlwe = 256;     // 2048 mask words, 8 per block

// Mask words 8 blk .. 8 blk + 7 of GLWE g of direction dir (0 = inverse / ECB key, 1 = forward / CTR key) under the
// 32-byte mask seed `key` (8 little-endian words): key = the seed, counter = blk, nonce = (g, dir, "mask"); word i is
// out[2i] | out[2i+1] << 32.  The direction in the nonce keeps an inverse and a forward key with one seed apart: shared masks
// would reveal the difference of their tables.
CBS_HD void mask_block(const uint32_t key[8], uint32_t dir, uint32_t g, uint32_t blk, uint64_t words[8])
{
    uint32_t in[16] = {0x61707865, 0x3320646e, 0x79622d32, 0x6b206574};  // "expand 32-byte k"
    CBS_UNROLL
    for (int i = 0; i < 8; i++) in[4 + i] = key[i];
    in[12] = blk;
    in[13] = g;
    in[14] = dir;
    in[15] = kMaskTag;
    uint32_t out[16];
    block(in, out);
    CBS_UNROLL
    for (int i = 0; i < 8; i++) words[i] = (uint64_t)out[2 * i] | ((uint64_t)out[2 * i + 1] << 32);
}

}  // namespace cbs_chacha
