// host_common.h — shared between the host-only translation units and the CUDA API layer.
#pragma once
#include "cbs_b200.h"

#include <cstdint>
#include <functional>
#include <memory>
#include <string>
#include <vector>

namespace cbs_host {
extern thread_local std::string g_last_error;
void set_error(const std::string &s);

// The two AES transciphering directions run one round pipeline over one key shape (AllRdKeys, src/data_struct.rs:11-26):
// first-round keyed LUTs [nmult][16][2] (encrypted), 8 middle rounds of [nmult][16][2] and a last round of [16][2] (trivial),
// each LUT a GLWE.  The key files, the key generation and the device upload differ only in these numbers and in the keyed
// tables; the device pipeline also picks the direction's linear layer and finishing kernel.
enum AesDir { kAesInv = 0, kAesFwd = 1 };  // ECB block decryption (inverse AES) / CTR mode (forward AES on the counters)
struct AesDirDesc {
    int nmult;                                 // GF(2^8) multiples per byte of the first and middle rounds
    uint8_t mults[4];                          // their values, in key (AllRdKeys tuple) order
    uint32_t first_words, mid_words, last_words;
    uint64_t seed_base;                        // first-round LUT `id` is encrypted with the Rng stream seed_base + id
    uint64_t seeded_noise_base;                // seeded keys: the noise of LUT g comes from the Rng stream seeded_noise_base + g
};
inline constexpr AesDirDesc kAesDirs[2] = {
    {4, {9, 11, 13, 14}, CBS_K10_9_WORDS, CBS_K8_1_WORDS, CBS_K0_WORDS, 9000, 1ull << 40},  // data_struct.rs:76-81
    {3, {1, 2, 3, 0}, CBS_KF_FIRST_WORDS, CBS_KF_MID_WORDS, CBS_KF_LAST_WORDS, 11000, (1ull << 40) + (1u << 20)},
};
// the seeded generators' deterministic test variant draws the mask seed from this stream of its seed
inline constexpr uint64_t kMaskSeedStream = (1ull << 40) + (2u << 20);
}  // namespace cbs_host

// Host-side key material in the standard domain (flat layouts of include/cbs_b200.h).
struct cbs_keyset {
    std::vector<uint64_t> bsk, ksk, autok, ss, lwe_sk_small, glwe_sk;
};
