/*
 * cbs_b200.h — C ABI of libcbs_b200.so: the B200 (sm_100a) implementation of the server-side hot
 * path of code-perspective/temp-fhe-transciphering (AES-128 transciphering over bit-wise TFHE
 * ciphertexts with the cbs_lib circuit-bootstrapping pipeline, parameter set AES_TIGHT,
 * submission/cbs_lib/src/aes_instances.rs:76-97).
 *
 * The reference has no FFI of its own: its boundary is (1) the stage executables' file contract and
 * (2) cbs_lib's public Rust functions (SURVEY.md 8(b)).  This header is what a Rust `-sys` crate
 * (cc/bindgen) would bind; INTEGRATION.md shows that binding next to each cbs_lib function it
 * replaces.  Plain pointers and sizes only; every call returns 0 on success, non-zero on error
 * (cbs_last_error() gives the message); the caller owns all host buffers, a context owns all device
 * memory; one context may be used from one host thread at a time.  There is NO CPU fallback: every
 * compute entry point fails with CBS_ERR_CUDA if no sm_100 device / kernel image is available.
 *
 * Array layouts (little-endian u64, wrapping arithmetic; same flat layouts the reference's
 * containers hold, SURVEY.md 8(a) row a11):
 *   LWE small   [768 mask][body]                         769 words
 *   LWE big     [2048 mask][body]                        2049 words
 *   GLWE        [2 mask polys][body] x 1024              3072 words
 *   GLEV        [7 levels] GLWE                          21504 words
 *   GGSW        [7 levels][3 rows][3 polys][1024]        64512 words  (level 1 = coarsest first)
 *   bsk         [768][1][3][3][1024]      ksk [8][3][4][256]      ss [2][2][3][3][1024]
 *   auto        [10][2][3][3][1024] standard-domain GLWE keyswitch keys, index i <-> X -> X^((1024>>i)+1)
 *   k10_9       [4 (x9,x11,x13,x14)][16 bytes][2 acc] GLWE
 *   k8_1        [8 (round-1)][4][16][2] GLWE              k0 [16][2] GLWE
 */
#ifndef CBS_B200_H
#define CBS_B200_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CBS_OK          0
#define CBS_ERR_ARG     1
#define CBS_ERR_IO      2
#define CBS_ERR_FORMAT  3
#define CBS_ERR_CUDA    4
#define CBS_ERR_NOMEM   5

#define CBS_LWE_SMALL_WORDS 769
#define CBS_LWE_BIG_WORDS   2049
#define CBS_GLWE_WORDS      3072
#define CBS_GLEV_WORDS      21504
#define CBS_GGSW_WORDS      64512
#define CBS_BSK_WORDS       (768u * 9u * 1024u)
#define CBS_KSK_WORDS       (8u * 3u * 4u * 256u)
#define CBS_AUTO_WORDS      (10u * 2u * 3u * 3u * 1024u)
#define CBS_SS_WORDS        (2u * 2u * 3u * 3u * 1024u)
#define CBS_K10_9_WORDS     (4u * 16u * 2u * 3072u)
#define CBS_K8_1_WORDS      (8u * 4u * 16u * 2u * 3072u)
#define CBS_K0_WORDS        (16u * 2u * 3072u)
#define CBS_KF_FIRST_WORDS  (3u * 16u * 2u * 3072u)
#define CBS_KF_MID_WORDS    (8u * 3u * 16u * 2u * 3072u)
#define CBS_KF_LAST_WORDS   (16u * 2u * 3072u)

typedef struct cbs_keyset cbs_keyset; /* host-side key material, standard domain */
typedef struct cbs_ctx cbs_ctx;       /* one GPU: Fourier-domain keys + workspaces */

const char *cbs_last_error(void);
const char *cbs_version(void);

/* ---------------------------------------------------------------------------------------------
 * Key material and the io/ file formats (bincode 1.3, SURVEY.md 8(b) table).
 * Replaces the deserialisation block of both server mains
 * (src/bin/server_encrypted_aes_decryption.rs:619-643, src/bin/server_encrypted_compute.rs:131-201). */

/* read io_dir/public_keys/{bsk,ksk,auto_keys,ss_key}.bin; with_secret != 0 also reads
 * io_dir/secret_keys/{lwe_sk,glwe_sk}.bin (tests / client side only). */
int cbs_keyset_load_dir(const char *io_dir, int with_secret, cbs_keyset **out);
/* write the same files (auto_keys.bin in the reference's Fourier split-limb form). */
int cbs_keyset_save_dir(const cbs_keyset *ks, const char *io_dir, int with_secret);
/* adopt caller-provided standard-domain arrays (copied). secret keys may be NULL. */
int cbs_keyset_from_arrays(const uint64_t *bsk, const uint64_t *ksk, const uint64_t *auto_std, const uint64_t *ss,
                           const uint64_t *lwe_sk_small /*768 or NULL*/, const uint64_t *glwe_sk /*2048 or NULL*/,
                           cbs_keyset **out);
/* Seeded client-side key generation with the reference's distributions (binary secrets, Gaussian
 * noise; cbs_lib/src/keygen.rs:187-243, src/bin/client_key_generation.rs:20-86).  Client-side helper
 * for tests and benches: the reference's own keygen is unseeded. */
int cbs_keyset_generate(uint64_t seed, cbs_keyset **out);
/* The same generation with secrets, masks and noise drawn from ChaCha20 keyed with 256 bits of getrandom(2): what
 * bin/client_key_generation uses when no seed is given (the harness expects fresh keys on every run,
 * harness/run_submission.py:74-77).  The seeded variant above is deterministic and NOT cryptographically secure. */
int cbs_keyset_generate_os_entropy(cbs_keyset **out);
void cbs_keyset_free(cbs_keyset *ks);
const uint64_t *cbs_keyset_bsk(const cbs_keyset *ks);
const uint64_t *cbs_keyset_ksk(const cbs_keyset *ks);
const uint64_t *cbs_keyset_auto(const cbs_keyset *ks);
const uint64_t *cbs_keyset_ss(const cbs_keyset *ks);
const uint64_t *cbs_keyset_lwe_sk_small(const cbs_keyset *ks); /* NULL if absent */
const uint64_t *cbs_keyset_glwe_sk(const cbs_keyset *ks);      /* NULL if absent; == big LWE key */

/* AllRdKeys (src/data_struct.rs:11-26) <-> flat arrays. */
int cbs_trans_key_load(const char *path, uint64_t *k10_9, uint64_t *k8_1, uint64_t *k0);
int cbs_trans_key_save(const char *path, const uint64_t *k10_9, const uint64_t *k8_1, const uint64_t *k0);
/* client_encode_encrypt equivalent (src/bin/client_encode_encrypt.rs:9-22, src/data_struct.rs:30-269):
 * rounds 10/9 encrypted LUTs, rounds 8..1 and 0 trivial LUTs, for ECB block decryption. */
int cbs_trans_key_generate(const cbs_keyset *ks, const uint8_t aes_key[16], uint64_t seed, uint64_t *k10_9,
                           uint64_t *k8_1, uint64_t *k0);
int cbs_trans_key_generate_os_entropy(const cbs_keyset *ks, const uint8_t aes_key[16], uint64_t *k10_9, uint64_t *k8_1,
                                      uint64_t *k0);
/* Forward-direction transciphering key for CTR mode (SURVEY.md 8(f)1; the harness uses CTR for sizes 1/2,
 * harness/aes_keygen_and_encrypt.py:45-55, which the reference does not implement).  Keyed S-boxes as
 * cbs_lib/src/aes_ref.rs:334-380: kf_first [3 (x1,x2,x3)][16][2] encrypted GLWE LUTs of
 * m*S(x ^ rk0), kf_mid [8 (rounds 2..9)][3][16][2] trivial LUTs of m*S(x ^ rk_{r-1}), kf_last [16][2]
 * trivial LUTs of S(x ^ rk9) ^ rk10 (key byte of the post-ShiftRows position).  Same bincode shape as
 * AllRdKeys with 3-tuples. */
int cbs_fwd_trans_key_generate(const cbs_keyset *ks, const uint8_t aes_key[16], uint64_t seed, uint64_t *kf_first,
                               uint64_t *kf_mid, uint64_t *kf_last);
int cbs_fwd_trans_key_generate_os_entropy(const cbs_keyset *ks, const uint8_t aes_key[16], uint64_t *kf_first, uint64_t *kf_mid,
                                          uint64_t *kf_last);
int cbs_fwd_trans_key_load(const char *path, uint64_t *kf_first, uint64_t *kf_mid, uint64_t *kf_last);
int cbs_fwd_trans_key_save(const char *path, const uint64_t *kf_first, const uint64_t *kf_mid, const uint64_t *kf_last);

/* Seeded transciphering keys: every LUT encrypted, masks expanded from a public seed.
 *   WARNING: the generators above write the middle and last LUTs as trivial GLWE, as the reference does: zero mask, keyed
 *   table in the body, so the top bit of body coefficient i of a LUT is its table bit and anyone holding the key reads the
 *   round keys rk1..rk10 - and from any one of them the AES key.  The seeded keys below encrypt every LUT.
 *   Layout.  GLWE g counts through the direction's AllRdKeys order: first-round LUTs [nmult][16][2], middle [8][nmult][16][2],
 *   last [16][2]; nmult = 4 for the inverse (ECB) key, 3 for the forward (CTR) key: G = 1184 / 896 GLWE.  A seeded key is
 *   mask_seed (32 bytes) + bodies[G][1024] u64 (CBS_TRANS_KEY_SEEDED_WORDS / CBS_FWD_TRANS_KEY_SEEDED_WORDS words, 9.7 / 7.3 MB
 *   against 29.1 / 22.0 MB for the full key).  Mask word w (0..2047) of GLWE g is the RFC 8439 ChaCha20 block with key =
 *   mask_seed as 8 little-endian u32, counter = w / 8, nonce = (g, dir, 0x6b73616d "mask"), dir = 0 inverse / 1 forward:
 *   the u64 out[2i] | out[2i+1] << 32, i = w % 8, after the feed-forward.  Expanded GLWE g = [mask(g)][bodies[g]], word for word
 *   the AllRdKeys layout, so an expanded key goes to every call that takes k10_9/k8_1/k0 (or kf_*).
 *   Security rests on ChaCha20 as a PRF, as tfhe-rs's seeded ciphertexts rest on their CSPRNG.
 *   *_seeded_generate: the same keyed tables as cbs_trans_key_generate / cbs_fwd_trans_key_generate, every LUT a fresh
 *   encryption body = sum mask_c * S_c + e + pt with the noise from the secret stream; the mask seed is an output: from
 *   getrandom(2), apart from the noise key (_os_entropy), or derived from `seed` (deterministic test variant, NOT secure).
 *   *_seeded_expand: the host form of the device expansion: mask_seed + bodies -> the three AllRdKeys arrays.
 *   *_seeded_save / _load: "CBSSEED1", u64 direction, the 32-byte seed, u64 word count, the bodies (56 + 8192 G bytes); load
 *   returns CBS_ERR_FORMAT for another magic, the other direction, another count, a truncated file or trailing bytes.
 *   Null arguments return CBS_ERR_ARG (load: CBS_ERR_IO). */
#define CBS_SEED_BYTES                 32u
#define CBS_TRANS_KEY_SEEDED_WORDS     (1184u * 1024u)
#define CBS_FWD_TRANS_KEY_SEEDED_WORDS (896u * 1024u)
int cbs_trans_key_seeded_generate(const cbs_keyset *ks, const uint8_t aes_key[16], uint64_t seed, uint8_t mask_seed_out[32],
                                  uint64_t *bodies);
int cbs_trans_key_seeded_generate_os_entropy(const cbs_keyset *ks, const uint8_t aes_key[16], uint8_t mask_seed_out[32],
                                             uint64_t *bodies);
int cbs_fwd_trans_key_seeded_generate(const cbs_keyset *ks, const uint8_t aes_key[16], uint64_t seed, uint8_t mask_seed_out[32],
                                      uint64_t *bodies);
int cbs_fwd_trans_key_seeded_generate_os_entropy(const cbs_keyset *ks, const uint8_t aes_key[16], uint8_t mask_seed_out[32],
                                                 uint64_t *bodies);
int cbs_trans_key_seeded_expand(const uint8_t mask_seed[32], const uint64_t *bodies, uint64_t *k10_9, uint64_t *k8_1, uint64_t *k0);
int cbs_fwd_trans_key_seeded_expand(const uint8_t mask_seed[32], const uint64_t *bodies, uint64_t *kf_first, uint64_t *kf_mid,
                                    uint64_t *kf_last);
int cbs_trans_key_seeded_save(const char *path, const uint8_t mask_seed[32], const uint64_t *bodies);
int cbs_trans_key_seeded_load(const char *path, uint8_t mask_seed[32], uint64_t *bodies);
int cbs_fwd_trans_key_seeded_save(const char *path, const uint8_t mask_seed[32], const uint64_t *bodies);
int cbs_fwd_trans_key_seeded_load(const char *path, uint8_t mask_seed[32], uint64_t *bodies);

/* LweCiphertextList<Vec<u64>> result.bin */
int cbs_lwe_list_load(const char *path, uint64_t **data /* malloc'd, free with cbs_free */, uint64_t *count,
                      uint64_t *lwe_words);
int cbs_lwe_list_save(const char *path, const uint64_t *data, uint64_t count, uint64_t lwe_words);
void cbs_free(void *p);
/* client side: decrypt_decode_lwe_list (submission/src/help_fun.rs:12-42), delta = 2^63; sk has n words */
int cbs_lwe_decrypt_bits(const uint64_t *sk, int n, const uint64_t *lwe, uint64_t count, uint64_t *bits_out);
/* client side, packed results (cbs_pack_lwes): glwe [nglwe][3072] under glwe_sk [2][1024] (the big LWE key); coefficient j
 * of GLWE g decrypts to bits_out[g * 1024 + j], delta = 2^63, for the first nbits <= nglwe * 1024 bits */
int cbs_glwe_decrypt_bits(const uint64_t *glwe_sk, const uint64_t *glwe, uint64_t nglwe, uint64_t nbits, uint64_t *bits_out);
/* GlweCiphertextList<Vec<u64>> {data, glwe_size = 3, polynomial_size = 1024, modulus} of nglwe GLWE (the packed result);
 * load malloc's *data (free with cbs_free) and rejects any other glwe_size or polynomial size */
int cbs_glwe_list_save(const char *path, const uint64_t *glwe, uint64_t nglwe);
int cbs_glwe_list_load(const char *path, uint64_t **data, uint64_t *nglwe);
/* bincode Vec<u64>: io/<s>/intermediate/decoded_result{,_aes}.txt */
int cbs_u64_vec_save(const char *path, const uint64_t *data, uint64_t n);
int cbs_u64_vec_load(const char *path, uint64_t **data /* free with cbs_free */, uint64_t *n);
/* encrypt bits (0/1) at delta = 2^63 under the big LWE key (tests / microbench inputs) */
int cbs_encrypt_bits_big(const cbs_keyset *ks, const uint8_t *bits, int count, uint64_t seed, uint64_t *out);
/* ... and under the small (768) key, input format of the blind rotation */
int cbs_encrypt_bits_small(const cbs_keyset *ks, const uint8_t *bits, int count, uint64_t seed, uint64_t *out);

/* ---------------------------------------------------------------------------------------------
 * Device context: uploads the keys, converts them to the Fourier domain ON THE GPU
 * (replaces server_encrypted_aes_decryption.rs:645-687). */
int cbs_device_count(int *count); /* visible CUDA devices (CBS_ERR_CUDA if the driver is absent) */
/* create the CUDA primary context of `device` now (cudaSetDevice + cudaFree(0)) so that a caller can account for
 * driver start-up separately from cbs_ctx_create; optional - cbs_ctx_create does it implicitly otherwise. */
int cbs_device_init(int device);
int cbs_ctx_create(const cbs_keyset *ks, int device, cbs_ctx **out);
void cbs_ctx_destroy(cbs_ctx *ctx);
int cbs_ctx_device(const cbs_ctx *ctx);
/* kernels launched by this context since creation (bench.py's gpu_launches claim) */
uint64_t cbs_ctx_launch_count(const cbs_ctx *ctx);
/* make the context issue its work on an existing CUDA stream (cudaStream_t as void*); NULL = own stream */
int cbs_ctx_set_stream(cbs_ctx *ctx, void *cuda_stream);
int cbs_ctx_synchronize(cbs_ctx *ctx);

/* ---------------------------------------------------------------------------------------------
 * Batched stage entry points, HOST buffers (H2D + kernels + D2H inside the call).
 * Each mirrors one cbs_lib function, applied to `count` independent ciphertexts. */

/* keyswitch_lwe_ciphertext_by_glwe_keyswitch, cbs_lib/src/fourier_glwe_keyswitch.rs:344 */
int cbs_lwe_keyswitch(cbs_ctx *ctx, const uint64_t *in_big, uint64_t *out_small, int count);
/* accumulator + gen_blind_rotate_local_assign, cbs_lib/src/ggsw_conv.rs:250-300, pbs.rs:70 */
int cbs_blind_rotate(cbs_ctx *ctx, const uint64_t *in_small, uint64_t *acc_out, int count);
/* cbs_lib/src/ggsw_conv.rs:302-314 (everything between blind rotation and trace) */
int cbs_glev_from_acc(cbs_ctx *ctx, const uint64_t *acc, uint64_t *glev_out, int count);
/* trace_assign, cbs_lib/src/automorphism.rs:195 — in place on `count` GLWE */
int cbs_trace(cbs_ctx *ctx, uint64_t *glwe_inout, int count);
/* lwe_msb_bit_to_glev_by_trace_with_preprocessing, cbs_lib/src/ggsw_conv.rs:231 */
int cbs_lwe_msb_bit_to_glev(cbs_ctx *ctx, const uint64_t *in_small, uint64_t *glev_out, int count);
/* switch_scheme, cbs_lib/src/ggsw_conv.rs:163 */
int cbs_scheme_switch(cbs_ctx *ctx, const uint64_t *glev, uint64_t *ggsw_out, int count);
/* circuit_bootstrap_lwe_ciphertext_by_trace_with_preprocessing, cbs_lib/src/ggsw_conv.rs:409
 * (output in the standard domain; the Fourier form stays on the device) */
int cbs_circuit_bootstrap(cbs_ctx *ctx, const uint64_t *in_small, uint64_t *ggsw_out, int count);
/* evaluate_8_to_8_cipher_lut, src/bin/server_encrypted_aes_decryption.rs:550: nbytes groups of 8 GGSW
 * bits (LSB first), nluts LUTs per byte, each LUT = 2 GLWE accumulators;
 * out[nbytes][nluts][8] big LWE, bit 4*a + t of accumulator a. */
int cbs_lut8_eval(cbs_ctx *ctx, const uint64_t *ggsw_bits, int nbytes, const uint64_t *luts, int nluts, uint64_t *out);
/* max_of_two, src/bin/server_encrypted_compute.rs:34-98: the CMux ladder of one tree level of cbs_max_u16, on given inputs.
 * ggsw[nvals][16] standard-domain GGSW of the values' bits (MSB first), op[nvals][16] GLWE data operands (cbs_max_u16 takes
 * them from the bootstraps' level-1 GLEV, doubled); pair p = (a_idx[p], b_idx[p]) -> out[npairs][16] big LWE, output bit j
 * of pair p computed with e starting from operand a's bit j (DESIGN.md section 4a).  npairs = 0 returns CBS_OK; negative
 * counts, null pointers and a pair index outside [0, nvals) return CBS_ERR_ARG before anything is queued. */
int cbs_max_of_two(cbs_ctx *ctx, const uint64_t *ggsw, const uint64_t *op, int nvals, const int32_t *a_idx, const int32_t *b_idx,
                   int npairs, uint64_t *out);
/* The gathered LUT ladder of the stage-8 LUT circuits (csrc/host/ip_plan.h) on given inputs.  ggsw[nbits] standard-domain
 * GGSW; job j runs the accumulator luts[lut_index[j]] (luts[nluts] GLWE) through the selectors sel[j][0..7] (selector i
 * rotates by 2^i; -1 = the constant-0 selector, its CMux is skipped) and writes the 4 extractions at 0, 256, 512, 768 to rows
 * out_index[j] .. out_index[j] + 3 of out[nout] big LWE; every other row of out is zero.  njobs = 0 returns CBS_OK; negative
 * counts, null pointers, a selector outside [-1, nbits), a lut_index outside [0, nluts) and an output window outside
 * [0, nout) or overlapping another job's return CBS_ERR_ARG before anything is queued. */
int cbs_lut8_gather_eval(cbs_ctx *ctx, const uint64_t *ggsw, int nbits, const int32_t *sel, const uint64_t *luts, int nluts,
                         const int32_t *lut_index, const int32_t *out_index, int njobs, uint64_t *out, int nout);
/* known_rotate_keyed_lut x4 + he_inv_mix_columns_precomp + he_inv_shift_rows
 * (cbs_lib/src/aes_he.rs:64, server_encrypted_aes_decryption.rs:89-128): first two rounds */
int cbs_aes_first_rounds(cbs_ctx *ctx, const uint8_t *ct, int nblocks, const uint64_t *k10_9, uint64_t *state_out);
/* he_inv_mix_columns_precomp + he_inv_shift_rows on t4 = [4 (x9,x11,x13,x14)][nblocks][128] big LWE */
int cbs_aes_inv_linear(cbs_ctx *ctx, const uint64_t *t4, int nblocks, uint64_t *state_out);

/* aes_to_lwe_trasnciphering, src/bin/server_encrypted_aes_decryption.rs:28-191, for nblocks
 * independent 16-byte ECB blocks.  out[nblocks][128] big LWE, MSB-first inside each byte
 * (the exact payload of ciphertext_aes_download/result.bin).  Synchronous for the caller (all host buffers are free again
 * on return); inside, the round 8..0 LUTs travel on a copy stream while the first rounds and the first blind rotation run. */
int cbs_aes128_transcipher(cbs_ctx *ctx, const uint8_t *ct, int nblocks, const uint64_t *k10_9, const uint64_t *k8_1,
                           const uint64_t *k0, uint64_t *out);
/* CTR-mode transciphering (forward AES on the public counter blocks IV+i, 128-bit big-endian counter as
 * pyaes.Counter; he_sub_bytes_8_to_24 / he_shift_rows / he_mix_columns_precomp, cbs_lib/src/aes_he.rs:285-474),
 * then XOR with the public AES-CTR ciphertext bits.  out, and the overlapped key upload, as cbs_aes128_transcipher. */
int cbs_aes128_ctr_transcipher(cbs_ctx *ctx, const uint8_t *ct, int nblocks, const uint8_t iv[16], const uint64_t *kf_first,
                               const uint64_t *kf_mid, const uint64_t *kf_last, uint64_t *out);
/* stage 8, src/bin/server_encrypted_compute.rs:99-359: encrypted max of nvals 16-bit values
 * (in[nvals][16] big LWE, MSB first) -> out[16] big LWE.  The reference accepts exactly 8 values
 * (sequential fold); any nvals >= 1 is reduced as a balanced tree here. */
int cbs_max_u16(cbs_ctx *ctx, const uint64_t *in, int nvals, uint64_t *out);

/* The same maximum as a LUT circuit (csrc/host/ip_plan.h max_make_plan: nibble comparators, one select ladder per output
 * bit, fresh operands; 55 circuit bootstraps per max_of_two, two bootstrap layers per tree level).  Its output noise
 * (2^58) depends neither on the data nor on the tree depth; cbs_max_u16 switches to it above the reference's 8 values
 * (CBS_MAX_VARIANT=ladder|lut overrides).  cbs_max_plan_check dry-runs the plan on cleartext values (host only). */
int cbs_max_u16_lut(cbs_ctx *ctx, const uint64_t *in, int nvals, uint64_t *out);
int cbs_max_plan_check(const uint16_t *vals, int nvals, uint16_t *result, int64_t *circuit_bootstraps, int *layers,
                       int64_t *lut_ladders);

/* Mini-workload #2 of the harness (harness/cleartext_impl.py:65-70, README.md:43; the reference submission has
 * no implementation): encrypted  sum_i (x_i * y_i mod 2^16) mod 2^16  with x = the first nvals/2 values and
 * y = the second half; in[nvals][16] big LWE (MSB first, the payload of ciphertext_aes_download/result.bin)
 * -> out[16] big LWE (MSB first).  nvals must be even.  Boolean circuit of nibble-product, population-count
 * and nibble-adder LUT ladders over circuit-bootstrapped bits (csrc/host/ip_plan.h). */
int cbs_inner_product_u16(cbs_ctx *ctx, const uint64_t *in, int nvals, uint64_t *out);
/* sum of nvals 16-bit values mod 2^16 (the compression stage of the inner product alone; same formats): combines the
 * per-GPU partial inner products when the pairs are sharded across GPUs (SURVEY.md 8(e)) */
int cbs_sum_u16(cbs_ctx *ctx, const uint64_t *in, int nvals, uint64_t *out);
/* Host-only dry run of the SAME circuit plan on cleartext values (no GPU, no ciphertexts): checks the circuit
 * against the harness formula in the CPU test suite and reports its size.  Any output pointer may be NULL. */
int cbs_inner_product_plan_check(const uint16_t *vals, int nvals, uint16_t *result, int64_t *circuit_bootstraps,
                                 int *layers, int64_t *lut_ladders);

/* ---------------------------------------------------------------------------------------------
 * Device-resident variants (inputs/outputs already in HBM, asynchronous on the context's stream).
 * Used by bench.py's `value` leg and by callers that keep state on the GPU: stage 7 and stage 8 both have one, so
 * transciphered ciphertexts can go on to the mini-workloads without leaving HBM. */
int cbs_trans_key_upload(cbs_ctx *ctx, const uint64_t *k10_9, const uint64_t *k8_1, const uint64_t *k0);
int cbs_aes128_transcipher_dev(cbs_ctx *ctx, const uint8_t *d_ct, int nblocks, uint64_t *d_out);
int cbs_fwd_trans_key_upload(cbs_ctx *ctx, const uint64_t *kf_first, const uint64_t *kf_mid, const uint64_t *kf_last);
/* d_ctr = the nblocks counter blocks (16 bytes each), d_ct = the AES-CTR ciphertext bytes */
int cbs_aes128_ctr_transcipher_dev(cbs_ctx *ctx, const uint8_t *d_ctr, const uint8_t *d_ct, int nblocks, uint64_t *d_out);
/* Seeded keys (above) -> the device: the bodies are copied into the LUT buffers and the masks expanded there from the seed
 * (k_expand_lut_masks), so only the 9.7 / 7.3 MB of bodies cross the bus; the device key is then word for word the
 * *_seeded_expand arrays, and the *_transcipher_dev calls run with it unchanged.  Synchronous like cbs_trans_key_upload (the
 * host buffers are free on return); a later upload of either form of the same direction replaces it. */
int cbs_trans_key_seeded_upload(cbs_ctx *ctx, const uint8_t mask_seed[32], const uint64_t *bodies);
int cbs_fwd_trans_key_seeded_upload(cbs_ctx *ctx, const uint8_t mask_seed[32], const uint64_t *bodies);

/* Key slots: many transciphering keys resident at once (one per AES sender), and one call over blocks of many keys.
 *   Each direction has a pool of slots; a slot holds one key in the expanded AllRdKeys layout (29.1 MB inverse, 22.0 MB
 *   forward).  Every slot is under the context's one FHE keyset: slots separate AES senders, not FHE clients.
 *   *_slots_reserve: the pool gets nslots contiguous slots.  A later reserve with a larger count grows it and keeps every
 *   uploaded slot (device-to-device copy on the context's stream; the old buffers are freed stream-ordered).  The same count
 *   does nothing; a smaller count or nslots <= 0 returns CBS_ERR_ARG; a failed allocation returns CBS_ERR_NOMEM and leaves
 *   the pool as it was.
 *   *_slot_upload / *_seeded_slot_upload: put a key of either form into a reserved slot (slot < 0 or >= the reserved count:
 *   CBS_ERR_ARG), replacing what it held.  Synchronous like cbs_trans_key_upload, and ordered after earlier work of the
 *   context that may still read the slot.  Slots and the single key of cbs_trans_key_upload and its twins are independent:
 *   neither kind of upload changes what the other kind of call computes.
 *   *_transcipher_slots_dev: block b is transciphered under slot slots[b].  slots is a HOST array [nblocks]; d_ct (ECB), d_ctr
 *   and d_ct (CTR) and d_out [nblocks][128] big LWE are as in the single-key _dev calls, and block b's rows are bit for bit
 *   the rows the single-key call gives for that block under that key.  The slot array is checked before anything is queued:
 *   a slot < 0, >= the reserved count, or never uploaded in the call's direction, nblocks <= 0 or a null pointer returns
 *   CBS_ERR_ARG.  Queued on the context's stream, never synchronises; the slot array is copied before the call returns, so
 *   the queued work reads no host memory.
 *   *_transcipher_slots: host buffers (ct, ctr = the nblocks counter blocks [nblocks][16], out [nblocks][128] big LWE);
 *   synchronous: the inputs go up, the _dev call runs, the rows come down. */
int cbs_trans_key_slots_reserve(cbs_ctx *ctx, int nslots);
int cbs_fwd_trans_key_slots_reserve(cbs_ctx *ctx, int nslots);
int cbs_trans_key_slot_upload(cbs_ctx *ctx, int slot, const uint64_t *k10_9, const uint64_t *k8_1, const uint64_t *k0);
int cbs_fwd_trans_key_slot_upload(cbs_ctx *ctx, int slot, const uint64_t *kf_first, const uint64_t *kf_mid, const uint64_t *kf_last);
int cbs_trans_key_seeded_slot_upload(cbs_ctx *ctx, int slot, const uint8_t mask_seed[32], const uint64_t *bodies);
int cbs_fwd_trans_key_seeded_slot_upload(cbs_ctx *ctx, int slot, const uint8_t mask_seed[32], const uint64_t *bodies);
int cbs_aes128_transcipher_slots_dev(cbs_ctx *ctx, const uint8_t *d_ct, const int32_t *slots, int nblocks, uint64_t *d_out);
int cbs_aes128_ctr_transcipher_slots_dev(cbs_ctx *ctx, const uint8_t *d_ctr, const uint8_t *d_ct, const int32_t *slots,
                                         int nblocks, uint64_t *d_out);
int cbs_aes128_transcipher_slots(cbs_ctx *ctx, const uint8_t *ct, const int32_t *slots, int nblocks, uint64_t *out);
int cbs_aes128_ctr_transcipher_slots(cbs_ctx *ctx, const uint8_t *ctr, const uint8_t *ct, const int32_t *slots, int nblocks,
                                     uint64_t *out);

/* Stage 8 on device buffers: the same computations and results as cbs_max_u16, cbs_max_u16_lut, cbs_sum_u16 and
 * cbs_inner_product_u16, bit for bit.
 *   Layout: d_in [nvals][16] big LWE (MSB first), d_out [16] big LWE.  The transcipher output [nblocks][128] big LWE is
 *   [8*nblocks][16], so a *_transcipher_dev output buffer can be passed as it is.
 *   cbs_max_u16_dev picks the ladder or the LUT circuit by the same rule as cbs_max_u16, CBS_MAX_VARIANT included.
 *   The inner product takes x and y from separate buffers, d_x [npairs][16] and d_y [npairs][16] big LWE, so npairs may be
 *   odd; cbs_inner_product_u16_dev(ctx, X, X + npairs*16*2049, npairs, out) equals cbs_inner_product_u16(ctx, X, 2*npairs, out).
 *   Asynchronous: the work is queued on the context's stream (cbs_ctx_set_stream) behind earlier work of the context,
 *   lanes of a *_transcipher_dev call included, so its output can be passed on without synchronising; the call
 *   synchronises neither the stream nor the device, and once it returns the queued work reads no host memory.
 *   Counts <= 0, null pointers and a d_out that overlaps an input range return CBS_ERR_ARG. */
int cbs_max_u16_dev(cbs_ctx *ctx, const uint64_t *d_in, int nvals, uint64_t *d_out);
int cbs_max_u16_lut_dev(cbs_ctx *ctx, const uint64_t *d_in, int nvals, uint64_t *d_out);
int cbs_sum_u16_dev(cbs_ctx *ctx, const uint64_t *d_in, int nvals, uint64_t *d_out);
int cbs_inner_product_u16_dev(cbs_ctx *ctx, const uint64_t *d_x, const uint64_t *d_y, int npairs, uint64_t *d_out);

/* LWE-to-GLWE packing (Chen-Dai-Kim-Song 2020; cbs_lib glwe_conv.rs pack_lwes): count big LWE bits at delta = 2^63
 * -> ceil(count / 1024) GLWE, 3072 words each instead of 1024 x 2049.  Input i goes to GLWE i / 1024, where coefficient
 * i % 1024 decrypts to its bit (cbs_glwe_decrypt_bits); the coefficients past count in the last GLWE decrypt to 0.
 *   Tree of 10 levels, stride s = 1024 >> L, kappa = 2^L + 1 (the trace's automorphism keys, nothing new from the client):
 *   p[j] = const_embed(lwe_j >> 10), then q[t] = (p[t] + X^s p[t+s]) + keyswitch(auto, (p[t] - X^s p[t+s])(X^kappa)) for
 *   t < s.  A group of c inputs costs sum_L min(c, s) keyswitches (10 for one input, 1023 for 1024) and gives the same
 *   words as the same inputs padded with zero rows.  Packed bits decrypt with the input's noise plus at most about 2^41.
 *   cbs_pack_lwes: host buffers in_big [count][2049], glwe_out [ceil(count/1024)][3072]; synchronous; count 0 does nothing.
 *   cbs_pack_lwes_dev: device buffers of the same layouts, so a *_transcipher_dev output ([nblocks][128] big LWE,
 *   count = 128 nblocks) can be passed as it is; queued on the context's stream behind earlier work (lanes of a
 *   *_transcipher_dev call included), never synchronises; count <= 0, null pointers and a d_out that overlaps d_in
 *   return CBS_ERR_ARG. */
int cbs_pack_lwes(cbs_ctx *ctx, const uint64_t *in_big, int count, uint64_t *glwe_out);
int cbs_pack_lwes_dev(cbs_ctx *ctx, const uint64_t *d_in, int count, uint64_t *d_out);

int cbs_circuit_bootstrap_dev(cbs_ctx *ctx, const uint64_t *d_in_small, int count);  /* GGSW stays in the workspace */
int cbs_blind_rotate_dev(cbs_ctx *ctx, const uint64_t *d_in_small, uint64_t *d_acc_out, int count);
/* measured FP64 FMA throughput of the device (roofline denominator of the FFT kernels) */
int cbs_measure_fp64_tflops(cbs_ctx *ctx, double *tflops);
/* plain device buffers for callers without their own allocator */
int cbs_dev_alloc(cbs_ctx *ctx, size_t bytes, void **dptr);
int cbs_dev_free(cbs_ctx *ctx, void *dptr);
int cbs_dev_upload(cbs_ctx *ctx, void *dptr, const void *host, size_t bytes);
int cbs_dev_download(cbs_ctx *ctx, void *host, const void *dptr, size_t bytes);

#ifdef __cplusplus
}
#endif
#endif
