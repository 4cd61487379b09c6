// cbs_api.cu — device context, workspaces and the compute entry points of include/cbs_b200.h.
//
// Orchestration mirrors the reference's server mains, batched over all ciphertexts of all blocks:
//   stage 7  src/bin/server_encrypted_aes_decryption.rs:28-191  (aes_to_lwe_trasnciphering)
//   stage 8  src/bin/server_encrypted_compute.rs:99-359
// Everything is enqueued on one CUDA stream; there is no host synchronisation inside a
// transciphering call except the final download in the host-buffer variants.
#include "cbs_b200.h"
#include "cbs_kernels.cuh"
#include "fft_tables.h"
#include "host/host_common.h"

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "host/ip_plan.h"

using namespace cbs;
using cbs_host::AesDir;
using cbs_host::kAesDirs;
using cbs_host::kAesFwd;
using cbs_host::kAesInv;
using cbs_host::set_error;

namespace {

struct DevBuf {
    void *p = nullptr;
    size_t bytes = 0;
};

// A host-planned LUT circuit (host/ip_plan.h) compiled for one value count by lut_plan_get and executed by run_lut_plan:
// the launch schedule stays on the host, the index tables live on the device.
struct PlanBatch {
    int idx_off, m, job_off, njobs, ref_off, nref;
};
struct PlanLayer {
    int pre_off, npre, post_off, npost;
    std::vector<PlanBatch> batches;
};
struct LutPlanExec {
    int nvals = 0;  // value count the entry was built for (0: none)
    int nin_bits = 0, pool_size = 0, max_m = 1;
    std::vector<PlanLayer> layers;
    int *d_tab = nullptr;  // one allocation holding the tables below, in this order
    const int *idx = nullptr, *sel = nullptr, *lut = nullptr, *out = nullptr, *add = nullptr, *ref = nullptr;
    int final_idx = 0;  // offset in idx of the 16 result rows, MSB first
};
enum PlanKind { kPlanInnerProduct, kPlanSum, kPlanMax, kNumPlanKinds };

}  // namespace

struct cbs_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    uint64_t launches = 0;
    DeviceKeys K{};
    std::vector<void *> key_allocs;
    // transciphering keys per direction (AesDir): device LUTs of the first, middle and last rounds (host_common.h kAesDirs)
    struct AesKeys {
        uint64_t *first = nullptr, *mid = nullptr, *last = nullptr;
        bool uploaded = false;
    } aes[2];
    // [dir]: 0 = every mask word of the direction's middle and last LUTs is zero (always true for AllRdKeys written by the
    // reference, src/data_struct.rs:145-151,258-263); set by k_masks_nonzero at upload, enables the first-CMux shortcut
    int *d_masks_nonzero = nullptr;
    // key slots per direction (cbs_trans_key_slots_reserve): `n` transciphering keys side by side, first [n][nmult][16][2],
    // mid [n][8][nmult][16][2], last [n][16][2] GLWE (each slot in the single-key buffers' layout), flags[n] = that slot's
    // k_masks_nonzero result; a slot is read only once `uploaded[slot]` is set
    struct KeySlots {
        uint64_t *first = nullptr, *mid = nullptr, *last = nullptr;
        int *flags = nullptr;
        int n = 0;
        std::vector<bool> uploaded;
    } slots[2];
    std::map<std::string, DevBuf> ws;
    int chunk_blocks = 64;
    // circuit bootstraps per sub-batch of a stage-8 LUT-circuit layer (bounds the Fourier GGSW workspace to 4.2 GB at
    // the default; CBS_PLAN_CAP lowers it so that small inputs take the sub-batch path too)
    int plan_cap = 8192;
    // Lanes: a chunk is processed as up to kMaxLanes block-aligned parts on separate side streams so that
    // the second (partial) wave of one part's blind rotation overlaps the trace / scheme switch / LUT
    // kernels of another part.  lane = -1: work is issued on `stream` with un-prefixed workspaces.
    static constexpr int kMaxLanes = 4;
    int lanes = 2;
    int lane = -1;
    cudaStream_t side[kMaxLanes] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[kMaxLanes] = {nullptr, nullptr, nullptr, nullptr};
    // block count the LUT job tables of [lane + 1][nmult] were built for (0: none)
    int jobs_nblocks[kMaxLanes + 1][5] = {};
    // end-to-end calls upload the middle and last LUTs (ECB 26 MB) on a copy stream while the first rounds and the first
    // blind rotation already run; the first middle-round LUT launch of every lane waits for ev_keys
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_keys = nullptr, ev_copy_after = nullptr;
    bool keys_in_flight = false;
    // stage-8 circuits: one compiled plan per kind (rebuilt when the count changes, so a repeated call uploads nothing),
    // the trivial LUT accumulators of ip_plan.h's tables (uploaded once), and the ladder max's pair tables, which hold
    // (2i, 2i+1) for i < ladder_pairs in the "max_a" / "max_b" workspaces
    LutPlanExec plans[kNumPlanKinds];
    uint64_t *d_plan_luts = nullptr;
    int ladder_pairs = 0;
};

namespace {

#define CUDA_TRY(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess) {                                                                         \
            set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                               \
            return CBS_ERR_CUDA;                                                                         \
        }                                                                                                \
    } while (0)

int check_launch(const char *what)
{
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error(std::string(what) + ": " + cudaGetErrorString(e));
        return CBS_ERR_CUDA;
    }
    return CBS_OK;
}

// stream the current lane issues on
inline cudaStream_t S(const cbs_ctx *ctx) { return ctx->lane >= 0 ? ctx->side[ctx->lane] : ctx->stream; }

int ws_get(cbs_ctx *ctx, const char *name, size_t bytes, void **out)
{
    DevBuf &b = ctx->ws[ctx->lane >= 0 ? std::string("lane") + std::to_string(ctx->lane) + ":" + name : std::string(name)];
    if (b.bytes < bytes) {
        // stream-ordered growth (no device-wide synchronisation inside a compute call): a workspace is only ever used on
        // the stream of the lane that owns it, so freeing and re-allocating on that stream orders correctly with its work;
        // the device's default pool keeps freed blocks (release threshold set in cbs_ctx_create)
        cudaStream_t st = S(ctx);
        if (b.p) {
            CUDA_TRY(cudaFreeAsync(b.p, st));
            b.p = nullptr;
            b.bytes = 0;
        }
        CUDA_TRY(cudaMallocAsync(&b.p, bytes, st));
        b.bytes = bytes;
    }
    *out = b.p;
    return CBS_OK;
}

template <typename T>
int ws_typed(cbs_ctx *ctx, const char *name, size_t count, T **out)
{
    void *p = nullptr;
    int rc = ws_get(ctx, name, count * sizeof(T), &p);
    *out = static_cast<T *>(p);
    return rc;
}

int key_alloc(cbs_ctx *ctx, size_t bytes, void **out)
{
    CUDA_TRY(cudaMalloc(out, bytes));
    ctx->key_allocs.push_back(*out);
    return CBS_OK;
}

struct Activate {
    int prev = -1;
    bool ok = true;
    explicit Activate(const cbs_ctx *ctx)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (cudaSetDevice(ctx->device) != cudaSuccess) ok = false;
    }
    ~Activate()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

#define ENTER(ctx)                                           \
    if (!(ctx)) {                                            \
        set_error("null context");                           \
        return CBS_ERR_ARG;                                  \
    }                                                        \
    Activate _act(ctx);                                      \
    if (!_act.ok) {                                          \
        set_error("cudaSetDevice failed");                   \
        return CBS_ERR_CUDA;                                 \
    }

int upload(cbs_ctx *ctx, void *d, const void *h, size_t bytes)
{
    CUDA_TRY(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return CBS_OK;
}
int download(cbs_ctx *ctx, void *h, const void *d, size_t bytes)
{
    CUDA_TRY(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return CBS_OK;
}

#define TRY(expr)                  \
    do {                           \
        int _rc = (expr);          \
        if (_rc != CBS_OK) return _rc; \
    } while (0)

// ---- device pipelines (all pointers device, async on S(ctx)) ----

int dev_keyswitch(cbs_ctx *ctx, const uint64_t *d_in, uint64_t *d_out, int count)
{
    launch_lwe_keyswitch(ctx->K, d_in, d_out, count, S(ctx));
    ctx->launches++;
    return check_launch("k_lwe_keyswitch");
}

int dev_blind_rotate(cbs_ctx *ctx, const uint64_t *d_in, uint64_t *d_acc, int count)
{
    launch_blind_rotate(ctx->K, d_in, d_acc, count, S(ctx));
    ctx->launches++;
    return check_launch("k_blind_rotate");
}

// lwe_msb_bit_to_glev_by_trace_with_preprocessing for `count` small LWE -> glev[count][7][3072]
int dev_msb_to_glev(cbs_ctx *ctx, const uint64_t *d_in, uint64_t *d_glev, int count)
{
    uint64_t *d_acc;
    TRY(ws_typed(ctx, "acc", (size_t)count * kGlweWords, &d_acc));
    TRY(dev_blind_rotate(ctx, d_in, d_acc, count));
    launch_trace(ctx->K, d_acc, d_glev, count * kCbsLevel, 1, S(ctx));
    ctx->launches++;
    return check_launch("k_trace");
}

// full circuit bootstrap: small LWE -> GGSW (Fourier and/or standard)
int dev_circuit_bootstrap(cbs_ctx *ctx, const uint64_t *d_in, uint64_t *d_ggsw_std, double *d_ggsw_f, int count)
{
    uint64_t *d_glev;
    TRY(ws_typed(ctx, "glev", (size_t)count * kGlevWords, &d_glev));
    TRY(dev_msb_to_glev(ctx, d_in, d_glev, count));
    launch_scheme_switch(ctx->K, d_glev, d_ggsw_std, d_ggsw_f, count, S(ctx));
    ctx->launches++;
    return check_launch("k_scheme_switch");
}

// 8-bit LUT ladders (a7); masks_nonzero = the device flag of the LUTs' direction, nullptr if not known
int dev_lut8(cbs_ctx *ctx, const double *ggsw_f, const uint64_t *luts, const int *lut_index, const int *out_index, uint64_t *out,
             int njobs, int accs_per_byte, const int *masks_nonzero)
{
    if (launch_lut8(ctx->K, ggsw_f, luts, lut_index, out_index, out, njobs, accs_per_byte, masks_nonzero, S(ctx))) {
        set_error("k_lut8_v2: " + std::to_string(njobs) + " jobs are not a whole number of bytes of " + std::to_string(accs_per_byte) +
                  " accumulators");
        return CBS_ERR_ARG;
    }
    ctx->launches++;
    return check_launch("k_lut8_v2");
}

// LUT job tables of nb blocks with nmult LUTs per byte (4: inverse middle rounds, 3: forward middle rounds, 1: last round):
// job (blk, byte, m, a) runs accumulator a of LUT (m, byte) and writes its 4 LWE to row (m, blk, byte*8 + 4a) of the
// [nmult][nb][128] state.  Cached per lane and nmult, so repeated calls at one block count rebuild nothing.
int job_tables(cbs_ctx *ctx, int nb, int nmult, int **lut, int **out)
{
    const int n = nb * 16 * nmult * 2;
    const std::string jobs = std::to_string(nmult * 8);
    TRY(ws_typed(ctx, ("job_lut" + jobs).c_str(), (size_t)n, lut));
    TRY(ws_typed(ctx, ("job_out" + jobs).c_str(), (size_t)n, out));
    int &built = ctx->jobs_nblocks[ctx->lane + 1][nmult];
    if (built == nb) return CBS_OK;
    std::vector<int> l(n), o(n);
    for (int blk = 0; blk < nb; blk++)
        for (int byte = 0; byte < 16; byte++)
            for (int m = 0; m < nmult; m++)
                for (int a = 0; a < 2; a++) {
                    const int job = ((blk * 16 + byte) * nmult + m) * 2 + a;
                    l[job] = (m * 16 + byte) * 2 + a;
                    o[job] = (m * nb + blk) * 128 + byte * 8 + 4 * a;
                }
    CUDA_TRY(cudaMemcpyAsync(*lut, l.data(), sizeof(int) * n, cudaMemcpyHostToDevice, S(ctx)));
    CUDA_TRY(cudaMemcpyAsync(*out, o.data(), sizeof(int) * n, cudaMemcpyHostToDevice, S(ctx)));
    CUDA_TRY(cudaStreamSynchronize(S(ctx)));  // host vectors go out of scope
    built = nb;
    return CBS_OK;
}

// One chunk of nb blocks through the AES rounds of direction `dir`.  Inverse (ECB, aes_to_lwe_trasnciphering,
// server_encrypted_aes_decryption.rs:89-189): rounds 10 + 9 on the public ciphertext blocks d_in, rounds 8..1, the last
// round and the per-byte bit reversal.  Forward (CTR, aes_he.rs:285-474): round 1 on the public counter blocks d_in,
// rounds 2..9, the last round, then XOR with the public CTR ciphertext d_ct.
//
// The key a call reads.  One key: the direction's buffers, flags = its device trivial-LUT flag, slots = nullptr.  Key slots: the
// direction's slot pool, flags = its per-slot flags, slots = the device slot table of the blocks (in dev_aes_part: of the part's
// first block); the part then builds its LUT index tables and its trivial-LUT flag on the device (k_slot_lut_index).
struct AesKeyView {
    const uint64_t *first, *mid, *last;
    const int *flags;
    const int *slots;
};

int dev_aes_part(cbs_ctx *ctx, AesDir dir, const AesKeyView &key, const uint8_t *d_in, const uint8_t *d_ct, int nb, uint64_t *d_out)
{
    const int nmult = kAesDirs[dir].nmult, B = nb * 128;
    const bool inv = dir == kAesInv;
    const int *masks_nonzero = key.flags;
    uint64_t *d_t, *d_st, *d_ks;
    double *d_ggsw_f;
    int *lut_m, *out_m, *lut_1, *out_1;
    TRY(ws_typed(ctx, "t4", (size_t)4 * B * kLweBig, &d_t));
    TRY(ws_typed(ctx, "st", (size_t)B * kLweBig, &d_st));
    TRY(ws_typed(ctx, "ks", (size_t)B * kLweSmall, &d_ks));
    TRY(ws_typed(ctx, "ggsw_f", (size_t)B * kGgswWords, &d_ggsw_f));
    TRY(job_tables(ctx, nb, nmult, &lut_m, &out_m));
    TRY(job_tables(ctx, nb, 1, &lut_1, &out_1));
    if (key.slots) {
        // the out-index tables are the single key's; the LUT indices and the trivial-LUT flag follow the blocks' slots
        int *flag;
        TRY(ws_typed(ctx, "slot_lut_m", (size_t)nb * 16 * nmult * 2, &lut_m));
        TRY(ws_typed(ctx, "slot_lut_1", (size_t)nb * 16 * 2, &lut_1));
        TRY(ws_typed(ctx, "slot_flag", 1, &flag));
        launch_slot_lut_index(key.slots, nb, nmult, key.flags, lut_m, lut_1, flag, S(ctx));
        ctx->launches++;
        TRY(check_launch("k_slot_lut_index"));
        masks_nonzero = flag;
    }
    auto linear = [&]() { inv ? launch_inv_linear(d_t, d_st, nb, S(ctx)) : launch_fwd_linear(d_t, d_st, nb, S(ctx)); };
    // first round(s): the input block is public, so the keyed LUTs are "rotated" by sample extraction
    launch_known_rotate(d_in, key.first, d_t, nb, nmult, inv, key.slots, S(ctx));
    linear();
    ctx->launches += 2;
    TRY(check_launch("first rounds"));
    for (int i = 0; i < 8; i++) {
        TRY(dev_keyswitch(ctx, d_st, d_ks, B));
        TRY(dev_circuit_bootstrap(ctx, d_ks, nullptr, d_ggsw_f, B));
        // middle block r is keyed with round key r + 1: decryption runs the blocks from the last one down
        const uint64_t *luts = key.mid + (size_t)(inv ? 7 - i : i) * nmult * 16 * 2 * kGlweWords;
        if (ctx->keys_in_flight && i == 0) CUDA_TRY(cudaStreamWaitEvent(S(ctx), ctx->ev_keys, 0));
        TRY(dev_lut8(ctx, d_ggsw_f, luts, lut_m, out_m, d_t, nb * 16 * nmult * 2, nmult * 2, masks_nonzero));
        linear();
        ctx->launches++;
        TRY(check_launch("round"));
    }
    TRY(dev_keyswitch(ctx, d_st, d_ks, B));
    TRY(dev_circuit_bootstrap(ctx, d_ks, nullptr, d_ggsw_f, B));
    TRY(dev_lut8(ctx, d_ggsw_f, key.last, lut_1, out_1, d_st, nb * 16 * 2, 2, masks_nonzero));
    inv ? launch_reverse_bits(d_st, d_out, nb, S(ctx)) : launch_ctr_finish(d_st, d_ct, d_out, nb, S(ctx));
    ctx->launches++;
    return check_launch("last round");
}

// Run `part(lane_index, first_block, block_count)` over a chunk split into block-aligned lanes on the side
// streams, forked from and joined back into ctx->stream with events (no host synchronisation).
template <typename Fn>
int run_in_lanes(cbs_ctx *ctx, int nb, Fn part)
{
    const int P = std::max(1, std::min(std::min(ctx->lanes, (int)cbs_ctx::kMaxLanes), nb));
    if (P == 1) return part(0, nb);
    CUDA_TRY(cudaEventRecord(ctx->ev_fork, ctx->stream));
    int rc = CBS_OK;
    for (int l = 0; l < P && rc == CBS_OK; l++) {
        const int b0 = (int)((long)nb * l / P), b1 = (int)((long)nb * (l + 1) / P);
        CUDA_TRY(cudaStreamWaitEvent(ctx->side[l], ctx->ev_fork, 0));
        ctx->lane = l;
        rc = part(b0, b1 - b0);
        ctx->lane = -1;
        if (rc != CBS_OK) break;
        CUDA_TRY(cudaEventRecord(ctx->ev_join[l], ctx->side[l]));
        CUDA_TRY(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[l], 0));
    }
    return rc;
}

// nblocks blocks in chunks of chunk_blocks, each split into lanes; d_ct is nullptr for the inverse direction
int dev_aes(cbs_ctx *ctx, AesDir dir, const AesKeyView &key, const uint8_t *d_in, const uint8_t *d_ct, int nblocks, uint64_t *d_out)
{
    for (int c0 = 0; c0 < nblocks; c0 += ctx->chunk_blocks) {
        auto part = [&](int b0, int n) {
            const size_t b = (size_t)c0 + b0;
            AesKeyView k = key;
            if (k.slots) k.slots += b;
            return dev_aes_part(ctx, dir, k, d_in + b * 16, d_ct ? d_ct + b * 16 : nullptr, n, d_out + b * 128 * kLweBig);
        };
        TRY(run_in_lanes(ctx, std::min(ctx->chunk_blocks, nblocks - c0), part));
    }
    return CBS_OK;
}

// dev_aes under the direction's single key (cbs_trans_key_upload and its twins)
int dev_aes_single(cbs_ctx *ctx, AesDir dir, const uint8_t *d_in, const uint8_t *d_ct, int nblocks, uint64_t *d_out)
{
    const cbs_ctx::AesKeys &k = ctx->aes[dir];
    if (!k.uploaded) {
        set_error(dir == kAesInv ? "transciphering key not uploaded (cbs_trans_key_upload)"
                                 : "forward transciphering key not uploaded (cbs_fwd_trans_key_upload)");
        return CBS_ERR_ARG;
    }
    return dev_aes(ctx, dir, {k.first, k.mid, k.last, ctx->d_masks_nonzero + dir, nullptr}, d_in, d_ct, nblocks, d_out);
}

// Every block's slot must be reserved and uploaded in direction `dir`: checked on the host before anything is queued, so no
// unchecked slot value reaches a kernel.  The checked table is returned in `table` for the device copy.
int check_slots(const cbs_ctx *ctx, AesDir dir, const int32_t *slots, int nblocks, const char *what, std::vector<int> *table)
{
    const cbs_ctx::KeySlots &P = ctx->slots[dir];
    table->resize(nblocks);
    for (int b = 0; b < nblocks; b++) {
        const int s = slots[b];
        if (s < 0 || s >= P.n || !P.uploaded[s]) {
            set_error(std::string(what) + ": block " + std::to_string(b) + " names slot " + std::to_string(s) +
                      (s < 0 || s >= P.n ? ", outside the " + std::to_string(P.n) + " reserved slots" : ", which holds no key"));
            return CBS_ERR_ARG;
        }
        (*table)[b] = s;
    }
    return CBS_OK;
}

// dev_aes under key slots: block b under slot slots[b] (host array).  The table goes to the device from a pageable host copy,
// and cudaMemcpyAsync returns once pageable memory is staged, so the queued work reads no host memory after the return.
int dev_aes_slots(cbs_ctx *ctx, AesDir dir, const uint8_t *d_in, const uint8_t *d_ct, const int32_t *slots, int nblocks,
                  uint64_t *d_out, const char *what)
{
    std::vector<int> table;
    TRY(check_slots(ctx, dir, slots, nblocks, what, &table));
    int *d_slots;
    TRY(ws_typed(ctx, "slot_table", (size_t)nblocks, &d_slots));
    CUDA_TRY(cudaMemcpyAsync(d_slots, table.data(), sizeof(int) * nblocks, cudaMemcpyHostToDevice, ctx->stream));
    const cbs_ctx::KeySlots &P = ctx->slots[dir];
    return dev_aes(ctx, dir, {P.first, P.mid, P.last, P.flags, d_slots}, d_in, d_ct, nblocks, d_out);
}

// Uploads direction `dir`'s transciphering key and answers "are its middle and last LUTs trivial?" on the device, right behind
// the copies (k_masks_nonzero; a host scan of them would sit on the critical path).  overlap = false: all on the compute stream,
// synchronised before returning, so the caller owns the host buffers again.  overlap = true: the first-round LUTs go on the
// compute stream; the middle and last LUTs, first read by the ladders of the first middle round (one keyswitch + blind rotation,
// >= 2.4 ms, into the call), go with the check on the copy stream, and ev_keys marks their end.  The caller then sets
// keys_in_flight for dev_aes_part and orders the compute stream after ev_keys before it releases the host buffers.
int aes_key_alloc(cbs_ctx *ctx, AesDir dir)
{
    const cbs_host::AesDirDesc &d = kAesDirs[dir];
    cbs_ctx::AesKeys &key = ctx->aes[dir];
    // each buffer on its own: a failed allocation leaves its pointer null and the next call retries it
    if (!key.first) CUDA_TRY(cudaMalloc(&key.first, (size_t)d.first_words * 8));
    if (!key.mid) CUDA_TRY(cudaMalloc(&key.mid, (size_t)d.mid_words * 8));
    if (!key.last) CUDA_TRY(cudaMalloc(&key.last, (size_t)d.last_words * 8));
    return CBS_OK;
}

// Where an upload writes one key of direction `dir`: the direction's single-key buffers and flag, or one key slot's parts
struct AesKeyDst {
    uint64_t *first, *mid, *last;
    int *flag;
};

AesKeyDst single_key_dst(cbs_ctx *ctx, AesDir dir)
{
    cbs_ctx::AesKeys &k = ctx->aes[dir];
    return {k.first, k.mid, k.last, ctx->d_masks_nonzero + dir};
}

AesKeyDst slot_dst(cbs_ctx *ctx, AesDir dir, int slot)
{
    const cbs_host::AesDirDesc &d = kAesDirs[dir];
    cbs_ctx::KeySlots &P = ctx->slots[dir];
    return {P.first + (size_t)slot * d.first_words, P.mid + (size_t)slot * d.mid_words, P.last + (size_t)slot * d.last_words,
            P.flags + slot};
}

// the key's device flag: 1 if a mask word of its middle or last LUTs is non-zero, queued on `cs`
int aes_key_check_masks(AesDir dir, const AesKeyDst &key, cudaStream_t cs)
{
    const cbs_host::AesDirDesc &d = kAesDirs[dir];
    CUDA_TRY(cudaMemsetAsync(key.flag, 0, sizeof(int), cs));
    launch_masks_nonzero(key.mid, 8 * d.nmult * 16 * 2, key.flag, cs);
    launch_masks_nonzero(key.last, 16 * 2, key.flag, cs);
    return CBS_OK;
}

int aes_key_write(cbs_ctx *ctx, AesDir dir, const AesKeyDst &key, const uint64_t *first, const uint64_t *mid, const uint64_t *last,
                  bool overlap)
{
    const cbs_host::AesDirDesc &d = kAesDirs[dir];
    cudaStream_t cs = ctx->stream;
    if (overlap) {
        if (!ctx->copy_stream) {
            CUDA_TRY(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
            CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_keys, cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_copy_after, cudaEventDisableTiming));
        }
        // the copy must not overtake earlier work on the compute stream that may still read the old keys
        CUDA_TRY(cudaEventRecord(ctx->ev_copy_after, ctx->stream));
        CUDA_TRY(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy_after, 0));
        cs = ctx->copy_stream;
    }
    CUDA_TRY(cudaMemcpyAsync(key.mid, mid, (size_t)d.mid_words * 8, cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaMemcpyAsync(key.last, last, (size_t)d.last_words * 8, cudaMemcpyHostToDevice, cs));
    TRY(aes_key_check_masks(dir, key, cs));
    if (overlap) CUDA_TRY(cudaEventRecord(ctx->ev_keys, cs));
    TRY(upload(ctx, key.first, first, (size_t)d.first_words * 8));
    if (!overlap) CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return CBS_OK;
}

int aes_key_upload(cbs_ctx *ctx, AesDir dir, const uint64_t *first, const uint64_t *mid, const uint64_t *last, bool overlap)
{
    TRY(aes_key_alloc(ctx, dir));
    TRY(aes_key_write(ctx, dir, single_key_dst(ctx, dir), first, mid, last, overlap));
    ctx->aes[dir].uploaded = true;
    return CBS_OK;
}

// Seeded key (include/cbs_b200.h) of direction `dir`: the bodies go into words 2048..3071 of every LUT GLWE (three strided
// copies, one per key buffer), k_expand_lut_masks writes words 0..2047, and the same mask check as aes_key_upload follows (the
// expanded masks are not zero, so the LUT ladders run their full first CMux).  On the compute stream, synchronised.
int aes_key_seeded_write(cbs_ctx *ctx, AesDir dir, const AesKeyDst &key, const uint8_t mask_seed[32], const uint64_t *bodies)
{
    const cbs_host::AesDirDesc &d = kAesDirs[dir];
    uint64_t *const dst[3] = {key.first, key.mid, key.last};
    const uint32_t words[3] = {d.first_words, d.mid_words, d.last_words};
    const uint64_t *src = bodies;
    for (int i = 0; i < 3; i++) {
        const size_t n = words[i] / kGlweWords;
        CUDA_TRY(cudaMemcpy2DAsync(dst[i] + 2048, kGlweWords * 8, src, 1024 * 8, 1024 * 8, n, cudaMemcpyHostToDevice, ctx->stream));
        src += n * 1024;
    }
    LutMaskSeed seed;
    memcpy(seed.w, mask_seed, sizeof seed.w);
    const int nfirst = d.first_words / kGlweWords, nglwe = (d.first_words + d.mid_words + d.last_words) / kGlweWords;
    launch_expand_lut_masks(seed, dir, nfirst, nglwe, key.first, key.mid, key.last, ctx->stream);
    ctx->launches++;
    TRY(check_launch("k_expand_lut_masks"));
    TRY(aes_key_check_masks(dir, key, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return CBS_OK;
}

int aes_key_seeded_upload(cbs_ctx *ctx, AesDir dir, const uint8_t mask_seed[32], const uint64_t *bodies)
{
    TRY(aes_key_alloc(ctx, dir));
    TRY(aes_key_seeded_write(ctx, dir, single_key_dst(ctx, dir), mask_seed, bodies));
    ctx->aes[dir].uploaded = true;
    return CBS_OK;
}

// Host-buffer transciphering in direction `dir` with the key upload overlapped.  in = the public blocks of the first round
// (ECB: the ciphertext; CTR: the counter blocks), ct = the CTR ciphertext (nullptr for ECB).  Synchronous for the caller.
int aes_transcipher_host(cbs_ctx *ctx, AesDir dir, const uint8_t *in, const uint8_t *ct, int nblocks, const uint64_t *first,
                         const uint64_t *mid, const uint64_t *last, uint64_t *out)
{
    TRY(aes_key_upload(ctx, dir, first, mid, last, true));
    ctx->keys_in_flight = true;
    uint64_t *d_out = nullptr;
    auto run = [&]() {
        uint8_t *d_in, *d_ct = nullptr;
        TRY(ws_typed(ctx, ct ? "io_ctr" : "io_ct", (size_t)nblocks * 16, &d_in));
        if (ct) TRY(ws_typed(ctx, "io_ct", (size_t)nblocks * 16, &d_ct));
        TRY(ws_typed(ctx, "io_result", (size_t)nblocks * 128 * kLweBig, &d_out));
        TRY(upload(ctx, d_in, in, (size_t)nblocks * 16));
        if (ct) TRY(upload(ctx, d_ct, ct, (size_t)nblocks * 16));
        return dev_aes_single(ctx, dir, d_in, d_ct, nblocks, d_out);
    };
    const int rc = run();
    // whatever happened, the compute stream is ordered after the key copy before the call returns (host buffers, later calls)
    cudaStreamWaitEvent(ctx->stream, ctx->ev_keys, 0);
    ctx->keys_in_flight = false;
    if (rc != CBS_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    return download(ctx, out, d_out, (size_t)nblocks * 128 * kLweBig * 8);
}

// ---- key slots (include/cbs_b200.h) ----

// Grows direction `dir`'s pool to nslots slots: new buffers from the stream-ordered allocator, the uploaded slots copied over
// device to device and the old buffers freed, all on the compute stream behind earlier work that may read them.  An allocation
// failure frees what was allocated and leaves the old pool as it was.
int key_slots_reserve(cbs_ctx *ctx, AesDir dir, int nslots, const char *what)
{
    cbs_ctx::KeySlots &P = ctx->slots[dir];
    if (nslots <= 0 || nslots < P.n) {
        set_error(std::string(what) + ": " + std::to_string(nslots) + " slots requested, " + std::to_string(P.n) +
                  " reserved (a pool only grows)");
        return CBS_ERR_ARG;
    }
    if (nslots == P.n) return CBS_OK;
    const cbs_host::AesDirDesc &d = kAesDirs[dir];
    const size_t slot_bytes[4] = {(size_t)d.first_words * 8, (size_t)d.mid_words * 8, (size_t)d.last_words * 8, sizeof(int)};
    void **old[4] = {(void **)&P.first, (void **)&P.mid, (void **)&P.last, (void **)&P.flags};
    void *grown[4] = {};
    for (int i = 0; i < 4; i++) {
        const cudaError_t e = cudaMallocAsync(&grown[i], slot_bytes[i] * nslots, ctx->stream);
        if (e != cudaSuccess) {
            cudaGetLastError();
            for (int j = 0; j < i; j++) cudaFreeAsync(grown[j], ctx->stream);
            set_error(std::string(what) + ": cannot allocate " + std::to_string(nslots) + " slots: " + cudaGetErrorString(e));
            return CBS_ERR_NOMEM;
        }
    }
    for (int i = 0; i < 4; i++) {
        if (P.n) CUDA_TRY(cudaMemcpyAsync(grown[i], *old[i], slot_bytes[i] * P.n, cudaMemcpyDeviceToDevice, ctx->stream));
        if (*old[i]) CUDA_TRY(cudaFreeAsync(*old[i], ctx->stream));
        *old[i] = grown[i];
    }
    P.n = nslots;
    P.uploaded.resize(nslots, false);
    return CBS_OK;
}

// a slot upload replaces the slot's key: it is not readable until the upload has completed
int key_slot_begin(cbs_ctx *ctx, AesDir dir, int slot, const char *what)
{
    cbs_ctx::KeySlots &P = ctx->slots[dir];
    if (slot < 0 || slot >= P.n) {
        set_error(std::string(what) + ": slot " + std::to_string(slot) + " outside the " + std::to_string(P.n) + " reserved slots");
        return CBS_ERR_ARG;
    }
    P.uploaded[slot] = false;
    return CBS_OK;
}

int key_slot_upload(cbs_ctx *ctx, AesDir dir, int slot, const uint64_t *first, const uint64_t *mid, const uint64_t *last,
                    const char *what)
{
    TRY(key_slot_begin(ctx, dir, slot, what));
    TRY(aes_key_write(ctx, dir, slot_dst(ctx, dir, slot), first, mid, last, false));
    ctx->slots[dir].uploaded[slot] = true;
    return CBS_OK;
}

int key_slot_seeded_upload(cbs_ctx *ctx, AesDir dir, int slot, const uint8_t mask_seed[32], const uint64_t *bodies, const char *what)
{
    TRY(key_slot_begin(ctx, dir, slot, what));
    TRY(aes_key_seeded_write(ctx, dir, slot_dst(ctx, dir, slot), mask_seed, bodies));
    ctx->slots[dir].uploaded[slot] = true;
    return CBS_OK;
}

// Host-buffer transciphering under key slots: the inputs go up, dev_aes_slots runs, the rows come down.  Synchronous.
int aes_transcipher_slots_host(cbs_ctx *ctx, AesDir dir, const uint8_t *in, const uint8_t *ct, const int32_t *slots, int nblocks,
                               uint64_t *out, const char *what)
{
    std::vector<int> table;
    TRY(check_slots(ctx, dir, slots, nblocks, what, &table));
    uint8_t *d_in, *d_ct = nullptr;
    uint64_t *d_out;
    TRY(ws_typed(ctx, ct ? "io_ctr" : "io_ct", (size_t)nblocks * 16, &d_in));
    if (ct) TRY(ws_typed(ctx, "io_ct", (size_t)nblocks * 16, &d_ct));
    TRY(ws_typed(ctx, "io_result", (size_t)nblocks * 128 * kLweBig, &d_out));
    TRY(upload(ctx, d_in, in, (size_t)nblocks * 16));
    if (ct) TRY(upload(ctx, d_ct, ct, (size_t)nblocks * 16));
    const int rc = dev_aes_slots(ctx, dir, d_in, d_ct, table.data(), nblocks, d_out, what);
    if (rc != CBS_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    return download(ctx, out, d_out, (size_t)nblocks * 128 * kLweBig * 8);
}

}  // namespace

extern "C" {

int cbs_device_count(int *count)
{
    if (!count) return CBS_ERR_ARG;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *count = 0;
        set_error(std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
        return CBS_ERR_CUDA;
    }
    *count = n;
    return CBS_OK;
}

// workspaces come from the stream-ordered allocator (ws_get): keep what it frees cached in the device's default pool
static void keep_pool_memory(int device)
{
    cudaMemPool_t pool = nullptr;
    uint64_t keep = UINT64_MAX;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    cudaGetLastError();
}

int cbs_device_init(int device)
{
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaFree(nullptr));
    keep_pool_memory(device);
    return CBS_OK;
}

int cbs_ctx_create(const cbs_keyset *ks, int device, cbs_ctx **out)
{
    if (!ks || !out) {
        set_error("cbs_ctx_create: null argument");
        return CBS_ERR_ARG;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_error("no CUDA device: libcbs_b200 has no CPU fallback");
        return CBS_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) {
        set_error("cbs_ctx_create: device index out of range");
        return CBS_ERR_ARG;
    }
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error(std::string("device ") + prop.name + " is not sm_100: kernels are built for sm_100a only");
        return CBS_ERR_CUDA;
    }
    auto *ctx = new cbs_ctx;
    ctx->device = device;
    if (const char *e = getenv("CBS_CHUNK_BLOCKS")) ctx->chunk_blocks = std::max(1, atoi(e));
    if (const char *e = getenv("CBS_LANES")) ctx->lanes = std::max(1, std::min((int)cbs_ctx::kMaxLanes, atoi(e)));
    // at least 8: one job of a layer can bring 8 new bits into a sub-batch
    if (const char *e = getenv("CBS_PLAN_CAP")) ctx->plan_cap = std::max(8, atoi(e));
    Activate act(ctx);
    keep_pool_memory(device);
    cudaError_t e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        set_error(std::string("cudaStreamCreate: ") + cudaGetErrorString(e));
        delete ctx;
        return CBS_ERR_CUDA;
    }
    auto fail = [&](int rc) {
        cbs_ctx_destroy(ctx);
        return rc;
    };
    for (int l = 0; l < cbs_ctx::kMaxLanes; l++) {
        if (cudaStreamCreateWithFlags(&ctx->side[l], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_join[l], cudaEventDisableTiming) != cudaSuccess) {
            set_error("cannot create lane streams");
            return fail(CBS_ERR_CUDA);
        }
    }
    if (cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess) {
        set_error("cannot create lane events");
        return fail(CBS_ERR_CUDA);
    }
    // twiddle tables
    std::vector<double> tw = make_twiddle_table();
    std::vector<double> tw128(256 + 128);
    for (int j = 0; j < 128; j++) {
        long double a = 3.14159265358979323846264338327950288L * j / 256.0L;
        tw128[2 * j] = (double)cosl(a);
        tw128[2 * j + 1] = (double)sinl(a);
    }
    for (int j = 0; j < 64; j++) {
        long double a = -2.0L * 3.14159265358979323846264338327950288L * j / 128.0L;
        tw128[256 + 2 * j] = (double)cosl(a);
        tw128[256 + 2 * j + 1] = (double)sinl(a);
    }
    void *d_tw, *d_tw128, *d_bsk_f, *d_auto_f, *d_ss_f, *d_ksk_f, *d_tmp;
    int rc;
    if ((rc = key_alloc(ctx, tw.size() * 8, &d_tw)) || (rc = key_alloc(ctx, tw128.size() * 8, &d_tw128)) ||
        (rc = key_alloc(ctx, (size_t)CBS_BSK_WORDS * 8, &d_bsk_f)) ||
        (rc = key_alloc(ctx, (size_t)CBS_AUTO_WORDS * 2 * 8, &d_auto_f)) ||
        (rc = key_alloc(ctx, (size_t)CBS_SS_WORDS * 8, &d_ss_f)) ||
        (rc = key_alloc(ctx, (size_t)CBS_KSK_WORDS * 8, &d_ksk_f)))
        return fail(rc);
    if ((rc = upload(ctx, d_tw, tw.data(), tw.size() * 8)) || (rc = upload(ctx, d_tw128, tw128.data(), tw128.size() * 8)))
        return fail(rc);
    {
        // device flags "some LUT mask word is non-zero" (k_masks_nonzero after every LUT upload); 1 = not trivial until known
        void *d_flags = nullptr;
        const int ones[2] = {1, 1};
        if ((rc = key_alloc(ctx, sizeof(ones), &d_flags))) return fail(rc);
        ctx->d_masks_nonzero = (int *)d_flags;
        if (cudaMemcpy(d_flags, ones, sizeof(ones), cudaMemcpyHostToDevice) != cudaSuccess) {
            set_error("cudaMemcpy(flags) failed");
            return fail(CBS_ERR_CUDA);
        }
    }
    ctx->K.tw = (const double *)d_tw;
    ctx->K.tw128 = (const double *)d_tw128;
    // staging buffer for the standard-domain keys (largest = bsk)
    if (cudaMalloc(&d_tmp, (size_t)CBS_BSK_WORDS * 8) != cudaSuccess) {
        set_error("cudaMalloc(staging) failed");
        return fail(CBS_ERR_NOMEM);
    }
    auto conv = [&](const uint64_t *h, size_t words, double *dst, int mode) -> int {
        TRY(upload(ctx, d_tmp, h, words * 8));
        launch_std_to_fourier((const uint64_t *)d_tmp, dst, (int)(words / 1024), mode, 41, ctx->K.tw, ctx->stream);
        ctx->launches++;
        return check_launch("k_std_to_fourier");
    };
    // bsk: convert_standard_lwe_bootstrap_key_to_fourier (server_encrypted_aes_decryption.rs:656-663)
    if ((rc = conv(ks->bsk.data(), CBS_BSK_WORDS, (double *)d_bsk_f, 0))) {
        cudaFree(d_tmp);
        return fail(rc);
    }
    // ss key (:665-687)
    if ((rc = conv(ks->ss.data(), CBS_SS_WORDS, (double *)d_ss_f, 0))) {
        cudaFree(d_tmp);
        return fail(rc);
    }
    // automorphism keys: Split(41) limbs, layout [10][2 in][2 split][3 level][3 col]
    // (convert_standard_glwe_keyswitch_key_to_fourier, fourier_glwe_keyswitch.rs:154-211)
    if ((rc = upload(ctx, d_tmp, ks->autok.data(), (size_t)CBS_AUTO_WORDS * 8))) {
        cudaFree(d_tmp);
        return fail(rc);
    }
    for (int idx = 0; idx < 10; idx++)
        for (int in = 0; in < 2; in++)
            for (int sp = 0; sp < 2; sp++) {
                const uint64_t *src = (const uint64_t *)d_tmp + ((size_t)idx * 2 + in) * 9 * 1024;
                double *dst = (double *)d_auto_f + (((size_t)idx * 2 + in) * 2 + sp) * 9 * kFourierPolyDoubles;
                launch_std_to_fourier(src, dst, 9, sp ? 2 : 1, 41, ctx->K.tw, ctx->stream);
                ctx->launches++;
            }
    if ((rc = check_launch("auto key conversion"))) {
        cudaFree(d_tmp);
        return fail(rc);
    }
    cudaStreamSynchronize(ctx->stream);
    // ksk over N' = 256 (:646-654)
    if ((rc = upload(ctx, d_tmp, ks->ksk.data(), (size_t)CBS_KSK_WORDS * 8))) {
        cudaFree(d_tmp);
        return fail(rc);
    }
    launch_ksk_to_fourier((const uint64_t *)d_tmp, (double *)d_ksk_f, 8 * 3 * 4, ctx->K.tw128, ctx->stream);
    ctx->launches++;
    rc = check_launch("k_ksk_to_fourier");
    cudaError_t se = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_tmp);
    if (rc) return fail(rc);
    if (se != cudaSuccess) {
        set_error(std::string("key conversion failed: ") + cudaGetErrorString(se));
        return fail(CBS_ERR_CUDA);
    }
    ctx->K.bsk_f = (const double *)d_bsk_f;
    ctx->K.auto_f = (const double *)d_auto_f;
    ctx->K.ss_f = (const double *)d_ss_f;
    ctx->K.ksk_f = (const double *)d_ksk_f;
    *out = ctx;
    return CBS_OK;
}

void cbs_ctx_destroy(cbs_ctx *ctx)
{
    if (!ctx) return;
    Activate act(ctx);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    cudaDeviceSynchronize();
    for (void *p : ctx->key_allocs) cudaFree(p);
    for (auto &kv : ctx->ws)
        if (kv.second.p) cudaFree(kv.second.p);
    for (const LutPlanExec &E : ctx->plans)
        if (E.d_tab) cudaFree(E.d_tab);
    if (ctx->d_plan_luts) cudaFree(ctx->d_plan_luts);
    for (const cbs_ctx::AesKeys &key : ctx->aes)
        for (uint64_t *p : {key.first, key.mid, key.last})
            if (p) cudaFree(p);
    for (const cbs_ctx::KeySlots &P : ctx->slots)
        for (void *p : {(void *)P.first, (void *)P.mid, (void *)P.last, (void *)P.flags})
            if (p) cudaFree(p);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->ev_keys) cudaEventDestroy(ctx->ev_keys);
    if (ctx->ev_copy_after) cudaEventDestroy(ctx->ev_copy_after);
    for (int l = 0; l < cbs_ctx::kMaxLanes; l++) {
        if (ctx->side[l]) cudaStreamDestroy(ctx->side[l]);
        if (ctx->ev_join[l]) cudaEventDestroy(ctx->ev_join[l]);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int cbs_ctx_device(const cbs_ctx *ctx) { return ctx ? ctx->device : -1; }
uint64_t cbs_ctx_launch_count(const cbs_ctx *ctx) { return ctx ? ctx->launches : 0; }

int cbs_ctx_set_stream(cbs_ctx *ctx, void *cuda_stream)
{
    ENTER(ctx);
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (cuda_stream) {
        ctx->stream = (cudaStream_t)cuda_stream;
        ctx->own_stream = false;
    } else {
        CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->own_stream = true;
    }
    return CBS_OK;
}

int cbs_ctx_synchronize(cbs_ctx *ctx)
{
    ENTER(ctx);
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return CBS_OK;
}

int cbs_measure_fp64_tflops(cbs_ctx *ctx, double *tflops)
{
    ENTER(ctx);
    if (!tflops) return CBS_ERR_ARG;
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, ctx->device));
    const int blocks = prop.multiProcessorCount * 8, iters = 20000;
    double *d;
    TRY(ws_typed(ctx, "fp64_probe", (size_t)blocks * 256, &d));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        CUDA_TRY(cudaEventRecord(e0, ctx->stream));
        launch_fp64_peak(d, blocks, iters, ctx->stream);
        CUDA_TRY(cudaEventRecord(e1, ctx->stream));
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms;
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    ctx->launches += 4;
    *tflops = 2.0 * 16.0 * (double)iters * 256.0 * blocks / (best * 1e-3) * 1e-12;
    return check_launch("k_fp64_peak");
}

int cbs_dev_alloc(cbs_ctx *ctx, size_t bytes, void **dptr)
{
    ENTER(ctx);
    CUDA_TRY(cudaMalloc(dptr, bytes));
    return CBS_OK;
}
int cbs_dev_free(cbs_ctx *ctx, void *dptr)
{
    ENTER(ctx);
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaFree(dptr));
    return CBS_OK;
}
int cbs_dev_upload(cbs_ctx *ctx, void *dptr, const void *host, size_t bytes)
{
    ENTER(ctx);
    TRY(upload(ctx, dptr, host, bytes));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return CBS_OK;
}
int cbs_dev_download(cbs_ctx *ctx, void *host, const void *dptr, size_t bytes)
{
    ENTER(ctx);
    return download(ctx, host, dptr, bytes);
}

// ---- host-buffer stage entry points ----

int cbs_lwe_keyswitch(cbs_ctx *ctx, const uint64_t *in_big, uint64_t *out_small, int count)
{
    ENTER(ctx);
    if (count < 0 || (count && (!in_big || !out_small))) return set_error("cbs_lwe_keyswitch: bad argument"), CBS_ERR_ARG;
    if (!count) return CBS_OK;
    uint64_t *d_in, *d_out;
    TRY(ws_typed(ctx, "io_in", (size_t)count * kLweBig, &d_in));
    TRY(ws_typed(ctx, "ks", (size_t)count * kLweSmall, &d_out));
    TRY(upload(ctx, d_in, in_big, (size_t)count * kLweBig * 8));
    TRY(dev_keyswitch(ctx, d_in, d_out, count));
    return download(ctx, out_small, d_out, (size_t)count * kLweSmall * 8);
}

int cbs_blind_rotate(cbs_ctx *ctx, const uint64_t *in_small, uint64_t *acc_out, int count)
{
    ENTER(ctx);
    if (count < 0 || (count && (!in_small || !acc_out))) return set_error("cbs_blind_rotate: bad argument"), CBS_ERR_ARG;
    if (!count) return CBS_OK;
    uint64_t *d_in, *d_acc;
    TRY(ws_typed(ctx, "ks", (size_t)count * kLweSmall, &d_in));
    TRY(ws_typed(ctx, "acc", (size_t)count * kGlweWords, &d_acc));
    TRY(upload(ctx, d_in, in_small, (size_t)count * kLweSmall * 8));
    TRY(dev_blind_rotate(ctx, d_in, d_acc, count));
    return download(ctx, acc_out, d_acc, (size_t)count * kGlweWords * 8);
}

int cbs_blind_rotate_dev(cbs_ctx *ctx, const uint64_t *d_in_small, uint64_t *d_acc_out, int count)
{
    ENTER(ctx);
    if (count <= 0 || !d_in_small || !d_acc_out) return set_error("cbs_blind_rotate_dev: bad argument"), CBS_ERR_ARG;
    return dev_blind_rotate(ctx, d_in_small, d_acc_out, count);
}

int cbs_glev_from_acc(cbs_ctx *ctx, const uint64_t *acc, uint64_t *glev_out, int count)
{
    ENTER(ctx);
    if (count < 0 || (count && (!acc || !glev_out))) return set_error("cbs_glev_from_acc: bad argument"), CBS_ERR_ARG;
    if (!count) return CBS_OK;
    uint64_t *d_acc, *d_glev;
    TRY(ws_typed(ctx, "acc", (size_t)count * kGlweWords, &d_acc));
    TRY(ws_typed(ctx, "glev", (size_t)count * kGlevWords, &d_glev));
    TRY(upload(ctx, d_acc, acc, (size_t)count * kGlweWords * 8));
    launch_glev_from_acc(d_acc, d_glev, count, ctx->stream);
    ctx->launches++;
    TRY(check_launch("k_glev_from_acc"));
    return download(ctx, glev_out, d_glev, (size_t)count * kGlevWords * 8);
}

int cbs_trace(cbs_ctx *ctx, uint64_t *glwe_inout, int count)
{
    ENTER(ctx);
    if (count < 0 || (count && !glwe_inout)) return set_error("cbs_trace: bad argument"), CBS_ERR_ARG;
    if (!count) return CBS_OK;
    uint64_t *d_in, *d_out;
    TRY(ws_typed(ctx, "io_in", (size_t)count * kGlweWords, &d_in));
    TRY(ws_typed(ctx, "glev", (size_t)count * kGlweWords, &d_out));
    TRY(upload(ctx, d_in, glwe_inout, (size_t)count * kGlweWords * 8));
    launch_trace(ctx->K, d_in, d_out, count, 0, ctx->stream);
    ctx->launches++;
    TRY(check_launch("k_trace"));
    return download(ctx, glwe_inout, d_out, (size_t)count * kGlweWords * 8);
}

int cbs_lwe_msb_bit_to_glev(cbs_ctx *ctx, const uint64_t *in_small, uint64_t *glev_out, int count)
{
    ENTER(ctx);
    if (count < 0 || (count && (!in_small || !glev_out))) return set_error("cbs_lwe_msb_bit_to_glev: bad argument"), CBS_ERR_ARG;
    if (!count) return CBS_OK;
    uint64_t *d_in, *d_glev;
    TRY(ws_typed(ctx, "ks", (size_t)count * kLweSmall, &d_in));
    TRY(ws_typed(ctx, "glev", (size_t)count * kGlevWords, &d_glev));
    TRY(upload(ctx, d_in, in_small, (size_t)count * kLweSmall * 8));
    TRY(dev_msb_to_glev(ctx, d_in, d_glev, count));
    return download(ctx, glev_out, d_glev, (size_t)count * kGlevWords * 8);
}

int cbs_scheme_switch(cbs_ctx *ctx, const uint64_t *glev, uint64_t *ggsw_out, int count)
{
    ENTER(ctx);
    if (count < 0 || (count && (!glev || !ggsw_out))) return set_error("cbs_scheme_switch: bad argument"), CBS_ERR_ARG;
    if (!count) return CBS_OK;
    uint64_t *d_glev, *d_ggsw;
    TRY(ws_typed(ctx, "glev", (size_t)count * kGlevWords, &d_glev));
    TRY(ws_typed(ctx, "ggsw_std", (size_t)count * kGgswWords, &d_ggsw));
    TRY(upload(ctx, d_glev, glev, (size_t)count * kGlevWords * 8));
    launch_scheme_switch(ctx->K, d_glev, d_ggsw, nullptr, count, ctx->stream);
    ctx->launches++;
    TRY(check_launch("k_scheme_switch"));
    return download(ctx, ggsw_out, d_ggsw, (size_t)count * kGgswWords * 8);
}

int cbs_circuit_bootstrap(cbs_ctx *ctx, const uint64_t *in_small, uint64_t *ggsw_out, int count)
{
    ENTER(ctx);
    if (count < 0 || (count && (!in_small || !ggsw_out))) return set_error("cbs_circuit_bootstrap: bad argument"), CBS_ERR_ARG;
    if (!count) return CBS_OK;
    uint64_t *d_in, *d_ggsw;
    double *d_ggsw_f;
    TRY(ws_typed(ctx, "ks", (size_t)count * kLweSmall, &d_in));
    TRY(ws_typed(ctx, "ggsw_std", (size_t)count * kGgswWords, &d_ggsw));
    TRY(ws_typed(ctx, "ggsw_f", (size_t)count * kGgswWords, &d_ggsw_f));
    TRY(upload(ctx, d_in, in_small, (size_t)count * kLweSmall * 8));
    TRY(dev_circuit_bootstrap(ctx, d_in, d_ggsw, d_ggsw_f, count));
    return download(ctx, ggsw_out, d_ggsw, (size_t)count * kGgswWords * 8);
}

int cbs_circuit_bootstrap_dev(cbs_ctx *ctx, const uint64_t *d_in_small, int count)
{
    ENTER(ctx);
    if (count <= 0 || !d_in_small) return set_error("cbs_circuit_bootstrap_dev: bad argument"), CBS_ERR_ARG;
    double *d_ggsw_f;
    TRY(ws_typed(ctx, "ggsw_f", (size_t)count * kGgswWords, &d_ggsw_f));
    return dev_circuit_bootstrap(ctx, d_in_small, nullptr, d_ggsw_f, count);
}

int cbs_lut8_eval(cbs_ctx *ctx, const uint64_t *ggsw_bits, int nbytes, const uint64_t *luts, int nluts, uint64_t *out)
{
    ENTER(ctx);
    if (nbytes < 0 || nluts <= 0 || (nbytes && (!ggsw_bits || !luts || !out))) return set_error("cbs_lut8_eval: bad argument"), CBS_ERR_ARG;
    if (!nbytes) return CBS_OK;
    const int nbits = nbytes * 8, apb = nluts * 2, njobs = nbytes * apb;
    uint64_t *d_ggsw, *d_luts, *d_out;
    double *d_ggsw_f;
    int *d_li, *d_oi;
    TRY(ws_typed(ctx, "ggsw_std", (size_t)nbits * kGgswWords, &d_ggsw));
    TRY(ws_typed(ctx, "ggsw_f", (size_t)nbits * kGgswWords, &d_ggsw_f));
    TRY(ws_typed(ctx, "io_luts", (size_t)njobs * kGlweWords, &d_luts));
    TRY(ws_typed(ctx, "io_out", (size_t)njobs * 4 * kLweBig, &d_out));
    TRY(ws_typed(ctx, "io_li", (size_t)njobs, &d_li));
    TRY(ws_typed(ctx, "io_oi", (size_t)njobs, &d_oi));
    std::vector<int> li(njobs), oi(njobs);
    for (int j = 0; j < njobs; j++) {
        li[j] = j;      // luts[nbytes][nluts][2] in job order
        oi[j] = j * 4;  // out[nbytes][nluts][8]
    }
    TRY(upload(ctx, d_ggsw, ggsw_bits, (size_t)nbits * kGgswWords * 8));
    TRY(upload(ctx, d_luts, luts, (size_t)njobs * kGlweWords * 8));
    TRY(upload(ctx, d_li, li.data(), sizeof(int) * njobs));
    TRY(upload(ctx, d_oi, oi.data(), sizeof(int) * njobs));
    launch_ggsw_to_fourier(ctx->K, d_ggsw, d_ggsw_f, nbits, ctx->stream);
    ctx->launches++;
    TRY(dev_lut8(ctx, d_ggsw_f, d_luts, d_li, d_oi, d_out, njobs, apb, nullptr));
    return download(ctx, out, d_out, (size_t)njobs * 4 * kLweBig * 8);
}

int cbs_max_of_two(cbs_ctx *ctx, const uint64_t *ggsw, const uint64_t *op, int nvals, const int32_t *a_idx, const int32_t *b_idx,
                   int npairs, uint64_t *out)
{
    ENTER(ctx);
    // counts bounded so that nvals * 16 * 63 Fourier polynomials and npairs * 16 groups stay ints
    bool ok = nvals >= 0 && npairs >= 0 && nvals <= (INT_MAX >> 10) && npairs <= (INT_MAX >> 5) &&
              (!npairs || (ggsw && op && a_idx && b_idx && out));
    for (int p = 0; ok && p < npairs; p++) ok = a_idx[p] >= 0 && a_idx[p] < nvals && b_idx[p] >= 0 && b_idx[p] < nvals;
    if (!ok) return set_error("cbs_max_of_two: bad argument (negative count, null pointer or pair index outside [0, nvals))"), CBS_ERR_ARG;
    if (!npairs) return CBS_OK;
    const int nbits = nvals * 16;
    uint64_t *d_ggsw, *d_op, *d_out;
    double *d_ggsw_f;
    int *d_a, *d_b;
    TRY(ws_typed(ctx, "ggsw_std", (size_t)nbits * kGgswWords, &d_ggsw));
    TRY(ws_typed(ctx, "ggsw_f", (size_t)nbits * kGgswWords, &d_ggsw_f));
    TRY(ws_typed(ctx, "io_luts", (size_t)nbits * kGlweWords, &d_op));
    TRY(ws_typed(ctx, "io_out", (size_t)npairs * 16 * kLweBig, &d_out));
    TRY(ws_typed(ctx, "io_li", (size_t)npairs, &d_a));
    TRY(ws_typed(ctx, "io_oi", (size_t)npairs, &d_b));
    TRY(upload(ctx, d_ggsw, ggsw, (size_t)nbits * kGgswWords * 8));
    TRY(upload(ctx, d_op, op, (size_t)nbits * kGlweWords * 8));
    TRY(upload(ctx, d_a, a_idx, sizeof(int) * npairs));
    TRY(upload(ctx, d_b, b_idx, sizeof(int) * npairs));
    launch_ggsw_to_fourier(ctx->K, d_ggsw, d_ggsw_f, nbits, ctx->stream);
    ctx->launches++;
    launch_max_ladder(ctx->K, d_ggsw_f, d_op, d_a, d_b, d_out, npairs, ctx->stream);
    ctx->launches++;
    TRY(check_launch("k_max_ladder"));
    return download(ctx, out, d_out, (size_t)npairs * 16 * kLweBig * 8);
}

int cbs_lut8_gather_eval(cbs_ctx *ctx, const uint64_t *ggsw, int nbits, const int32_t *sel, const uint64_t *luts, int nluts,
                         const int32_t *lut_index, const int32_t *out_index, int njobs, uint64_t *out, int nout)
{
    ENTER(ctx);
    bool ok = nbits >= 0 && nluts >= 0 && njobs >= 0 && nout >= 0 && nbits <= (INT_MAX >> 10) && njobs <= (INT_MAX >> 3) &&
              (!njobs || (sel && luts && lut_index && out_index && out && (ggsw || !nbits)));
    // output windows [out_index, out_index + 4) inside [0, nout) and pairwise disjoint
    std::vector<int> starts;
    starts.reserve(ok ? (size_t)njobs : 0);
    for (int j = 0; ok && j < njobs; j++) {
        for (int i = 0; ok && i < 8; i++) ok = sel[(size_t)j * 8 + i] >= -1 && sel[(size_t)j * 8 + i] < nbits;
        ok = ok && lut_index[j] >= 0 && lut_index[j] < nluts && out_index[j] >= 0 && out_index[j] <= nout - 4;
        starts.push_back(out_index[j]);
    }
    std::sort(starts.begin(), starts.end());
    for (size_t j = 1; ok && j < starts.size(); j++) ok = starts[j] - starts[j - 1] >= 4;
    if (!ok)
        return set_error("cbs_lut8_gather_eval: bad argument (negative count, null pointer, selector outside [-1, nbits), "
                         "LUT index outside [0, nluts), or an output window outside [0, nout) or overlapping another)"),
               CBS_ERR_ARG;
    if (!njobs) return CBS_OK;
    uint64_t *d_ggsw = nullptr, *d_luts, *d_out;
    double *d_ggsw_f = nullptr;
    int *d_sel, *d_li, *d_oi;
    TRY(ws_typed(ctx, "io_luts", (size_t)nluts * kGlweWords, &d_luts));
    TRY(ws_typed(ctx, "io_out", (size_t)nout * kLweBig, &d_out));
    TRY(ws_typed(ctx, "io_sel", (size_t)njobs * 8, &d_sel));
    TRY(ws_typed(ctx, "io_li", (size_t)njobs, &d_li));
    TRY(ws_typed(ctx, "io_oi", (size_t)njobs, &d_oi));
    if (nbits) {
        TRY(ws_typed(ctx, "ggsw_std", (size_t)nbits * kGgswWords, &d_ggsw));
        TRY(ws_typed(ctx, "ggsw_f", (size_t)nbits * kGgswWords, &d_ggsw_f));
        TRY(upload(ctx, d_ggsw, ggsw, (size_t)nbits * kGgswWords * 8));
    }
    TRY(upload(ctx, d_luts, luts, (size_t)nluts * kGlweWords * 8));
    TRY(upload(ctx, d_sel, sel, sizeof(int) * njobs * 8));
    TRY(upload(ctx, d_li, lut_index, sizeof(int) * njobs));
    TRY(upload(ctx, d_oi, out_index, sizeof(int) * njobs));
    CUDA_TRY(cudaMemsetAsync(d_out, 0, (size_t)nout * kLweBig * 8, ctx->stream));
    if (nbits) {
        launch_ggsw_to_fourier(ctx->K, d_ggsw, d_ggsw_f, nbits, ctx->stream);
        ctx->launches++;
    }
    launch_lut8_gather(ctx->K, d_ggsw_f, d_sel, d_luts, d_li, d_oi, d_out, njobs, ctx->stream);
    ctx->launches++;
    TRY(check_launch("k_lut8_gather"));
    return download(ctx, out, d_out, (size_t)nout * kLweBig * 8);
}

int cbs_aes_first_rounds(cbs_ctx *ctx, const uint8_t *ct, int nblocks, const uint64_t *k10_9, uint64_t *state_out)
{
    ENTER(ctx);
    if (nblocks < 0 || (nblocks && (!ct || !k10_9 || !state_out))) return set_error("cbs_aes_first_rounds: bad argument"), CBS_ERR_ARG;
    if (!nblocks) return CBS_OK;
    uint8_t *d_ct;
    uint64_t *d_k, *d_t4, *d_st;
    TRY(ws_typed(ctx, "io_ct", (size_t)nblocks * 16, &d_ct));
    TRY(ws_typed(ctx, "io_luts", (size_t)CBS_K10_9_WORDS, &d_k));
    TRY(ws_typed(ctx, "t4", (size_t)4 * nblocks * 128 * kLweBig, &d_t4));
    TRY(ws_typed(ctx, "st", (size_t)nblocks * 128 * kLweBig, &d_st));
    TRY(upload(ctx, d_ct, ct, (size_t)nblocks * 16));
    TRY(upload(ctx, d_k, k10_9, (size_t)CBS_K10_9_WORDS * 8));
    launch_known_rotate(d_ct, d_k, d_t4, nblocks, 4, 1, nullptr, ctx->stream);
    launch_inv_linear(d_t4, d_st, nblocks, ctx->stream);
    ctx->launches += 2;
    TRY(check_launch("first rounds"));
    return download(ctx, state_out, d_st, (size_t)nblocks * 128 * kLweBig * 8);
}

int cbs_aes_inv_linear(cbs_ctx *ctx, const uint64_t *t4, int nblocks, uint64_t *state_out)
{
    ENTER(ctx);
    if (nblocks < 0 || (nblocks && (!t4 || !state_out))) return set_error("cbs_aes_inv_linear: bad argument"), CBS_ERR_ARG;
    if (!nblocks) return CBS_OK;
    uint64_t *d_t4, *d_st;
    TRY(ws_typed(ctx, "t4", (size_t)4 * nblocks * 128 * kLweBig, &d_t4));
    TRY(ws_typed(ctx, "st", (size_t)nblocks * 128 * kLweBig, &d_st));
    TRY(upload(ctx, d_t4, t4, (size_t)4 * nblocks * 128 * kLweBig * 8));
    launch_inv_linear(d_t4, d_st, nblocks, ctx->stream);
    ctx->launches++;
    TRY(check_launch("k_inv_linear"));
    return download(ctx, state_out, d_st, (size_t)nblocks * 128 * kLweBig * 8);
}

int cbs_trans_key_upload(cbs_ctx *ctx, const uint64_t *k10_9, const uint64_t *k8_1, const uint64_t *k0)
{
    ENTER(ctx);
    if (!k10_9 || !k8_1 || !k0) return set_error("cbs_trans_key_upload: null argument"), CBS_ERR_ARG;
    return aes_key_upload(ctx, kAesInv, k10_9, k8_1, k0, false);
}

int cbs_aes128_transcipher_dev(cbs_ctx *ctx, const uint8_t *d_ct, int nblocks, uint64_t *d_out)
{
    ENTER(ctx);
    if (nblocks <= 0 || !d_ct || !d_out) return set_error("cbs_aes128_transcipher_dev: bad argument"), CBS_ERR_ARG;
    return dev_aes_single(ctx, kAesInv, d_ct, nullptr, nblocks, d_out);
}

int cbs_aes128_transcipher(cbs_ctx *ctx, const uint8_t *ct, int nblocks, const uint64_t *k10_9, const uint64_t *k8_1,
                           const uint64_t *k0, uint64_t *out)
{
    ENTER(ctx);
    if (nblocks < 0 || (nblocks && (!ct || !out)) || !k10_9 || !k8_1 || !k0) return set_error("cbs_aes128_transcipher: bad argument"), CBS_ERR_ARG;
    if (!nblocks) return CBS_OK;
    return aes_transcipher_host(ctx, kAesInv, ct, nullptr, nblocks, k10_9, k8_1, k0, out);
}

int cbs_fwd_trans_key_upload(cbs_ctx *ctx, const uint64_t *kf_first, const uint64_t *kf_mid, const uint64_t *kf_last)
{
    ENTER(ctx);
    if (!kf_first || !kf_mid || !kf_last) return set_error("cbs_fwd_trans_key_upload: null argument"), CBS_ERR_ARG;
    return aes_key_upload(ctx, kAesFwd, kf_first, kf_mid, kf_last, false);
}

int cbs_trans_key_seeded_upload(cbs_ctx *ctx, const uint8_t mask_seed[32], const uint64_t *bodies)
{
    ENTER(ctx);
    if (!mask_seed || !bodies) return set_error("cbs_trans_key_seeded_upload: null argument"), CBS_ERR_ARG;
    return aes_key_seeded_upload(ctx, kAesInv, mask_seed, bodies);
}

int cbs_fwd_trans_key_seeded_upload(cbs_ctx *ctx, const uint8_t mask_seed[32], const uint64_t *bodies)
{
    ENTER(ctx);
    if (!mask_seed || !bodies) return set_error("cbs_fwd_trans_key_seeded_upload: null argument"), CBS_ERR_ARG;
    return aes_key_seeded_upload(ctx, kAesFwd, mask_seed, bodies);
}

int cbs_aes128_ctr_transcipher_dev(cbs_ctx *ctx, const uint8_t *d_ctr, const uint8_t *d_ct, int nblocks, uint64_t *d_out)
{
    ENTER(ctx);
    if (nblocks <= 0 || !d_ctr || !d_ct || !d_out) return set_error("cbs_aes128_ctr_transcipher_dev: bad argument"), CBS_ERR_ARG;
    return dev_aes_single(ctx, kAesFwd, d_ctr, d_ct, nblocks, d_out);
}

int cbs_aes128_ctr_transcipher(cbs_ctx *ctx, const uint8_t *ct, int nblocks, const uint8_t iv[16], const uint64_t *kf_first,
                               const uint64_t *kf_mid, const uint64_t *kf_last, uint64_t *out)
{
    ENTER(ctx);
    if (nblocks < 0 || (nblocks && (!ct || !out)) || !iv || !kf_first || !kf_mid || !kf_last)
        return set_error("cbs_aes128_ctr_transcipher: bad argument"), CBS_ERR_ARG;
    if (!nblocks) return CBS_OK;
    // counter blocks: 128-bit big-endian IV + block index (pyaes.Counter, harness/aes_keygen_and_encrypt.py:52)
    std::vector<uint8_t> ctr((size_t)nblocks * 16);
    uint8_t cur[16];
    memcpy(cur, iv, 16);
    for (int b = 0; b < nblocks; b++) {
        memcpy(ctr.data() + (size_t)b * 16, cur, 16);
        for (int i = 15; i >= 0; i--)
            if (++cur[i] != 0) break;
    }
    return aes_transcipher_host(ctx, kAesFwd, ctr.data(), ct, nblocks, kf_first, kf_mid, kf_last, out);
}

int cbs_trans_key_slots_reserve(cbs_ctx *ctx, int nslots)
{
    ENTER(ctx);
    return key_slots_reserve(ctx, kAesInv, nslots, "cbs_trans_key_slots_reserve");
}

int cbs_fwd_trans_key_slots_reserve(cbs_ctx *ctx, int nslots)
{
    ENTER(ctx);
    return key_slots_reserve(ctx, kAesFwd, nslots, "cbs_fwd_trans_key_slots_reserve");
}

int cbs_trans_key_slot_upload(cbs_ctx *ctx, int slot, const uint64_t *k10_9, const uint64_t *k8_1, const uint64_t *k0)
{
    ENTER(ctx);
    if (!k10_9 || !k8_1 || !k0) return set_error("cbs_trans_key_slot_upload: null argument"), CBS_ERR_ARG;
    return key_slot_upload(ctx, kAesInv, slot, k10_9, k8_1, k0, "cbs_trans_key_slot_upload");
}

int cbs_fwd_trans_key_slot_upload(cbs_ctx *ctx, int slot, const uint64_t *kf_first, const uint64_t *kf_mid, const uint64_t *kf_last)
{
    ENTER(ctx);
    if (!kf_first || !kf_mid || !kf_last) return set_error("cbs_fwd_trans_key_slot_upload: null argument"), CBS_ERR_ARG;
    return key_slot_upload(ctx, kAesFwd, slot, kf_first, kf_mid, kf_last, "cbs_fwd_trans_key_slot_upload");
}

int cbs_trans_key_seeded_slot_upload(cbs_ctx *ctx, int slot, const uint8_t mask_seed[32], const uint64_t *bodies)
{
    ENTER(ctx);
    if (!mask_seed || !bodies) return set_error("cbs_trans_key_seeded_slot_upload: null argument"), CBS_ERR_ARG;
    return key_slot_seeded_upload(ctx, kAesInv, slot, mask_seed, bodies, "cbs_trans_key_seeded_slot_upload");
}

int cbs_fwd_trans_key_seeded_slot_upload(cbs_ctx *ctx, int slot, const uint8_t mask_seed[32], const uint64_t *bodies)
{
    ENTER(ctx);
    if (!mask_seed || !bodies) return set_error("cbs_fwd_trans_key_seeded_slot_upload: null argument"), CBS_ERR_ARG;
    return key_slot_seeded_upload(ctx, kAesFwd, slot, mask_seed, bodies, "cbs_fwd_trans_key_seeded_slot_upload");
}

int cbs_aes128_transcipher_slots_dev(cbs_ctx *ctx, const uint8_t *d_ct, const int32_t *slots, int nblocks, uint64_t *d_out)
{
    ENTER(ctx);
    if (nblocks <= 0 || !d_ct || !slots || !d_out) return set_error("cbs_aes128_transcipher_slots_dev: bad argument"), CBS_ERR_ARG;
    return dev_aes_slots(ctx, kAesInv, d_ct, nullptr, slots, nblocks, d_out, "cbs_aes128_transcipher_slots_dev");
}

int cbs_aes128_ctr_transcipher_slots_dev(cbs_ctx *ctx, const uint8_t *d_ctr, const uint8_t *d_ct, const int32_t *slots, int nblocks,
                                         uint64_t *d_out)
{
    ENTER(ctx);
    if (nblocks <= 0 || !d_ctr || !d_ct || !slots || !d_out)
        return set_error("cbs_aes128_ctr_transcipher_slots_dev: bad argument"), CBS_ERR_ARG;
    return dev_aes_slots(ctx, kAesFwd, d_ctr, d_ct, slots, nblocks, d_out, "cbs_aes128_ctr_transcipher_slots_dev");
}

int cbs_aes128_transcipher_slots(cbs_ctx *ctx, const uint8_t *ct, const int32_t *slots, int nblocks, uint64_t *out)
{
    ENTER(ctx);
    if (nblocks <= 0 || !ct || !slots || !out) return set_error("cbs_aes128_transcipher_slots: bad argument"), CBS_ERR_ARG;
    return aes_transcipher_slots_host(ctx, kAesInv, ct, nullptr, slots, nblocks, out, "cbs_aes128_transcipher_slots");
}

int cbs_aes128_ctr_transcipher_slots(cbs_ctx *ctx, const uint8_t *ctr, const uint8_t *ct, const int32_t *slots, int nblocks,
                                     uint64_t *out)
{
    ENTER(ctx);
    if (nblocks <= 0 || !ctr || !ct || !slots || !out) return set_error("cbs_aes128_ctr_transcipher_slots: bad argument"), CBS_ERR_ARG;
    return aes_transcipher_slots_host(ctx, kAesFwd, ctr, ct, slots, nblocks, out, "cbs_aes128_ctr_transcipher_slots");
}

}  // extern "C"

// ---- stage 8: one core per computation, shared by the host-buffer and the device-resident entry points ----

namespace {

constexpr size_t kValueWords = (size_t)16 * kLweBig;  // one u16 value: 16 big LWE, MSB first

// `bytes` of input into the workspace `d`, from the caller's host memory (host = true) or HBM, on the context stream
int copy_in(cbs_ctx *ctx, void *d, const void *src, size_t bytes, bool host)
{
    CUDA_TRY(cudaMemcpyAsync(d, src, bytes, host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, ctx->stream));
    return CBS_OK;
}

// The plan of `kind` for nvals values, compiled into ctx->plans[kind] unless it is there already: host-side planning and
// the table upload run once per count, and a replaced table is freed in stream order behind the work that still reads it.
// The tables come from pageable vectors, which cudaMemcpyAsync has staged by the time it returns, so nothing here waits.
int lut_plan_get(cbs_ctx *ctx, PlanKind kind, int nvals, const LutPlanExec **out)
{
    using namespace cbs_host;
    const int kCap = ctx->plan_cap;  // circuit bootstraps per sub-batch
    LutPlanExec &E = ctx->plans[kind];
    *out = &E;
    if (E.nvals == nvals) return CBS_OK;
    if (!ctx->d_plan_luts) {
        // trivial LUT accumulators: coefficient i carries bit (4*acc + i/256) of table[i % 256] at 2^63
        // (same layout as generate_vec_keyed_lut_accumulator, cbs_lib/src/aes_he.rs:835-875)
        std::vector<uint64_t> h_luts((size_t)kIpNumLuts * 2 * kGlweWords, 0);
        for (int l = 0; l < kIpNumLuts; l++)
            for (int a = 0; a < 2; a++) {
                uint64_t *body = h_luts.data() + (size_t)(l * 2 + a) * kGlweWords + 2048;
                for (int i = 0; i < 1024; i++) body[i] = (uint64_t)((ip_lut_value(l, (unsigned)(i % 256)) >> (4 * a + i / 256)) & 1u) << 63;
            }
        uint64_t *d = nullptr;
        CUDA_TRY(cudaMallocAsync(&d, h_luts.size() * 8, ctx->stream));
        if (cudaMemcpyAsync(d, h_luts.data(), h_luts.size() * 8, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) {
            cudaFreeAsync(d, ctx->stream);
            set_error("cudaMemcpyAsync(LUT accumulators) failed");
            return CBS_ERR_CUDA;
        }
        ctx->d_plan_luts = d;
    }
    const IpPlan plan = kind == kPlanInnerProduct ? ip_make_plan(nvals) : kind == kPlanSum ? sum_make_plan(nvals) : max_make_plan(nvals);
    std::vector<PlanLayer> layers;
    std::vector<int> h_idx, h_sel, h_lut, h_out, h_add, h_ref;
    for (const IpLayer &L : plan.layers) {
        PlanLayer P;
        P.pre_off = (int)h_add.size() / 3;
        P.npre = (int)L.pre.size();
        for (const IpAdd &a : L.pre) h_add.insert(h_add.end(), {a.dst, a.a, a.b});
        P.post_off = (int)h_add.size() / 3;
        P.npost = (int)L.post.size();
        for (const IpAdd &a : L.post) h_add.insert(h_add.end(), {a.dst, a.a, a.b});
        std::vector<int> remap(L.cbs.size(), -1), ref_dst(L.cbs.size(), -1), touched;
        for (const IpRefresh &r : L.refresh) ref_dst[(size_t)r.pos] = r.dst;
        PlanBatch b{(int)h_idx.size(), 0, (int)h_lut.size(), 0, (int)h_ref.size() / 2, 0};
        auto flush = [&]() {
            if (b.njobs) P.batches.push_back(b);
            for (int pos : touched) remap[(size_t)pos] = -1;
            touched.clear();
            b = PlanBatch{(int)h_idx.size(), 0, (int)h_lut.size(), 0, (int)h_ref.size() / 2, 0};
        };
        for (const IpJob &j : L.jobs) {
            int fresh = 0;
            for (int i = 0; i < 8; i++)
                if (j.sel[i] >= 0 && remap[(size_t)j.sel[i]] < 0) fresh++;
            if (b.m + fresh > kCap) flush();
            for (int i = 0; i < 8; i++) {
                int v = -1;
                if (j.sel[i] >= 0) {
                    int &r = remap[(size_t)j.sel[i]];
                    if (r < 0) {
                        r = b.m++;
                        touched.push_back(j.sel[i]);
                        h_idx.push_back(L.cbs[(size_t)j.sel[i]]);
                        if (ref_dst[(size_t)j.sel[i]] >= 0) {
                            h_ref.insert(h_ref.end(), {r, ref_dst[(size_t)j.sel[i]]});
                            b.nref++;
                        }
                    }
                    v = r;
                }
                h_sel.push_back(v);
            }
            h_lut.push_back(j.lut * 2 + j.acc);
            h_out.push_back(j.out);
            b.njobs++;
        }
        flush();
        layers.push_back(std::move(P));
    }
    int max_m = 1;
    for (const PlanLayer &P : layers)
        for (const PlanBatch &b : P.batches) max_m = b.m > max_m ? b.m : max_m;
    for (int i = 0; i < 16; i++) h_idx.push_back(plan.result[15 - i]);  // final gather, MSB first

    std::vector<int> tab;
    size_t off[6];
    const std::vector<int> *parts[6] = {&h_idx, &h_sel, &h_lut, &h_out, &h_add, &h_ref};
    for (int k = 0; k < 6; k++) {
        off[k] = tab.size();
        tab.insert(tab.end(), parts[k]->begin(), parts[k]->end());
    }
    E.nvals = 0;
    if (E.d_tab) {
        CUDA_TRY(cudaFreeAsync(E.d_tab, ctx->stream));
        E.d_tab = nullptr;
    }
    CUDA_TRY(cudaMallocAsync(&E.d_tab, tab.size() * sizeof(int), ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(E.d_tab, tab.data(), tab.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    E.idx = E.d_tab + off[0];
    E.sel = E.d_tab + off[1];
    E.lut = E.d_tab + off[2];
    E.out = E.d_tab + off[3];
    E.add = E.d_tab + off[4];
    E.ref = E.d_tab + off[5];
    E.final_idx = (int)h_idx.size() - 16;
    E.nin_bits = plan.nin_bits;
    E.pool_size = plan.pool_size;
    E.max_m = max_m;
    E.layers = std::move(layers);
    E.nvals = nvals;
    return CBS_OK;
}

// Executes the LUT circuit `kind` (host/ip_plan.h) on nvals values: every layer is
// [LWE additions] -> [gather -> LWE keyswitch -> circuit bootstrap] -> [fresh operands from the bootstrap's GLEV] ->
// [gathered LUT ladders] -> [LWE additions]; layers whose bootstraps exceed the workspace cap run in sub-batches.
// The input rows are x, then y (y = nullptr: x holds them all).  host: x, y and out are host buffers and the call returns
// with the result downloaded; otherwise they are device pointers and the work is only queued.
int run_lut_plan(cbs_ctx *ctx, PlanKind kind, int nvals, const uint64_t *x, const uint64_t *y, bool host, uint64_t *out)
{
    const LutPlanExec *E;
    TRY(lut_plan_get(ctx, kind, nvals, &E));
    uint64_t *d_pool, *d_rows, *d_ks, *d_glev;
    double *d_ggsw_f;
    TRY(ws_typed(ctx, "ip_pool", (size_t)E->pool_size * kLweBig, &d_pool));
    TRY(ws_typed(ctx, "ip_rows", (size_t)std::max(E->max_m, 16) * kLweBig, &d_rows));  // also holds the 16 result rows
    TRY(ws_typed(ctx, "ks", (size_t)E->max_m * kLweSmall, &d_ks));
    TRY(ws_typed(ctx, "ggsw_f", (size_t)E->max_m * kGgswWords, &d_ggsw_f));
    TRY(ws_typed(ctx, "glev", (size_t)E->max_m * kGlevWords, &d_glev));  // the circuit bootstrap's own GLEV workspace
    const size_t x_words = (size_t)(y ? E->nin_bits / 2 : E->nin_bits) * kLweBig;
    TRY(copy_in(ctx, d_pool, x, x_words * 8, host));
    if (y) TRY(copy_in(ctx, d_pool + x_words, y, x_words * 8, host));
    for (const PlanLayer &P : E->layers) {
        if (P.npre) {
            launch_lwe_add_rows(d_pool, E->add + (size_t)P.pre_off * 3, P.npre, ctx->stream);
            ctx->launches++;
            TRY(check_launch("k_lwe_add_rows"));
        }
        for (const PlanBatch &b : P.batches) {
            launch_gather_lwe(d_pool, E->idx + b.idx_off, d_rows, b.m, ctx->stream);
            ctx->launches++;
            TRY(check_launch("k_gather_lwe"));
            TRY(dev_keyswitch(ctx, d_rows, d_ks, b.m));
            TRY(dev_circuit_bootstrap(ctx, d_ks, nullptr, d_ggsw_f, b.m));
            if (b.nref) {
                launch_glev_to_lwe(d_glev, E->ref + (size_t)b.ref_off * 2, d_pool, b.nref, ctx->stream);
                ctx->launches++;
                TRY(check_launch("k_glev_to_lwe"));
            }
            launch_lut8_gather(ctx->K, d_ggsw_f, E->sel + (size_t)b.job_off * 8, ctx->d_plan_luts, E->lut + b.job_off,
                               E->out + b.job_off, d_pool, b.njobs, ctx->stream);
            ctx->launches++;
            TRY(check_launch("k_lut8_gather"));
        }
        if (P.npost) {
            launch_lwe_add_rows(d_pool, E->add + (size_t)P.post_off * 3, P.npost, ctx->stream);
            ctx->launches++;
            TRY(check_launch("k_lwe_add_rows"));
        }
    }
    launch_gather_lwe(d_pool, E->idx + E->final_idx, host ? d_rows : out, 16, ctx->stream);
    ctx->launches++;
    TRY(check_launch("k_gather_lwe"));
    return host ? download(ctx, out, d_rows, kValueWords * 8) : CBS_OK;
}

// The reference's max_of_two CMux ladder over a balanced tree, nvals >= 2; host / device buffers as run_lut_plan.
int max_ladder(cbs_ctx *ctx, const uint64_t *in, int nvals, bool host, uint64_t *out)
{
    // balanced tree: level buffers A (current) and B (next)
    uint64_t *d_lwe[2], *d_op[2], *d_ks, *d_glev;
    double *d_ggsw[2];
    int *d_a, *d_b;
    const size_t vals_lwe = kValueWords, vals_ggsw = (size_t)16 * kGgswWords, vals_op = (size_t)16 * kGlweWords;
    TRY(ws_typed(ctx, "max_lwe0", (size_t)nvals * vals_lwe, &d_lwe[0]));
    TRY(ws_typed(ctx, "max_lwe1", (size_t)((nvals + 1) / 2) * vals_lwe, &d_lwe[1]));
    TRY(ws_typed(ctx, "max_ggsw0", (size_t)nvals * vals_ggsw, &d_ggsw[0]));
    TRY(ws_typed(ctx, "max_ggsw1", (size_t)((nvals + 1) / 2) * vals_ggsw, &d_ggsw[1]));
    TRY(ws_typed(ctx, "max_op0", (size_t)nvals * vals_op, &d_op[0]));
    TRY(ws_typed(ctx, "max_op1", (size_t)((nvals + 1) / 2) * vals_op, &d_op[1]));
    TRY(ws_typed(ctx, "ks", (size_t)nvals * 16 * kLweSmall, &d_ks));
    TRY(ws_typed(ctx, "glev", (size_t)nvals * 16 * kGlevWords, &d_glev));  // the circuit bootstrap's own GLEV workspace
    // pair tables (2i, 2i+1) do not depend on the count: one table sized to the largest count seen serves every call
    const int pairs = std::max(nvals / 2, ctx->ladder_pairs);
    TRY(ws_typed(ctx, "max_a", (size_t)pairs, &d_a));
    TRY(ws_typed(ctx, "max_b", (size_t)pairs, &d_b));
    if (pairs > ctx->ladder_pairs) {
        std::vector<int> ha(pairs), hb(pairs);
        for (int i = 0; i < pairs; i++) {
            ha[i] = 2 * i;
            hb[i] = 2 * i + 1;
        }
        TRY(upload(ctx, d_a, ha.data(), sizeof(int) * ha.size()));
        TRY(upload(ctx, d_b, hb.data(), sizeof(int) * hb.size()));
        ctx->ladder_pairs = pairs;
    }
    TRY(copy_in(ctx, d_lwe[0], in, (size_t)nvals * vals_lwe * 8, host));
    int cnt = nvals, cur = 0, fresh = nvals;  // `fresh` leading values of the current level still need a CBS
    while (cnt > 1) {
        // keyswitch + circuit bootstrap the values produced by the previous level (server_encrypted_compute.rs:213-263,314-342);
        // the level-1 GLEV of the same bootstrap, doubled, is the refreshed data operand of the ladder
        TRY(dev_keyswitch(ctx, d_lwe[cur], d_ks, fresh * 16));
        TRY(dev_circuit_bootstrap(ctx, d_ks, nullptr, d_ggsw[cur], fresh * 16));
        launch_glev_to_operand(d_glev, d_op[cur], fresh * 16, ctx->stream);
        ctx->launches++;
        TRY(check_launch("k_glev_to_operand"));
        const int npairs = cnt / 2;
        launch_max_ladder(ctx->K, d_ggsw[cur], d_op[cur], d_a, d_b, d_lwe[cur ^ 1], npairs, ctx->stream);
        ctx->launches++;
        TRY(check_launch("k_max_ladder"));
        int next = npairs;
        if (cnt & 1) {  // odd one out is carried with its GGSW and operand (no new bootstrap needed)
            CUDA_TRY(cudaMemcpyAsync(d_lwe[cur ^ 1] + (size_t)npairs * vals_lwe, d_lwe[cur] + (size_t)(cnt - 1) * vals_lwe,
                                     vals_lwe * 8, cudaMemcpyDeviceToDevice, ctx->stream));
            CUDA_TRY(cudaMemcpyAsync(d_ggsw[cur ^ 1] + (size_t)npairs * vals_ggsw, d_ggsw[cur] + (size_t)(cnt - 1) * vals_ggsw,
                                     vals_ggsw * 8, cudaMemcpyDeviceToDevice, ctx->stream));
            CUDA_TRY(cudaMemcpyAsync(d_op[cur ^ 1] + (size_t)npairs * vals_op, d_op[cur] + (size_t)(cnt - 1) * vals_op,
                                     vals_op * 8, cudaMemcpyDeviceToDevice, ctx->stream));
            next++;
        }
        fresh = npairs;
        cnt = next;
        cur ^= 1;
    }
    if (host) return download(ctx, out, d_lwe[cur], vals_lwe * 8);
    CUDA_TRY(cudaMemcpyAsync(out, d_lwe[cur], vals_lwe * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    return CBS_OK;
}

int max_u16(cbs_ctx *ctx, const uint64_t *in, int nvals, bool host, uint64_t *out)
{
    if (nvals == 1) {
        if (host) memcpy(out, in, kValueWords * 8);
        else CUDA_TRY(cudaMemcpyAsync(out, in, kValueWords * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        return CBS_OK;
    }
    // up to the reference's own 8 values: its max_of_two CMux ladder; above (where the reference cannot run and the
    // ladder's data-dependent noise becomes a real failure probability): the LUT circuit.  CBS_MAX_VARIANT=ladder|lut overrides.
    const char *e = getenv("CBS_MAX_VARIANT");
    const bool lut = e ? (strcmp(e, "lut") == 0) : nvals > 8;
    return lut ? run_lut_plan(ctx, kPlanMax, nvals, in, nullptr, host, out) : max_ladder(ctx, in, nvals, host, out);
}

// Arguments of the device-resident calls: count values in d_x (and as many in d_y when given), 16 result rows in d_out,
// which must not overlap either input.  Counts stay where count * 16 bit ciphertexts (both halves) fit an int.
int check_dev_args(const char *what, int count, const uint64_t *d_x, const uint64_t *d_y, bool need_y, const uint64_t *d_out)
{
    auto overlaps = [](const uint64_t *a, size_t a_words, const uint64_t *b, size_t b_words) { return a < b + b_words && b < a + a_words; };
    const bool ok = count > 0 && count <= (INT_MAX >> 5) && d_x && d_out && (d_y || !need_y) &&
                    !overlaps(d_out, kValueWords, d_x, (size_t)count * kValueWords) &&
                    !(d_y && overlaps(d_out, kValueWords, d_y, (size_t)count * kValueWords));
    if (ok) return CBS_OK;
    set_error(std::string(what) + ": bad argument (need a positive count, non-null pointers and a d_out apart from the inputs)");
    return CBS_ERR_ARG;
}

}  // namespace

extern "C" {

int cbs_max_u16(cbs_ctx *ctx, const uint64_t *in, int nvals, uint64_t *out)
{
    ENTER(ctx);
    if (nvals <= 0 || !in || !out) return set_error("cbs_max_u16: bad argument"), CBS_ERR_ARG;
    return max_u16(ctx, in, nvals, true, out);
}

// Mini-workload #2 of the harness (harness/cleartext_impl.py:65-70; no reference implementation exists, SURVEY.md
// 8(f)2): sum_i (x_i * y_i mod 2^16) mod 2^16 with x = first half, y = second half of the values.  The circuit
// (nibble products, column compression by population counts, nibble adders) is planned on the host by
// host/ip_plan.h and executed by run_lut_plan.
int cbs_inner_product_u16(cbs_ctx *ctx, const uint64_t *in, int nvals, uint64_t *out)
{
    ENTER(ctx);
    if (nvals <= 0 || (nvals & 1) || !in || !out) return set_error("cbs_inner_product_u16: bad argument (need an even number of values)"), CBS_ERR_ARG;
    return run_lut_plan(ctx, kPlanInnerProduct, nvals, in, nullptr, true, out);
}

// Sum of nvals 16-bit values mod 2^16 (the column-compression stage of the inner product alone): combines per-GPU
// partial inner products when the pairs are sharded across GPUs.
int cbs_sum_u16(cbs_ctx *ctx, const uint64_t *in, int nvals, uint64_t *out)
{
    ENTER(ctx);
    if (nvals <= 0 || !in || !out) return set_error("cbs_sum_u16: bad argument"), CBS_ERR_ARG;
    return run_lut_plan(ctx, kPlanSum, nvals, in, nullptr, true, out);
}

// Maximum as a LUT circuit (host/ip_plan.h max_make_plan): noise independent of the data and of the tree depth.
int cbs_max_u16_lut(cbs_ctx *ctx, const uint64_t *in, int nvals, uint64_t *out)
{
    ENTER(ctx);
    if (nvals <= 0 || !in || !out) return set_error("cbs_max_u16_lut: bad argument"), CBS_ERR_ARG;
    return run_lut_plan(ctx, kPlanMax, nvals, in, nullptr, true, out);
}

int cbs_max_u16_dev(cbs_ctx *ctx, const uint64_t *d_in, int nvals, uint64_t *d_out)
{
    ENTER(ctx);
    TRY(check_dev_args("cbs_max_u16_dev", nvals, d_in, nullptr, false, d_out));
    return max_u16(ctx, d_in, nvals, false, d_out);
}

int cbs_max_u16_lut_dev(cbs_ctx *ctx, const uint64_t *d_in, int nvals, uint64_t *d_out)
{
    ENTER(ctx);
    TRY(check_dev_args("cbs_max_u16_lut_dev", nvals, d_in, nullptr, false, d_out));
    return run_lut_plan(ctx, kPlanMax, nvals, d_in, nullptr, false, d_out);
}

int cbs_sum_u16_dev(cbs_ctx *ctx, const uint64_t *d_in, int nvals, uint64_t *d_out)
{
    ENTER(ctx);
    TRY(check_dev_args("cbs_sum_u16_dev", nvals, d_in, nullptr, false, d_out));
    return run_lut_plan(ctx, kPlanSum, nvals, d_in, nullptr, false, d_out);
}

int cbs_inner_product_u16_dev(cbs_ctx *ctx, const uint64_t *d_x, const uint64_t *d_y, int npairs, uint64_t *d_out)
{
    ENTER(ctx);
    TRY(check_dev_args("cbs_inner_product_u16_dev", npairs, d_x, d_y, true, d_out));
    return run_lut_plan(ctx, kPlanInnerProduct, 2 * npairs, d_x, d_y, false, d_out);
}

}  // extern "C"

// ---- LWE-to-GLWE packing: one core for the host-buffer and the device-resident call ----

namespace {

// count big LWE at `in` -> ceil(count / 1024) GLWE at `out` (host = true: host buffers, uploaded and downloaded around the
// kernels; otherwise device buffers and the work is only queued).  The tree levels live in the "pack_ws" workspace.
int pack_lwes(cbs_ctx *ctx, const uint64_t *in, int count, bool host, uint64_t *out)
{
    const size_t nglwe = ((size_t)count + 1023) / 1024;
    uint64_t *d_ws, *d_in = nullptr, *d_out = nullptr;
    TRY(ws_typed(ctx, "pack_ws", nglwe * std::min(count, 512) * kGlweWords, &d_ws));
    if (host) {
        TRY(ws_typed(ctx, "pack_in", (size_t)count * kLweBig, &d_in));
        TRY(ws_typed(ctx, "pack_out", nglwe * kGlweWords, &d_out));
        TRY(copy_in(ctx, d_in, in, (size_t)count * kLweBig * 8, true));
    }
    launch_pack_lwes(ctx->K, host ? d_in : in, d_ws, host ? d_out : out, count, ctx->stream);
    ctx->launches += 10;
    TRY(check_launch("k_pack_level"));
    return host ? download(ctx, out, d_out, nglwe * kGlweWords * 8) : CBS_OK;
}

}  // namespace

extern "C" {

int cbs_pack_lwes(cbs_ctx *ctx, const uint64_t *in_big, int count, uint64_t *glwe_out)
{
    ENTER(ctx);
    if (count < 0 || count > INT_MAX - 1023 || (count && (!in_big || !glwe_out))) return set_error("cbs_pack_lwes: bad argument"), CBS_ERR_ARG;
    if (count == 0) return CBS_OK;
    return pack_lwes(ctx, in_big, count, true, glwe_out);
}

int cbs_pack_lwes_dev(cbs_ctx *ctx, const uint64_t *d_in, int count, uint64_t *d_out)
{
    ENTER(ctx);
    const size_t in_words = (size_t)count * kLweBig, out_words = ((size_t)count + 1023) / 1024 * kGlweWords;
    if (count <= 0 || count > INT_MAX - 1023 || !d_in || !d_out || (d_out < d_in + in_words && d_in < d_out + out_words))
        return set_error("cbs_pack_lwes_dev: bad argument (need a positive count, non-null pointers and a d_out apart from d_in)"),
               CBS_ERR_ARG;
    return pack_lwes(ctx, d_in, count, false, d_out);
}

}  // extern "C"
