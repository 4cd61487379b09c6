// device_helpers.cu — the integer glue of the FFT kernels (csrc/digits.cuh, csrc/fft512.cuh) run on the device and
// compared with plain integer arithmetic.  Built and run by tests/test_exact_gpu.py:
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I<csrc> device_helpers.cu
// Every check counts mismatches and keeps the first one; the program prints one line per check and exits 0 when all
// counts are as expected.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include <random>
#include <vector>

#include "digits.cuh"

using namespace cbs;

struct Result {
    unsigned long long bad;
    unsigned long long first;  // the first failing input (smallest index wins)
    unsigned long long got, want;
};

__device__ void report(Result *r, unsigned long long input, unsigned long long got, unsigned long long want)
{
    atomicAdd(&r->bad, 1ull);
    if (atomicMin(&r->first, input) > input) {
        r->got = got;
        r->want = want;
    }
}

// reference digit of the one-level B = 2^23 decomposition: the generic decomposer on the full word hi:0
__device__ int32_t ref_b23(uint32_t hi)
{
    uint64_t st = decomp_init((uint64_t)hi << 32, 23, 1);
    return decomp_next(st, 23);
}

// every 32-bit input: digit_b23_l1_double and digit_b23_l1_hi against the generic decomposer, i32_to_double against
// the conversion instruction
__global__ void k_all_words(Result *r)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (1ull << 32); i += stride) {
        const uint32_t w = (uint32_t)i;
        const int32_t want = ref_b23(w);
        const double d = digit_b23_l1_double(w);
        if (d != (double)want) report(&r[0], i, __double_as_longlong(d), (unsigned long long)(int64_t)want);
        if (digit_b23_l1_hi(w) != want) report(&r[1], i, (unsigned long long)(int64_t)digit_b23_l1_hi(w), (unsigned long long)(int64_t)want);
        const double c = i32_to_double((int32_t)w);
        if (c != (double)(int32_t)w) report(&r[2], i, __double_as_longlong(c), __double_as_longlong((double)(int32_t)w));
    }
}

__device__ uint64_t mix(uint64_t x)
{
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// hi_condneg_sub against u64 arithmetic: random words, plus the borrow edges (x = 0, x = 2^63, low words equal, ~0)
__global__ void k_condneg(Result *r, uint64_t n)
{
    const uint64_t edge[6] = {0ull, 1ull << 63, 0xFFFFFFFFFFFFFFFFull, 0x00000000FFFFFFFFull, 0xFFFFFFFF00000000ull, 1ull};
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        uint64_t x = mix(3 * i), o = mix(3 * i + 1);
        const uint64_t sel = mix(3 * i + 2);
        if ((sel & 7) == 0) x = edge[(sel >> 3) % 6];
        if (((sel >> 8) & 7) == 0) o = edge[(sel >> 11) % 6];
        if (((sel >> 16) & 7) == 0) o = (o & ~0xFFFFFFFFull) | (x & 0xFFFFFFFFull);  // xl = ol: the low word cancels
        const uint64_t m = (sel >> 24) & 1 ? ~0ull : 0ull;
        const uint32_t got = hi_condneg_sub((uint32_t)x, (uint32_t)(x >> 32), (uint32_t)m, (uint32_t)o, (uint32_t)(o >> 32));
        const uint32_t want = (uint32_t)((((x ^ m) - m) - o) >> 32);
        if (got != want) report(r, i, got, want);
    }
}

// pack_digits / unpack_digit against decomp_init / decomp_next: random words, plus every rounding tie (the bit below the
// kept bits, and raw digit B/2 at each level with the next raw digit below and at B/2), each +-1
template <int B, int L, typename PackT>
__global__ void k_pack(Result *r, uint64_t n)
{
    constexpr int nr = 64 - B * L;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        uint64_t x = mix(i);
        const uint64_t sel = mix(i ^ 0x5555555555555555ull);
        if ((sel & 3) == 0) {
            const int t = (int)((sel >> 2) % L);
            uint64_t w = 1ull << (nr + B * t + B - 1);                              // raw digit B/2 at level t
            if ((sel >> 8) & 1 && t + 1 < L) w += 1ull << (nr + B * (t + 1) + B - 1);  // next raw digit B/2
            if ((sel >> 9) & 1) w += 1ull << (nr - 1);                               // closest-representable tie
            w += (uint64_t)((int64_t)((sel >> 10) % 3) - 1);                         // -1, 0, +1
            x = ((sel >> 12) & 1) ? w : (x & (~0ull << (nr + B * t))) + w;  // random digits above level t
        }
        const PackT p = pack_digits<B, L, PackT>(x);
        uint64_t st = decomp_init(x, B, L);
        for (int tt = 0; tt < L; tt++) {
            const int32_t want = decomp_next(st, B);
            const int32_t got = unpack_digit<B, PackT>(p, tt);
            if (got != want) {
                report(r, i, (unsigned long long)(int64_t)got, (unsigned long long)(int64_t)want);
                break;
            }
        }
    }
}

__global__ void k_torus(const double *in, uint64_t *out, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = torus_from_scaled(in[i]);
}

static int check(const char *name, const Result &r, unsigned long long expect_bad = 0)
{
    printf("%s mismatches=%llu", name, r.bad);
    if (r.bad) printf(" first_input=%#llx got=%#llx want=%#llx", r.first, r.got, r.want);
    printf("\n");
    return r.bad == expect_bad ? 0 : 1;
}

#define CK(x)                                                                            \
    do {                                                                                 \
        cudaError_t e_ = (x);                                                            \
        if (e_ != cudaSuccess) {                                                         \
            printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); \
            return 2;                                                                    \
        }                                                                                \
    } while (0)

int main()
{
    Result *d_r;
    const int nres = 8;
    CK(cudaMalloc(&d_r, sizeof(Result) * nres));
    std::vector<Result> init(nres, Result{0, ~0ull, 0, 0});
    CK(cudaMemcpy(d_r, init.data(), sizeof(Result) * nres, cudaMemcpyHostToDevice));
    const uint64_t n = 1ull << 26;
    k_all_words<<<148 * 8, 256>>>(d_r);
    k_condneg<<<148 * 8, 256>>>(d_r + 3, n);
    k_pack<2, 7, uint32_t><<<148 * 8, 256>>>(d_r + 4, n);
    k_pack<13, 3, uint64_t><<<148 * 8, 256>>>(d_r + 5, n);
    k_pack<17, 2, uint64_t><<<148 * 8, 256>>>(d_r + 6, n);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    std::vector<Result> res(nres);
    CK(cudaMemcpy(res.data(), d_r, sizeof(Result) * nres, cudaMemcpyDeviceToHost));
    int fail = 0;
    fail |= check("digit_b23_l1_double(all 2^32)", res[0]);
    fail |= check("digit_b23_l1_hi(all 2^32)", res[1]);
    fail |= check("i32_to_double(all 2^32)", res[2]);
    fail |= check("hi_condneg_sub", res[3]);
    fail |= check("pack_digits<2,7>", res[4]);
    fail |= check("pack_digits<13,3>", res[5]);
    fail |= check("pack_digits<17,2>", res[6]);

    // torus_from_scaled against exact rounding to the nearest integer (halves to even) mod 2^64, computed in int128 on the
    // host.  Inputs: r = k 2^64 +- 2^63 (the reduction's ties), +-0.5, +-1.5, -0.0, and random r with |r| up to 2^100.
    std::vector<double> in;
    for (int e = 0; e <= 36; e++)
        for (double k : {0.0, 1.0, 3.0, -1.0, -2.0})
            for (double s : {1.0, -1.0}) in.push_back(ldexp(k, 64 + e) + s * 0x1p63);  // exact: 39 significant bits at most
    for (double v : {0.5, -0.5, 1.5, -1.5, -0.0, 0.0, 0x1p63, -0x1p63, 0x1p64, -0x1p64, 0x1p63 - 1024.0, 0.49999999999999994})
        in.push_back(v);
    std::mt19937_64 g(7);
    for (int i = 0; i < 1 << 20; i++) {
        const double m = std::ldexp((double)(g() >> 11), -53) * ((g() & 1) ? 1.0 : -1.0);  // |m| < 1, 53 bits
        in.push_back(std::ldexp(m, (int)(g() % 101)));
    }
    const int nt = (int)in.size();
    double *d_in;
    uint64_t *d_out;
    CK(cudaMalloc(&d_in, sizeof(double) * nt));
    CK(cudaMalloc(&d_out, sizeof(uint64_t) * nt));
    CK(cudaMemcpy(d_in, in.data(), sizeof(double) * nt, cudaMemcpyHostToDevice));
    k_torus<<<(nt + 255) / 256, 256>>>(d_in, d_out, nt);
    CK(cudaGetLastError());
    std::vector<uint64_t> out(nt);
    CK(cudaMemcpy(out.data(), d_out, sizeof(uint64_t) * nt, cudaMemcpyDeviceToHost));
    Result tr{0, ~0ull, 0, 0}, dev{0, ~0ull, 0, 0};
    unsigned long long expect_dev = 0;
    for (int i = 0; i < nt; i++) {
        const __int128 v = (__int128)nearbyint(in[i]);  // exact: |r| < 2^101
        const uint64_t want = (uint64_t)v;
        // the one documented deviation (DESIGN.md section 2): r = 2^63 mod 2^65 reduces to f = +2^63, which the
        // conversion saturates to 2^63 - 1
        const bool tie_up = ((v - ((__int128)1 << 63)) & (((__int128)1 << 65) - 1)) == 0;
        expect_dev += tie_up;
        const uint64_t want_dev = tie_up ? 0x7FFFFFFFFFFFFFFFull : want;
        if (out[i] != want_dev) {
            if (!tr.bad) tr = Result{0, (unsigned long long)i, out[i], want_dev};
            tr.bad++;
        }
        if (out[i] != want) dev.bad++;
    }
    fail |= check("torus_from_scaled", tr);
    printf("torus_from_scaled inputs=%d deviations_at_f_plus_2^63=%llu expected=%llu\n", nt, dev.bad, expect_dev);
    fail |= (dev.bad != expect_dev || expect_dev == 0);
    cudaFree(d_in);
    cudaFree(d_out);
    cudaFree(d_r);
    printf(fail ? "FAIL\n" : "OK\n");
    return fail;
}
