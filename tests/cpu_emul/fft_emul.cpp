// CPU emulation of the 64-thread fft512.cuh group: runs the very same phase functions the CUDA
// kernels call, looping over the logical threads between barrier points.  Checks
//   (1) inverse(forward(x)) == 512 * x  (unnormalised),
//   (2) pointwise product in the transform domain == negacyclic convolution mod X^1024 + 1,
//   (3) every 128-bit shared access pattern is bank-conflict free per quarter-warp.
// Exit code 0 on success.  Built and run by tests/test_fft_emulation.py (no GPU needed).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <initializer_list>
#include <cmath>
#include "fft_tables.h"
using namespace cbs;

static std::vector<double> g_tab;

static void forward(const std::vector<int64_t> &p, cplx out[64][8])
{
    static cplx scr[512];
    cplx v[64][8];
    Twiddles tw[64];
    for (int t = 0; t < 64; t++) {
        load_twiddles(tw[t], g_tab.data(), t);
        for (int m = 0; m < 8; m++) v[t][m] = {(double)p[t + 64 * m], (double)p[t + 64 * m + 512]};
    }
    for (int t = 0; t < 64; t++) fwd_p1(v[t], scr, tw[t], t);
    for (int t = 0; t < 64; t++) fwd_p2(v[t], scr, tw[t], t);  // in place: thread owns its 8 slots
    for (int t = 0; t < 64; t++) fwd_p3(v[t], scr, t);
    memcpy(out, v, sizeof(v));
}

static void inverse(cplx in[64][8], std::vector<double> &coef)
{
    static cplx scr[512];
    cplx v[64][8];
    Twiddles tw[64];
    memcpy(v, in, sizeof(v));
    for (int t = 0; t < 64; t++) load_twiddles(tw[t], g_tab.data(), t);
    for (int t = 0; t < 64; t++) inv_p3(v[t], scr, t);
    for (int t = 0; t < 64; t++) inv_p2(v[t], scr, tw[t], t);
    for (int t = 0; t < 64; t++) inv_p1(v[t], scr, tw[t], t);
    coef.assign(1024, 0.0);
    for (int t = 0; t < 64; t++)
        for (int m = 0; m < 8; m++) {
            coef[t + 64 * m] = v[t][m].x;
            coef[t + 64 * m + 512] = v[t][m].y;
        }
}

// shuffle-exchange variant: same phase code, the width-8 lane exchange emulated
static void exchange_emul(cplx v[64][8], int dir)
{
    cplx w[64][8];
    memcpy(w, v, sizeof(w));
    for (int t = 0; t < 64; t++)
        for (int r = 1; r < 8; r++) {
            int a = t & 7, src = (t & ~7) | ((a + dir * r) & 7);
            v[t][r] = w[src][r];
        }
}

static void forward_x(const std::vector<int64_t> &p, cplx out[64][8])
{
    static cplx scr[512];
    cplx v[64][8];
    Twiddles tw[64];
    for (int t = 0; t < 64; t++) {
        load_twiddles_x(tw[t], g_tab.data(), t);
        for (int m = 0; m < 8; m++) v[t][m] = {(double)p[t + 64 * m], (double)p[t + 64 * m + 512]};
    }
    for (int t = 0; t < 64; t++) fwd_p1(v[t], scr, tw[t], t);
    for (int t = 0; t < 64; t++) fwd_p2x(v[t], scr, tw[t], t);
    exchange_emul(v, -1);
    for (int t = 0; t < 64; t++) fwd_p3x(v[t]);
    memcpy(out, v, sizeof(v));
}

static void inverse_x(cplx in[64][8], std::vector<double> &coef)
{
    static cplx scr[512];
    cplx v[64][8];
    Twiddles tw[64];
    memcpy(v, in, sizeof(v));
    for (int t = 0; t < 64; t++) load_twiddles_x(tw[t], g_tab.data(), t);
    for (int t = 0; t < 64; t++) inv_p3x(v[t]);
    exchange_emul(v, +1);
    for (int t = 0; t < 64; t++) inv_p2x(v[t], scr, tw[t], t);
    for (int t = 0; t < 64; t++) inv_p1(v[t], scr, tw[t], t);
    coef.assign(1024, 0.0);
    for (int t = 0; t < 64; t++)
        for (int m = 0; m < 8; m++) {
            coef[t + 64 * m] = v[t][m].x;
            coef[t + 64 * m + 512] = v[t][m].y;
        }
}

static int check_banks()
{
    // a quarter-warp (8 consecutive lanes) must touch 8 distinct 16-byte slots modulo 8
    int bad = 0;
    for (int q = 0; q < 8; q++) {
        for (int i = 0; i < 8; i++) {  // i = register index in the access loop
            int seen1 = 0, seen2 = 0, seen3 = 0;
            for (int l = 0; l < 8; l++) {
                int t = q * 8 + l;
                seen1 |= 1 << (slot(i, t & 7, t >> 3) & 7);  // p1 store / inv_p1 load
                seen2 |= 1 << (slot(t >> 3, t & 7, i) & 7);  // p2 load/store
                seen3 |= 1 << (slot(t >> 3, i, t & 7) & 7);  // p3 load / inv_p3 store
            }
            if (seen1 != 255 || seen2 != 255 || seen3 != 255) bad++;
        }
    }
    return bad;
}

int main()
{
    g_tab = make_twiddle_table();
    srand(7);
    std::vector<int64_t> a(1024), b(1024);
    for (int i = 0; i < 1024; i++) {
        a[i] = (rand() % 2001) - 1000;
        b[i] = (rand() % 2001) - 1000;
    }
    cplx fa[64][8], fb[64][8], fc[64][8];
    forward(a, fa);
    forward(b, fb);
    // (1) round trip
    std::vector<double> back;
    inverse(fa, back);
    double e1 = 0;
    for (int i = 0; i < 1024; i++) e1 = fmax(e1, fabs(back[i] / 512.0 - (double)a[i]));
    // (2) convolution
    for (int t = 0; t < 64; t++)
        for (int k = 0; k < 8; k++) fc[t][k] = cmul(fa[t][k], fb[t][k]);
    std::vector<double> conv;
    inverse(fc, conv);
    std::vector<double> ref(1024, 0.0);
    for (int i = 0; i < 1024; i++)
        for (int j = 0; j < 1024; j++) {
            int k = i + j;
            double p = (double)a[i] * (double)b[j];
            if (k >= 1024) ref[k - 1024] -= p;
            else ref[k] += p;
        }
    double e2 = 0;
    for (int i = 0; i < 1024; i++) e2 = fmax(e2, fabs(conv[i] / 512.0 - ref[i]));
    // (2b) bin identity: thread u slot k3 must be DFT bin k1 + 8*k2 + 64*k3 of the twisted fold
    double e3 = 0;
    for (int u = 0; u < 64; u += 13)
        for (int k3 = 0; k3 < 8; k3 += 3) {
            int k = (u >> 3) + 8 * (u & 7) + 64 * k3;
            long double sr = 0, si = 0;
            for (int j = 0; j < 512; j++) {
                long double ang = 3.14159265358979323846264338327950288L * j / 1024.0L - 2.0L * 3.14159265358979323846264338327950288L * (long double)((j * k) % 512) / 512.0L;
                long double cr = cosl(ang), ci = sinl(ang);
                sr += a[j] * cr - a[j + 512] * ci;
                si += a[j] * ci + a[j + 512] * cr;
            }
            e3 = fmax(e3, fmax(fabs((double)sr - fa[u][k3].x), fabs((double)si - fa[u][k3].y)));
        }
    // (3) shuffle-exchange variant: round trip, and data through forward_x/inverse_x multiplied by a key
    //     spectrum from the PLAIN forward transform must still give the negacyclic convolution
    double e4 = 0, e5 = 0;
    {
        cplx xa[64][8], xc[64][8];
        forward_x(a, xa);
        std::vector<double> bx;
        inverse_x(xa, bx);
        for (int i = 0; i < 1024; i++) e4 = fmax(e4, fabs(bx[i] / 512.0 - (double)a[i]));
        for (int t = 0; t < 64; t++)
            for (int k = 0; k < 8; k++) xc[t][k] = cmul(xa[t][k], fb[t][k]);
        std::vector<double> cx;
        inverse_x(xc, cx);
        for (int i = 0; i < 1024; i++) e5 = fmax(e5, fabs(cx[i] / 512.0 - ref[i]));
    }
    int bad = check_banks();
    // (4) helpers
    int bad_dec = 0;
    for (int i = 0; i < 100000; i++) {
        uint64_t x = ((uint64_t)rand() << 42) ^ ((uint64_t)rand() << 21) ^ (uint64_t)rand();
        for (int cfg = 0; cfg < 4; cfg++) {
            const int bl[4] = {23, 13, 17, 2}, lv[4] = {1, 3, 2, 7};
            uint64_t st = decomp_init(x, bl[cfg], lv[cfg]);
            __int128 recon = 0;
            for (int t = 0; t < lv[cfg]; t++) {
                int32_t d = decomp_next(st, bl[cfg]);
                if (d < -(1 << (bl[cfg] - 1)) || d > (1 << (bl[cfg] - 1))) bad_dec++;
                int lev = lv[cfg] - t;  // level index 1..l, finest first
                recon += (__int128)d << (64 - bl[cfg] * lev);
            }
            uint64_t r = (uint64_t)recon;
            int nr = 64 - bl[cfg] * lv[cfg];
            uint64_t closest = ((x >> nr) + ((x >> (nr - 1)) & 1)) << nr;
            if (r != closest) bad_dec++;
        }
        // the blind rotation's one-level digit from the high word only
        for (uint64_t y : std::initializer_list<uint64_t>{x, x | 0xffffff0000000000ull, x & 0x000000ffffffffffull, (x & 0xffffffffffull) | 0x7fffff0000000000ull,
                           (x & 0xffffffffffull) | 0x8000000000000000ull, (x & 0xffffffffffull) | 0x7fffff8000000000ull}) {
            uint64_t st = decomp_init(y, 23, 1);
            if (decomp_next(st, 23) != digit_b23_l1_hi((uint32_t)(y >> 32))) bad_dec++;
        }
    }
    int bad_tor = 0;
    for (int i = 0; i < 100000; i++) {
        double r = ((double)rand() / RAND_MAX - 0.5) * ldexp(1.0, 64 + (rand() % 30));
        uint64_t got = torus_from_scaled(r);
        long double fr = (long double)r / 18446744073709551616.0L;
        fr -= roundl(fr);
        long double want = roundl(fr * 18446744073709551616.0L);
        uint64_t w = (want >= 9223372036854775808.0L) ? 0x7FFFFFFFFFFFFFFFull : (uint64_t)(int64_t)want;  // saturates like the device
        if (got != w) bad_tor++;
    }
    printf("roundtrip_err=%.3e conv_err=%.3e bin_err=%.3e x_roundtrip_err=%.3e x_conv_err=%.3e bank_conflicts=%d bad_decomp=%d bad_torus=%d\n",
           e1, e2, e3, e4, e5, bad, bad_dec, bad_tor);
    return (e1 < 1e-9 && e2 < 1e-3 && e3 < 1e-6 && e4 < 1e-9 && e5 < 1e-3 && bad == 0 && bad_dec == 0 && bad_tor == 0) ? 0 : 1;
}
