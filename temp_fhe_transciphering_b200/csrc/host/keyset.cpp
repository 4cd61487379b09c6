// keyset.cpp — host side of libcbs_b200: the reference's io/ file formats (bincode 1.3) and the
// client-side helpers (seeded key generation, transciphering-key encoder, bit encryption).
//
// Formats: SURVEY.md 8(b); types serialised by src/bin/client_key_generation.rs:114-129,
// src/bin/client_encode_encrypt.rs:55-62, src/bin/server_encrypted_aes_decryption.rs:700-704.
// Key semantics: cbs_lib/src/keygen.rs:187-243 (bsk, ksk), cbs_lib/src/automorphism.rs:59-178
// (automorphism keys), cbs_lib/src/ggsw_conv.rs:15-77 (scheme-switching key),
// cbs_lib/src/glwe_keyswitch.rs:183-218 (GLWE keyswitch key = GLEV of -S_in),
// src/data_struct.rs:30-269 + src/aes_manager.rs:163-432 (AllRdKeys tables).
#include "cbs_b200.h"
#include "chacha20.h"
#include "host_common.h"
#include "ip_plan.h"

#include <algorithm>
#include <array>
#include <cmath>
#include <complex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <string>
#include <sys/random.h>
#include <sys/stat.h>
#include <thread>
#include <vector>

namespace cbs_host {

thread_local std::string g_last_error;
void set_error(const std::string &s) { g_last_error = s; }

// ------------------------------------------------------------------------------------------------
// bincode cursor
struct Reader {
    std::vector<uint8_t> buf;
    size_t off = 0;
    bool ok = true;
    bool load(const std::string &path)
    {
        std::ifstream f(path, std::ios::binary | std::ios::ate);
        if (!f) return false;
        std::streamsize n = f.tellg();
        f.seekg(0);
        buf.resize((size_t)n);
        return (bool)f.read(reinterpret_cast<char *>(buf.data()), n);
    }
    uint64_t u64()
    {
        if (off + 8 > buf.size()) {
            ok = false;
            return 0;
        }
        uint64_t v;
        memcpy(&v, buf.data() + off, 8);
        off += 8;
        return v;
    }
    bool vec(std::vector<uint64_t> &out, uint64_t expect)
    {
        uint64_t n = u64();
        if (!ok || n != expect || off + 8 * n > buf.size()) {
            ok = false;
            return false;
        }
        out.resize(n);
        memcpy(out.data(), buf.data() + off, 8 * n);
        off += 8 * n;
        return true;
    }
    bool vec_into(uint64_t *dst, uint64_t expect)
    {
        uint64_t n = u64();
        if (!ok || n != expect || off + 8 * n > buf.size()) {
            ok = false;
            return false;
        }
        memcpy(dst, buf.data() + off, 8 * n);
        off += 8 * n;
        return true;
    }
    void expect(uint64_t v)
    {
        if (u64() != v) ok = false;
    }
    void modulus()
    {  // CiphertextModulus<u64> native: u128 0, then scalar bits 64
        expect(0);
        expect(0);
        expect(64);
    }
    bool done() const { return ok && off == buf.size(); }
};

struct Writer {
    std::vector<uint8_t> buf;
    void u64(uint64_t v)
    {
        size_t o = buf.size();
        buf.resize(o + 8);
        memcpy(buf.data() + o, &v, 8);
    }
    void vec(const uint64_t *p, uint64_t n)
    {
        u64(n);
        size_t o = buf.size();
        buf.resize(o + 8 * n);
        memcpy(buf.data() + o, p, 8 * n);
    }
    void modulus()
    {
        u64(0);
        u64(0);
        u64(64);
    }
    bool save(const std::string &path) const
    {
        std::ofstream f(path, std::ios::binary);
        if (!f) return false;
        f.write(reinterpret_cast<const char *>(buf.data()), (std::streamsize)buf.size());
        return (bool)f;
    }
};

static void mkdirs(const std::string &path)
{
    std::string cur;
    for (size_t i = 0; i <= path.size(); i++) {
        if (i == path.size() || path[i] == '/') {
            if (!cur.empty()) mkdir(cur.c_str(), 0755);
        }
        if (i < path.size()) cur.push_back(path[i]);
    }
}

// ------------------------------------------------------------------------------------------------
// natural-order 512-point transform used only for the on-disk form of the automorphism keys
// (tfhe forward_as_torus convention, SURVEY.md 8(b) note 1)
using cd = std::complex<double>;
static void fft512_natural(std::vector<cd> &a, bool inverse)
{
    const int n = 512;
    for (int i = 1, j = 0; i < n; i++) {
        int bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) std::swap(a[i], a[j]);
    }
    static std::vector<cd> w;
    if (w.empty()) {
        w.resize(n / 2);
        for (int k = 0; k < n / 2; k++) {
            long double ang = -2.0L * 3.14159265358979323846264338327950288L * k / n;
            w[k] = cd((double)cosl(ang), (double)sinl(ang));
        }
    }
    for (int len = 2; len <= n; len <<= 1) {
        int step = n / len;
        for (int i = 0; i < n; i += len)
            for (int j = 0; j < len / 2; j++) {
                cd tw = inverse ? std::conj(w[j * step]) : w[j * step];
                cd u = a[i + j], v = a[i + j + len / 2] * tw;
                a[i + j] = u + v;
                a[i + j + len / 2] = u - v;
            }
    }
    if (inverse)
        for (auto &x : a) x /= (double)n;
}
static const std::vector<cd> &twist1024()
{
    static std::vector<cd> t;
    if (t.empty()) {
        t.resize(512);
        for (int j = 0; j < 512; j++) {
            long double ang = 3.14159265358979323846264338327950288L * j / 1024.0L;
            t[j] = cd((double)cosl(ang), (double)sinl(ang));
        }
    }
    return t;
}
static void limb_to_fourier(const uint64_t *limb /*1024*/, double *out /*1024 (re,im)*/)
{
    const auto &tw = twist1024();
    std::vector<cd> z(512);
    for (int j = 0; j < 512; j++)
        z[j] = cd((double)(int64_t)limb[j] * 0x1p-64, (double)(int64_t)limb[j + 512] * 0x1p-64) * tw[j];
    fft512_natural(z, false);
    for (int j = 0; j < 512; j++) {
        out[2 * j] = z[j].real();
        out[2 * j + 1] = z[j].imag();
    }
}
// returns max distance of the recovered coefficients from integers (sanity of the FFT ordering)
static double fourier_to_limb(const double *in, uint64_t *limb, double max_value)
{
    const auto &tw = twist1024();
    std::vector<cd> z(512);
    for (int j = 0; j < 512; j++) z[j] = cd(in[2 * j], in[2 * j + 1]);
    fft512_natural(z, true);
    double worst = 0;
    for (int j = 0; j < 512; j++) {
        cd v = z[j] * std::conj(tw[j]) * 0x1p64;
        double re = v.real(), im = v.imag();
        double rr = std::nearbyint(re), ri = std::nearbyint(im);
        worst = std::max(worst, std::max(std::fabs(re - rr), std::fabs(im - ri)));
        if (rr < 0 || rr >= max_value || ri < 0 || ri >= max_value) worst = 1e30;
        limb[j] = (uint64_t)rr;
        limb[j + 512] = (uint64_t)ri;
    }
    return worst;
}

// ------------------------------------------------------------------------------------------------
// randomness.  Two engines behind one interface, both as independent streams keyed by a stream id so results do not
// depend on threading:
//   * RngSource(seed): xoshiro256++ - deterministic, NOT cryptographically secure; only for reproducible tests, benches
//     and golden vectors (explicit seed argument / CBS_SEED);
//   * RngSource::os_entropy(): ChaCha20 (RFC 8439 block function) keyed with 256 bits from getrandom(2), stream id as
//     nonce - what the stage executables use when no seed is given, like the reference's own client
//     (client_key_generation.rs:91-96 new_seeder(); harness/run_submission.py:74-77: keys differ on every run).
static bool os_random(void *dst, size_t bytes)
{
    size_t got = 0;
    unsigned char *p = static_cast<unsigned char *>(dst);
    while (got < bytes) {
        ssize_t n = getrandom(p + got, bytes - got, 0);
        if (n <= 0) return false;
        got += (size_t)n;
    }
    return true;
}

struct RngSource {
    bool secure = false;
    uint64_t seed = 0;
    uint32_t key[8] = {0};
    explicit RngSource(uint64_t s) : seed(s) {}
    static bool os_entropy(RngSource &out)
    {
        out.secure = true;
        return os_random(out.key, sizeof out.key);
    }
};

struct Rng {
    bool secure;
    uint64_t s[4];             // xoshiro256++ state
    uint32_t cc[16];           // ChaCha20 input block (constants, key, counter, nonce)
    uint64_t buf[8];
    int have = 0;
    static uint64_t splitmix(uint64_t &x)
    {
        uint64_t z = (x += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    Rng(const RngSource &src, uint64_t stream) : secure(src.secure)
    {
        if (secure) {
            cc[0] = 0x61707865, cc[1] = 0x3320646e, cc[2] = 0x79622d32, cc[3] = 0x6b206574;  // "expand 32-byte k"
            for (int i = 0; i < 8; i++) cc[4 + i] = src.key[i];
            cc[12] = 0;
            cc[13] = (uint32_t)stream;
            cc[14] = (uint32_t)(stream >> 32);
            cc[15] = 0;
        } else {
            uint64_t x = src.seed * 0xD1342543DE82EF95ull + stream * 0xA0761D6478BD642Full + 0x1234567ull;
            for (auto &v : s) v = splitmix(x);
        }
    }
    static uint64_t rotl(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
    void chacha_block()
    {
        uint32_t x[16];
        cbs_chacha::block(cc, x);
        for (int i = 0; i < 8; i++) buf[i] = (uint64_t)x[2 * i] | ((uint64_t)x[2 * i + 1] << 32);
        if (++cc[12] == 0) cc[15]++;  // 2^32 blocks of 64 bytes per (stream, cc[15]): far beyond any use here
        have = 8;
    }
    uint64_t next()
    {
        if (secure) {
            if (!have) chacha_block();
            return buf[--have];
        }
        uint64_t r = rotl(s[0] + s[3], 23) + s[0];
        uint64_t t = s[1] << 17;
        s[2] ^= s[0];
        s[3] ^= s[1];
        s[1] ^= s[2];
        s[0] ^= s[3];
        s[2] ^= t;
        s[3] = rotl(s[3], 45);
        return r;
    }
    double uniform() { return ((double)(next() >> 11) + 0.5) * 0x1p-53; }
    double gauss()
    {
        double u1 = uniform(), u2 = uniform();
        return std::sqrt(-2.0 * std::log(u1)) * std::cos(6.283185307179586476925 * u2);
    }
    uint64_t noise(double std_torus) { return (uint64_t)(int64_t)std::nearbyint(gauss() * std_torus * 0x1p64); }
};

constexpr double kStdLwe = 0.00000702047462940120;               // aes_instances.rs:78
constexpr double kStdGlwe = 0.00000000000000029403601535432533;  // aes_instances.rs:81

// body += a * s  (negacyclic, binary s)
static void add_mul_binary(uint64_t *body, const uint64_t *a, const uint64_t *s, int N)
{
    for (int i = 0; i < N; i++) {
        if (!s[i]) continue;
        for (int j = i; j < N; j++) body[j] += a[j - i];
        for (int j = 0; j < i; j++) body[j] -= a[N + j - i];
    }
}

// fresh GLWE encryption: ct = (a_0..a_{k-1}, sum a_c * s_c + e + pt); the mask a is drawn from rng, or, with
// mask_given, is what ct already holds (the seeded keys' public mask stream; the noise still comes from rng)
static void glwe_encrypt(uint64_t *ct, const uint64_t *pt /*N or null*/, const uint64_t *sk, int k, int N, double std,
                         Rng &rng, bool mask_given = false)
{
    if (!mask_given)
        for (int i = 0; i < k * N; i++) ct[i] = rng.next();
    uint64_t *body = ct + (size_t)k * N;
    for (int j = 0; j < N; j++) body[j] = rng.noise(std) + (pt ? pt[j] : 0ull);
    for (int c = 0; c < k; c++) add_mul_binary(body, ct + (size_t)c * N, sk + (size_t)c * N, N);
}

static void eval_x_k(uint64_t *out, const uint64_t *in, int N, unsigned kappa)
{
    for (int i = 0; i < N; i++) {
        unsigned long prod = (unsigned long)i * kappa;
        int j = (int)(prod % (unsigned)N);
        out[j] = ((prod / (unsigned)N) & 1) ? (0ull - in[i]) : in[i];
    }
}

static void parallel_for(int n, const std::function<void(int)> &fn)
{
    unsigned nt = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    std::vector<std::thread> th;
    for (unsigned w = 0; w < nt; w++)
        th.emplace_back([&, w]() {
            for (int i = (int)w; i < n; i += (int)nt) fn(i);
        });
    for (auto &t : th) t.join();
}

// ------------------------------------------------------------------------------------------------
// AES tables (src/aes_manager.rs)
static uint8_t gmul(uint8_t a, uint8_t b)
{
    uint8_t r = 0;
    while (b) {
        if (b & 1) r ^= a;
        a = (uint8_t)((a << 1) ^ ((a & 0x80) ? 0x1B : 0));
        b >>= 1;
    }
    return r;
}
struct AesTables {
    uint8_t sbox[256], inv[256];
    uint8_t rk[11][16];
    AesTables(const uint8_t key[16])
    {
        // S-box from the field inverse + affine map
        uint8_t invf[256] = {0};
        for (int x = 1; x < 256; x++)
            for (int y = 1; y < 256; y++)
                if (gmul((uint8_t)x, (uint8_t)y) == 1) invf[x] = (uint8_t)y;
        for (int x = 0; x < 256; x++) {
            uint8_t b = invf[x], r = 0;
            for (int i = 0; i < 8; i++) {
                int bit = ((b >> i) ^ (b >> ((i + 4) % 8)) ^ (b >> ((i + 5) % 8)) ^ (b >> ((i + 6) % 8)) ^
                           (b >> ((i + 7) % 8)) ^ (0x63 >> i)) & 1;
                r |= (uint8_t)(bit << i);
            }
            sbox[x] = r;
        }
        for (int x = 0; x < 256; x++) inv[sbox[x]] = (uint8_t)x;
        // key schedule, round key byte index = 4*col + row (aes_manager.rs:163-205)
        static const uint8_t rcon[11] = {0, 1, 2, 4, 8, 16, 32, 64, 128, 0x1B, 0x36};
        memcpy(rk[0], key, 16);
        for (int r = 1; r <= 10; r++) {
            const uint8_t *p = rk[r - 1];
            uint8_t t[4] = {sbox[p[13]], sbox[p[14]], sbox[p[15]], sbox[p[12]]};
            t[0] ^= rcon[r];
            for (int row = 0; row < 4; row++) rk[r][row] = p[row] ^ t[row];
            for (int col = 1; col < 4; col++)
                for (int row = 0; row < 4; row++) rk[r][4 * col + row] = p[4 * col + row] ^ rk[r][4 * (col - 1) + row];
        }
    }
    // get_10_9_round_lut (aes_manager.rs:338-396), before the GF multiples
    void lut_10_9(uint8_t t[16][256]) const
    {
        for (int col = 0; col < 4; col++)
            for (int row = 0; row < 4; row++) {
                int src = 4 * ((4 + col - row) % 4) + row;
                for (int x = 0; x < 256; x++) t[4 * col + row][x] = inv[x ^ rk[10][src]] ^ rk[9][4 * col + row];
            }
    }
    // forward keyed S-box of round r+1: S(x ^ rk_r[b]) (cbs_lib/src/aes_ref.rs:334-380 get_keyed_sbox*)
    void lut_fwd(int prev_round, uint8_t t[16][256]) const
    {
        for (int b = 0; b < 16; b++)
            for (int x = 0; x < 256; x++) t[b][x] = sbox[x ^ rk[prev_round][b]];
    }
    // last round: S(x ^ rk9[b]) ^ rk10[position b lands on after ShiftRows]
    void lut_fwd_last(uint8_t t[16][256]) const
    {
        for (int col = 0; col < 4; col++)
            for (int row = 0; row < 4; row++) {
                const int b = 4 * col + row, dst = 4 * ((col - row + 4) % 4) + row;
                for (int x = 0; x < 256; x++) t[b][x] = sbox[x ^ rk[9][b]] ^ rk[10][dst];
            }
    }
    // get_round_lut / get_0_round_lut (aes_manager.rs:398-432)
    void lut_round(int round, uint8_t t[16][256]) const
    {
        for (int b = 0; b < 16; b++)
            for (int x = 0; x < 256; x++) t[b][x] = inv[x] ^ rk[round][b];
    }
};

// accumulator plaintext of generate_vec_keyed_lut_accumulator (cbs_lib/src/aes_he.rs:835-875) and
// src/data_struct.rs:140-150: coefficient i carries bit (acc_idx*4 + i/256) of table[i % 256] at 2^63
static void lut_plaintext(uint64_t *pt, const uint8_t table[256], int acc_idx, uint8_t mult)
{
    for (int i = 0; i < 1024; i++) {
        int lut_idx = acc_idx * 4 + i / 256;
        uint8_t v = mult ? gmul(table[i % 256], mult) : table[i % 256];
        pt[i] = (uint64_t)((v >> lut_idx) & 1) << 63;
    }
}

}  // namespace cbs_host

using namespace cbs_host;

// The keyed tables of direction `dir` in AllRdKeys order: [0] the first round, [1 + i] middle block i, [9] the last round.
// Inverse get_10_9_round_lut / get_round_lut / get_0_round_lut (aes_manager.rs:338-432), forward S(x ^ rk0) / S(x ^ rk_i) /
// the last round (cbs_lib/src/aes_ref.rs:334-380).  Middle block i is keyed with round key i + 1.
static void aes_key_tables(AesDir dir, const uint8_t aes_key[16], uint8_t tab[10][16][256])
{
    const bool inv = dir == kAesInv;
    AesTables aes(aes_key);
    inv ? aes.lut_10_9(tab[0]) : aes.lut_fwd(0, tab[0]);
    for (int i = 0; i < 8; i++) inv ? aes.lut_round(i + 1, tab[1 + i]) : aes.lut_fwd(i + 1, tab[1 + i]);
    inv ? aes.lut_round(0, tab[9]) : aes.lut_fwd_last(tab[9]);
}

// GLWE g of the direction's AllRdKeys order (first [nmult][16][2], middle [8][nmult][16][2], last [16][2], G GLWE in all): its
// plaintext, and where it sits in the three key arrays
static void aes_key_lut_plaintext(const AesDirDesc &d, const uint8_t tab[10][16][256], int g, uint64_t *pt)
{
    const int F = d.nmult * 32, round = g < F ? 0 : g < 9 * F ? 1 + (g - F) / F : 9;
    const int id = round == 0 ? g : round < 9 ? (g - F) % F : g - 9 * F;
    const int a = id & 1, b = (id >> 1) & 15, m = id >> 5;
    lut_plaintext(pt, tab[round][b], a, round == 9 ? 0 : d.mults[m]);
}
template <typename P>
static P aes_key_glwe(const AesDirDesc &d, int g, P first, P mid, P last)
{
    const int F = d.nmult * 32;
    return g < F ? first + (size_t)g * 3072 : g < 9 * F ? mid + (size_t)(g - F) * 3072 : last + (size_t)(g - 9 * F) * 3072;
}
static int aes_key_nglwe(const AesDirDesc &d) { return d.nmult * 32 * 9 + 32; }

// Transciphering key of direction `dir` (host_common.h kAesDirs): the first-round LUTs encrypted, one Rng stream per LUT; the
// middle and last rounds as trivial GLWE (zero mask, the table in the body), as src/data_struct.rs:140-151,258-263 writes them.
static int aes_key_generate(AesDir dir, const char *fn, const cbs_keyset *ks, const uint8_t aes_key[16], const RngSource &src,
                            uint64_t *first, uint64_t *mid, uint64_t *last)
{
    if (!ks || ks->glwe_sk.empty() || !aes_key || !first || !mid || !last) {
        set_error(std::string(fn) + ": needs a keyset with the GLWE secret key");
        return CBS_ERR_ARG;
    }
    const AesDirDesc &d = kAesDirs[dir];
    uint8_t tab[10][16][256];
    aes_key_tables(dir, aes_key, tab);
    const uint64_t *S = ks->glwe_sk.data();
    const int F = d.nmult * 16 * 2;
    parallel_for(F, [&](int id) {
        Rng rng(src, d.seed_base + (uint64_t)id);
        std::vector<uint64_t> pt(1024);
        aes_key_lut_plaintext(d, tab, id, pt.data());
        glwe_encrypt(first + (size_t)id * 3072, pt.data(), S, 2, 1024, kStdGlwe, rng);
    });
    memset(mid, 0, sizeof(uint64_t) * d.mid_words);
    memset(last, 0, sizeof(uint64_t) * d.last_words);
    for (int g = F; g < aes_key_nglwe(d); g++) aes_key_lut_plaintext(d, tab, g, aes_key_glwe(d, g, first, mid, last) + 2048);
    return CBS_OK;
}

// Seeded keys (include/cbs_b200.h): every LUT of the direction encrypted, its mask the public ChaCha20 stream of the mask seed
// (chacha20.h), its noise from the secret stream seeded_noise_base + g of `src`.  The mask seed is `mask_seed` as given.
static int aes_key_seeded_generate(AesDir dir, const char *fn, const cbs_keyset *ks, const uint8_t aes_key[16], const RngSource &src,
                                   const uint8_t mask_seed[32], uint64_t *bodies)
{
    const AesDirDesc &d = kAesDirs[dir];
    uint8_t tab[10][16][256];
    aes_key_tables(dir, aes_key, tab);
    uint32_t key[8];
    memcpy(key, mask_seed, 32);
    const uint64_t *S = ks->glwe_sk.data();
    parallel_for(aes_key_nglwe(d), [&](int g) {
        Rng rng(src, d.seeded_noise_base + (uint64_t)g);
        std::vector<uint64_t> pt(1024), ct(3072);
        aes_key_lut_plaintext(d, tab, g, pt.data());
        for (int blk = 0; blk < cbs_chacha::kMaskBlocksPerGlwe; blk++) cbs_chacha::mask_block(key, dir, g, blk, ct.data() + 8 * blk);
        glwe_encrypt(ct.data(), pt.data(), S, 2, 1024, kStdGlwe, rng, true);
        memcpy(bodies + (size_t)g * 1024, ct.data() + 2048, 1024 * 8);
    });
    return CBS_OK;
}

static bool seeded_args_ok(const char *fn, const cbs_keyset *ks, const uint8_t *aes_key, const uint8_t *mask_seed_out,
                           const uint64_t *bodies)
{
    if (!ks || ks->glwe_sk.empty() || !aes_key || !mask_seed_out || !bodies) {
        set_error(std::string(fn) + ": needs a keyset with the GLWE secret key and non-null buffers");
        return false;
    }
    return true;
}

// test variant: noise and mask seed both from the deterministic generator of `seed`, the seed on its own stream
static int aes_key_seeded_generate_seed(AesDir dir, const char *fn, const cbs_keyset *ks, const uint8_t aes_key[16], uint64_t seed,
                                        uint8_t mask_seed_out[32], uint64_t *bodies)
{
    if (!seeded_args_ok(fn, ks, aes_key, mask_seed_out, bodies)) return CBS_ERR_ARG;
    const RngSource src(seed);
    Rng rng(src, kMaskSeedStream);
    for (int i = 0; i < 4; i++) {
        const uint64_t w = rng.next();
        memcpy(mask_seed_out + 8 * i, &w, 8);
    }
    return aes_key_seeded_generate(dir, fn, ks, aes_key, src, mask_seed_out, bodies);
}

// the noise key and the mask seed from two separate getrandom(2) draws
static int aes_key_seeded_generate_os_entropy(AesDir dir, const char *fn, const cbs_keyset *ks, const uint8_t aes_key[16],
                                              uint8_t mask_seed_out[32], uint64_t *bodies)
{
    if (!seeded_args_ok(fn, ks, aes_key, mask_seed_out, bodies)) return CBS_ERR_ARG;
    RngSource src(0);
    if (!RngSource::os_entropy(src) || !os_random(mask_seed_out, 32)) {
        set_error("getrandom failed");
        return CBS_ERR_IO;
    }
    return aes_key_seeded_generate(dir, fn, ks, aes_key, src, mask_seed_out, bodies);
}

// host restatement of k_expand_lut_masks: the seeded key as the direction's three AllRdKeys arrays
static int aes_key_seeded_expand(AesDir dir, const char *fn, const uint8_t mask_seed[32], const uint64_t *bodies, uint64_t *first,
                                 uint64_t *mid, uint64_t *last)
{
    if (!mask_seed || !bodies || !first || !mid || !last) {
        set_error(std::string(fn) + ": null argument");
        return CBS_ERR_ARG;
    }
    const AesDirDesc &d = kAesDirs[dir];
    uint32_t key[8];
    memcpy(key, mask_seed, 32);
    parallel_for(aes_key_nglwe(d), [&](int g) {
        uint64_t *ct = aes_key_glwe(d, g, first, mid, last);
        for (int blk = 0; blk < cbs_chacha::kMaskBlocksPerGlwe; blk++) cbs_chacha::mask_block(key, dir, g, blk, ct + 8 * blk);
        memcpy(ct + 2048, bodies + (size_t)g * 1024, 1024 * 8);
    });
    return CBS_OK;
}

// "CBSSEED1", u64 direction, the 32-byte mask seed, u64 body word count, the bodies
static const char kSeededMagic[8] = {'C', 'B', 'S', 'S', 'E', 'E', 'D', '1'};

static int aes_key_seeded_save(AesDir dir, const char *fn, const char *path, const uint8_t mask_seed[32], const uint64_t *bodies)
{
    if (!path || !mask_seed || !bodies) {
        set_error(std::string(fn) + ": null argument");
        return CBS_ERR_ARG;
    }
    const uint64_t words = (uint64_t)aes_key_nglwe(kAesDirs[dir]) * 1024;
    Writer w;
    w.buf.reserve(56 + 8 * words);
    w.buf.insert(w.buf.end(), kSeededMagic, kSeededMagic + 8);
    w.u64((uint64_t)dir);
    w.buf.insert(w.buf.end(), mask_seed, mask_seed + 32);
    w.vec(bodies, words);
    std::string p(path);
    size_t slash = p.find_last_of('/');
    if (slash != std::string::npos) mkdirs(p.substr(0, slash));
    if (!w.save(p)) {
        set_error("cannot write " + p);
        return CBS_ERR_IO;
    }
    return CBS_OK;
}

static int aes_key_seeded_load(AesDir dir, const char *path, uint8_t mask_seed[32], uint64_t *bodies)
{
    Reader r;
    if (!path || !mask_seed || !bodies || !r.load(path)) {
        set_error(std::string("cannot read ") + (path ? path : "(null)"));
        return CBS_ERR_IO;
    }
    const uint64_t words = (uint64_t)aes_key_nglwe(kAesDirs[dir]) * 1024;
    bool ok = r.buf.size() == 56 + 8 * words && memcmp(r.buf.data(), kSeededMagic, 8) == 0;
    if (ok) {
        r.off = 8;
        ok = r.u64() == (uint64_t)dir;
        r.off = 48;
        ok = ok && r.u64() == words;
    }
    if (!ok) {
        set_error(std::string(path) + (dir == kAesInv ? ": not a seeded inverse (ECB) transciphering key"
                                                      : ": not a seeded forward (CTR) transciphering key"));
        return CBS_ERR_FORMAT;
    }
    memcpy(mask_seed, r.buf.data() + 16, 32);
    memcpy(bodies, r.buf.data() + 56, 8 * words);
    return CBS_OK;
}

static int aes_key_generate_os_entropy(AesDir dir, const char *fn, const cbs_keyset *ks, const uint8_t aes_key[16],
                                       uint64_t *first, uint64_t *mid, uint64_t *last)
{
    RngSource src(0);
    if (!RngSource::os_entropy(src)) {
        set_error("getrandom failed");
        return CBS_ERR_IO;
    }
    return aes_key_generate(dir, fn, ks, aes_key, src, first, mid, last);
}

// The AllRdKeys bincode shape for `nmult` multiples: [nmult] x GlweCiphertextList of the 16 first-round LUT pairs, then
// Vec of 8 rounds x [nmult] x Vec of 16 [GlweCiphertext; 2], then Vec of 16 [GlweCiphertext; 2].  shape(v) writes or checks
// one word of the layout, data(p, n) moves the n key words at p (with their length prefix).
template <typename P, typename Shape, typename Data>
static void all_rd_keys_walk(int nmult, P first, P mid, P last, Shape shape, Data data)
{
    auto modulus = [&]() {  // CiphertextModulus<u64> native: u128 0, then scalar bits 64
        shape(0);
        shape(0);
        shape(64);
    };
    for (int m = 0; m < nmult; m++) {
        shape(16);
        for (int b = 0; b < 16; b++) {  // GlweCiphertextList { data, glwe_size, poly, modulus }
            data(first + ((size_t)m * 16 + b) * 2 * 3072, 2 * 3072);
            shape(3);
            shape(1024);
            modulus();
        }
    }
    auto pairs = [&](P base) {
        shape(16);
        for (int b = 0; b < 16; b++) {
            shape(2);
            for (int a = 0; a < 2; a++) {  // GlweCiphertext { data, poly, modulus }
                data(base + ((size_t)b * 2 + a) * 3072, 3072);
                shape(1024);
                modulus();
            }
        }
    };
    shape(8);
    for (int rd = 0; rd < 8; rd++)
        for (int m = 0; m < nmult; m++) pairs(mid + ((size_t)rd * nmult + m) * 16 * 2 * 3072);
    pairs(last);
}

static int aes_key_load(AesDir dir, const char *not_what, const char *path, uint64_t *first, uint64_t *mid, uint64_t *last)
{
    Reader r;
    if (!path || !r.load(path)) {
        set_error(std::string("cannot read ") + (path ? path : "(null)"));
        return CBS_ERR_IO;
    }
    all_rd_keys_walk(kAesDirs[dir].nmult, first, mid, last, [&](uint64_t v) { r.expect(v); },
                     [&](uint64_t *p, uint64_t n) { r.vec_into(p, n); });
    if (!r.done()) {
        set_error(std::string(path) + ": " + not_what);
        return CBS_ERR_FORMAT;
    }
    return CBS_OK;
}

static int aes_key_save(AesDir dir, const char *path, const uint64_t *first, const uint64_t *mid, const uint64_t *last)
{
    if (!path) return CBS_ERR_ARG;
    const AesDirDesc &d = kAesDirs[dir];
    Writer w;
    w.buf.reserve(((size_t)d.first_words + d.mid_words + d.last_words) * 8 + 65536);
    all_rd_keys_walk(d.nmult, first, mid, last, [&](uint64_t v) { w.u64(v); }, [&](const uint64_t *p, uint64_t n) { w.vec(p, n); });
    std::string p(path);
    size_t slash = p.find_last_of('/');
    if (slash != std::string::npos) mkdirs(p.substr(0, slash));
    if (!w.save(p)) {
        set_error("cannot write " + p);
        return CBS_ERR_IO;
    }
    return CBS_OK;
}

extern "C" {

const char *cbs_last_error(void) { return g_last_error.c_str(); }
const char *cbs_version(void) { return "cbs_b200 0.1 (sm_100a)"; }
void cbs_free(void *p) { free(p); }

void cbs_keyset_free(cbs_keyset *ks) { delete ks; }
const uint64_t *cbs_keyset_bsk(const cbs_keyset *ks) { return ks->bsk.data(); }
const uint64_t *cbs_keyset_ksk(const cbs_keyset *ks) { return ks->ksk.data(); }
const uint64_t *cbs_keyset_auto(const cbs_keyset *ks) { return ks->autok.data(); }
const uint64_t *cbs_keyset_ss(const cbs_keyset *ks) { return ks->ss.data(); }
const uint64_t *cbs_keyset_lwe_sk_small(const cbs_keyset *ks) { return ks->lwe_sk_small.empty() ? nullptr : ks->lwe_sk_small.data(); }
const uint64_t *cbs_keyset_glwe_sk(const cbs_keyset *ks) { return ks->glwe_sk.empty() ? nullptr : ks->glwe_sk.data(); }

int cbs_keyset_from_arrays(const uint64_t *bsk, const uint64_t *ksk, const uint64_t *auto_std, const uint64_t *ss,
                           const uint64_t *lwe_sk_small, const uint64_t *glwe_sk, cbs_keyset **out)
{
    if (!bsk || !ksk || !auto_std || !ss || !out) {
        set_error("cbs_keyset_from_arrays: null argument");
        return CBS_ERR_ARG;
    }
    auto *k = new cbs_keyset;
    k->bsk.assign(bsk, bsk + CBS_BSK_WORDS);
    k->ksk.assign(ksk, ksk + CBS_KSK_WORDS);
    k->autok.assign(auto_std, auto_std + CBS_AUTO_WORDS);
    k->ss.assign(ss, ss + CBS_SS_WORDS);
    if (lwe_sk_small) k->lwe_sk_small.assign(lwe_sk_small, lwe_sk_small + 768);
    if (glwe_sk) k->glwe_sk.assign(glwe_sk, glwe_sk + 2048);
    *out = k;
    return CBS_OK;
}

int cbs_keyset_load_dir(const char *io_dir, int with_secret, cbs_keyset **out)
{
    if (!io_dir || !out) {
        set_error("cbs_keyset_load_dir: null argument");
        return CBS_ERR_ARG;
    }
    const std::string pk = std::string(io_dir) + "/public_keys/";
    auto k = std::unique_ptr<cbs_keyset>(new cbs_keyset);
    {
        Reader r;
        if (!r.load(pk + "bsk.bin")) {
            set_error("cannot read " + pk + "bsk.bin");
            return CBS_ERR_IO;
        }
        r.vec(k->bsk, CBS_BSK_WORDS);
        r.expect(3);
        r.expect(1024);
        r.expect(23);
        r.expect(1);
        r.modulus();
        if (!r.done()) {
            set_error("bsk.bin: not an AES_TIGHT LweBootstrapKey<u64>");
            return CBS_ERR_FORMAT;
        }
    }
    {
        Reader r;
        if (!r.load(pk + "ksk.bin")) {
            set_error("cannot read " + pk + "ksk.bin");
            return CBS_ERR_IO;
        }
        r.vec(k->ksk, CBS_KSK_WORDS);
        r.expect(8);
        r.expect(3);
        r.expect(256);
        r.expect(4);
        r.expect(3);
        r.modulus();
        if (!r.done()) {
            set_error("ksk.bin: not an AES_TIGHT GlweKeyswitchKey<u64>");
            return CBS_ERR_FORMAT;
        }
    }
    {
        Reader r;
        if (!r.load(pk + "ss_key.bin")) {
            set_error("cannot read " + pk + "ss_key.bin");
            return CBS_ERR_IO;
        }
        r.vec(k->ss, CBS_SS_WORDS);
        r.expect(3);
        r.expect(1024);
        r.expect(17);
        r.expect(2);
        r.modulus();
        if (!r.done()) {
            set_error("ss_key.bin: not an AES_TIGHT GgswCiphertextList<u64>");
            return CBS_ERR_FORMAT;
        }
    }
    {
        Reader r;
        if (!r.load(pk + "auto_keys.bin")) {
            set_error("cannot read " + pk + "auto_keys.bin");
            return CBS_ERR_IO;
        }
        k->autok.assign(CBS_AUTO_WORDS, 0);
        if (r.u64() != 10) {
            set_error("auto_keys.bin: expected 10 automorphism keys");
            return CBS_ERR_FORMAT;
        }
        int seen = 0;
        std::vector<uint64_t> data, lo(1024), hi(1024);
        for (int e = 0; e < 10; e++) {
            uint64_t kappa = r.u64();
            int idx = -1;
            for (int i = 0; i < 10; i++)
                if (kappa == (uint64_t)((1024 >> i) + 1)) idx = i;
            if (idx < 0 || !r.vec(data, 36864)) {
                set_error("auto_keys.bin: malformed entry");
                return CBS_ERR_FORMAT;
            }
            r.expect(13);
            r.expect(3);
            r.expect(2);
            r.expect(1024);
            r.expect(kappa);
            // [in 2][split 2][level 3][poly 3][512 c64] -> std [in 2][level 3][poly 3][1024]
            const double *f = reinterpret_cast<const double *>(data.data());
            for (int in = 0; in < 2; in++)
                for (int p = 0; p < 9; p++) {
                    double e0 = fourier_to_limb(f + ((size_t)(in * 2 + 0) * 9 + p) * 1024, lo.data(), 0x1p41);
                    double e1 = fourier_to_limb(f + ((size_t)(in * 2 + 1) * 9 + p) * 1024, hi.data(), 0x1p23);
                    if (e0 > 0.05 || e1 > 1e-4) {
                        set_error("auto_keys.bin: Fourier data is not in natural DFT order "
                                  "(limbs do not invert to integers)");
                        return CBS_ERR_FORMAT;
                    }
                    uint64_t *dst = k->autok.data() + ((size_t)idx * 18 + in * 9 + p) * 1024;
                    for (int j = 0; j < 1024; j++) dst[j] = lo[j] | (hi[j] << 41);
                }
            seen |= 1 << idx;
        }
        if (!r.done() || seen != 1023) {
            set_error("auto_keys.bin: unexpected contents");
            return CBS_ERR_FORMAT;
        }
    }
    if (with_secret) {
        const std::string sk = std::string(io_dir) + "/secret_keys/";
        Reader r;
        if (!r.load(sk + "glwe_sk.bin") || !r.vec(k->glwe_sk, 2048)) {
            set_error("cannot read " + sk + "glwe_sk.bin");
            return CBS_ERR_IO;
        }
        Reader r2;  // optional: the small key is not written by the reference
        if (r2.load(sk + "lwe_sk_small.bin")) r2.vec(k->lwe_sk_small, 768);
    }
    *out = k.release();
    return CBS_OK;
}

int cbs_keyset_save_dir(const cbs_keyset *ks, const char *io_dir, int with_secret)
{
    if (!ks || !io_dir) {
        set_error("cbs_keyset_save_dir: null argument");
        return CBS_ERR_ARG;
    }
    const std::string pk = std::string(io_dir) + "/public_keys/";
    mkdirs(pk);
    bool ok = true;
    {
        Writer w;
        w.vec(ks->bsk.data(), CBS_BSK_WORDS);
        w.u64(3);
        w.u64(1024);
        w.u64(23);
        w.u64(1);
        w.modulus();
        ok &= w.save(pk + "bsk.bin");
    }
    {
        Writer w;
        w.vec(ks->ksk.data(), CBS_KSK_WORDS);
        w.u64(8);
        w.u64(3);
        w.u64(256);
        w.u64(4);
        w.u64(3);
        w.modulus();
        ok &= w.save(pk + "ksk.bin");
    }
    {
        Writer w;
        w.vec(ks->ss.data(), CBS_SS_WORDS);
        w.u64(3);
        w.u64(1024);
        w.u64(17);
        w.u64(2);
        w.modulus();
        ok &= w.save(pk + "ss_key.bin");
    }
    {
        Writer w;
        w.u64(10);
        std::vector<uint64_t> data(36864), limb(1024);
        for (int idx = 0; idx < 10; idx++) {
            uint64_t kappa = (uint64_t)((1024 >> idx) + 1);
            double *f = reinterpret_cast<double *>(data.data());
            for (int in = 0; in < 2; in++)
                for (int sp = 0; sp < 2; sp++)
                    for (int p = 0; p < 9; p++) {
                        const uint64_t *src = ks->autok.data() + ((size_t)idx * 18 + in * 9 + p) * 1024;
                        for (int j = 0; j < 1024; j++) limb[j] = sp ? (src[j] >> 41) : ((src[j] << 23) >> 23);
                        limb_to_fourier(limb.data(), f + ((size_t)(in * 2 + sp) * 9 + p) * 1024);
                    }
            w.u64(kappa);
            w.vec(data.data(), 36864);
            w.u64(13);
            w.u64(3);
            w.u64(2);
            w.u64(1024);
            w.u64(kappa);
        }
        ok &= w.save(pk + "auto_keys.bin");
    }
    if (with_secret && !ks->glwe_sk.empty()) {
        const std::string sk = std::string(io_dir) + "/secret_keys/";
        mkdirs(sk);
        Writer a, b, c;
        a.vec(ks->glwe_sk.data(), 2048);  // LweSecretKey (big) == flattened GlweSecretKey
        ok &= a.save(sk + "lwe_sk.bin");
        b.vec(ks->glwe_sk.data(), 2048);
        b.u64(1024);
        ok &= b.save(sk + "glwe_sk.bin");
        if (!ks->lwe_sk_small.empty()) {
            c.vec(ks->lwe_sk_small.data(), 768);
            ok &= c.save(sk + "lwe_sk_small.bin");
        }
    }
    if (!ok) {
        set_error(std::string("cannot write key files under ") + io_dir);
        return CBS_ERR_IO;
    }
    return CBS_OK;
}

static int keyset_generate_impl(const RngSource &src, cbs_keyset **out)
{
    if (!out) return CBS_ERR_ARG;
    auto *k = new cbs_keyset;
    k->bsk.assign(CBS_BSK_WORDS, 0);
    k->ksk.assign(CBS_KSK_WORDS, 0);
    k->autok.assign(CBS_AUTO_WORDS, 0);
    k->ss.assign(CBS_SS_WORDS, 0);
    k->lwe_sk_small.resize(768);
    k->glwe_sk.resize(2048);
    Rng srng(src, 0);
    for (auto &b : k->lwe_sk_small) b = srng.next() >> 63;
    for (auto &b : k->glwe_sk) b = srng.next() >> 63;
    const uint64_t *S = k->glwe_sk.data();

    // bootstrap key: GGSW(s_i) under glwe_sk, B = 2^23, l = 1 (keygen.rs:213-221)
    parallel_for(768, [&](int i) {
        Rng rng(src, 1000 + (uint64_t)i);
        const uint64_t m = k->lwe_sk_small[i];
        std::vector<uint64_t> pt(1024);
        for (int row = 0; row < 3; row++) {
            std::fill(pt.begin(), pt.end(), 0ull);
            if (m) {
                if (row < 2)
                    for (int j = 0; j < 1024; j++) pt[j] = (0ull - S[row * 1024 + j]) << 41;  // -s_i * S_row * 2^(64-23)
                else
                    pt[0] = 1ull << 41;
            }
            glwe_encrypt(k->bsk.data() + ((size_t)i * 3 + row) * 3072, pt.data(), S, 2, 1024, kStdGlwe, rng);
        }
    });

    // LWE keyswitch key over the common ring N' = 256: big key (8 polys) -> small key (3 polys),
    // GLEV of -S_in,i, B = 2^4, l = 3, LWE noise (keygen.rs:224-240, glwe_keyswitch.rs:183-218)
    {
        std::vector<uint64_t> pt(256);
        for (int i = 0; i < 8; i++)
            for (int lev = 0; lev < 3; lev++) {
                Rng rng(src, 5000 + (uint64_t)(i * 3 + lev));
                const int log_scale = 64 - 4 * (lev + 1);
                for (int j = 0; j < 256; j++) pt[j] = (0ull - S[i * 256 + j]) << log_scale;
                glwe_encrypt(k->ksk.data() + ((size_t)i * 3 + lev) * 4 * 256, pt.data(), k->lwe_sk_small.data(), 3, 256,
                             kStdLwe, rng);
            }
    }

    // automorphism keys: keyswitch from S(X^kappa) back to S, B = 2^13, l = 3 (automorphism.rs:59-178)
    parallel_for(10, [&](int idx) {
        const unsigned kappa = (unsigned)((1024 >> idx) + 1);
        std::vector<uint64_t> before(1024), pt(1024);
        for (int i = 0; i < 2; i++) {
            eval_x_k(before.data(), S + i * 1024, 1024, kappa);
            for (int lev = 0; lev < 3; lev++) {
                Rng rng(src, 6000 + (uint64_t)((idx * 2 + i) * 3 + lev));
                const int log_scale = 64 - 13 * (lev + 1);
                for (int j = 0; j < 1024; j++) pt[j] = (0ull - before[j]) << log_scale;
                glwe_encrypt(k->autok.data() + (((size_t)idx * 2 + i) * 3 + lev) * 3072, pt.data(), S, 2, 1024, kStdGlwe,
                             rng);
            }
        }
    });

    // scheme-switching key: GGSW(0) then -S_i * 2^(64-17*lev) added to mask poly `col` (col < 2) or to
    // the body (col == 2) of row (lev, col)  (ggsw_conv.rs:41-74)
    for (int i = 0; i < 2; i++)
        for (int lev = 0; lev < 2; lev++)
            for (int col = 0; col < 3; col++) {
                Rng rng(src, 7000 + (uint64_t)((i * 2 + lev) * 3 + col));
                uint64_t *ct = k->ss.data() + (((size_t)i * 2 + lev) * 3 + col) * 3072;
                glwe_encrypt(ct, nullptr, S, 2, 1024, kStdGlwe, rng);
                const int log_scale = 64 - 17 * (lev + 1);
                uint64_t *dst = ct + (size_t)col * 1024;
                for (int j = 0; j < 1024; j++) dst[j] += (0ull - S[i * 1024 + j]) << log_scale;
            }
    *out = k;
    return CBS_OK;
}

int cbs_keyset_generate(uint64_t seed, cbs_keyset **out) { return keyset_generate_impl(RngSource(seed), out); }

int cbs_keyset_generate_os_entropy(cbs_keyset **out)
{
    RngSource src(0);
    if (!RngSource::os_entropy(src)) {
        set_error("getrandom failed");
        return CBS_ERR_IO;
    }
    return keyset_generate_impl(src, out);
}

int cbs_trans_key_generate(const cbs_keyset *ks, const uint8_t aes_key[16], uint64_t seed, uint64_t *k10_9,
                           uint64_t *k8_1, uint64_t *k0)
{
    return aes_key_generate(kAesInv, "cbs_trans_key_generate", ks, aes_key, RngSource(seed), k10_9, k8_1, k0);
}

int cbs_trans_key_generate_os_entropy(const cbs_keyset *ks, const uint8_t aes_key[16], uint64_t *k10_9, uint64_t *k8_1,
                                      uint64_t *k0)
{
    return aes_key_generate_os_entropy(kAesInv, "cbs_trans_key_generate", ks, aes_key, k10_9, k8_1, k0);
}

int cbs_trans_key_load(const char *path, uint64_t *k10_9, uint64_t *k8_1, uint64_t *k0)
{
    return aes_key_load(kAesInv, "not an AllRdKeys file for AES_TIGHT", path, k10_9, k8_1, k0);
}

int cbs_trans_key_save(const char *path, const uint64_t *k10_9, const uint64_t *k8_1, const uint64_t *k0)
{
    return aes_key_save(kAesInv, path, k10_9, k8_1, k0);
}

// Forward keys use the AllRdKeys bincode shape with 3-tuples (x1, x2, x3) and 8 middle rounds.
int cbs_fwd_trans_key_generate(const cbs_keyset *ks, const uint8_t aes_key[16], uint64_t seed, uint64_t *kf_first,
                               uint64_t *kf_mid, uint64_t *kf_last)
{
    return aes_key_generate(kAesFwd, "cbs_fwd_trans_key_generate", ks, aes_key, RngSource(seed), kf_first, kf_mid, kf_last);
}

int cbs_fwd_trans_key_generate_os_entropy(const cbs_keyset *ks, const uint8_t aes_key[16], uint64_t *kf_first, uint64_t *kf_mid,
                                          uint64_t *kf_last)
{
    return aes_key_generate_os_entropy(kAesFwd, "cbs_fwd_trans_key_generate", ks, aes_key, kf_first, kf_mid, kf_last);
}

int cbs_fwd_trans_key_save(const char *path, const uint64_t *kf_first, const uint64_t *kf_mid, const uint64_t *kf_last)
{
    return aes_key_save(kAesFwd, path, kf_first, kf_mid, kf_last);
}

int cbs_fwd_trans_key_load(const char *path, uint64_t *kf_first, uint64_t *kf_mid, uint64_t *kf_last)
{
    return aes_key_load(kAesFwd, "not a forward (CTR) transciphering key for AES_TIGHT", path, kf_first, kf_mid, kf_last);
}

int cbs_trans_key_seeded_generate(const cbs_keyset *ks, const uint8_t aes_key[16], uint64_t seed, uint8_t mask_seed_out[32],
                                  uint64_t *bodies)
{
    return aes_key_seeded_generate_seed(kAesInv, "cbs_trans_key_seeded_generate", ks, aes_key, seed, mask_seed_out, bodies);
}

int cbs_trans_key_seeded_generate_os_entropy(const cbs_keyset *ks, const uint8_t aes_key[16], uint8_t mask_seed_out[32],
                                             uint64_t *bodies)
{
    return aes_key_seeded_generate_os_entropy(kAesInv, "cbs_trans_key_seeded_generate", ks, aes_key, mask_seed_out, bodies);
}

int cbs_fwd_trans_key_seeded_generate(const cbs_keyset *ks, const uint8_t aes_key[16], uint64_t seed, uint8_t mask_seed_out[32],
                                      uint64_t *bodies)
{
    return aes_key_seeded_generate_seed(kAesFwd, "cbs_fwd_trans_key_seeded_generate", ks, aes_key, seed, mask_seed_out, bodies);
}

int cbs_fwd_trans_key_seeded_generate_os_entropy(const cbs_keyset *ks, const uint8_t aes_key[16], uint8_t mask_seed_out[32],
                                                 uint64_t *bodies)
{
    return aes_key_seeded_generate_os_entropy(kAesFwd, "cbs_fwd_trans_key_seeded_generate", ks, aes_key, mask_seed_out, bodies);
}

int cbs_trans_key_seeded_expand(const uint8_t mask_seed[32], const uint64_t *bodies, uint64_t *k10_9, uint64_t *k8_1, uint64_t *k0)
{
    return aes_key_seeded_expand(kAesInv, "cbs_trans_key_seeded_expand", mask_seed, bodies, k10_9, k8_1, k0);
}

int cbs_fwd_trans_key_seeded_expand(const uint8_t mask_seed[32], const uint64_t *bodies, uint64_t *kf_first, uint64_t *kf_mid,
                                    uint64_t *kf_last)
{
    return aes_key_seeded_expand(kAesFwd, "cbs_fwd_trans_key_seeded_expand", mask_seed, bodies, kf_first, kf_mid, kf_last);
}

int cbs_trans_key_seeded_save(const char *path, const uint8_t mask_seed[32], const uint64_t *bodies)
{
    return aes_key_seeded_save(kAesInv, "cbs_trans_key_seeded_save", path, mask_seed, bodies);
}

int cbs_trans_key_seeded_load(const char *path, uint8_t mask_seed[32], uint64_t *bodies)
{
    return aes_key_seeded_load(kAesInv, path, mask_seed, bodies);
}

int cbs_fwd_trans_key_seeded_save(const char *path, const uint8_t mask_seed[32], const uint64_t *bodies)
{
    return aes_key_seeded_save(kAesFwd, "cbs_fwd_trans_key_seeded_save", path, mask_seed, bodies);
}

int cbs_fwd_trans_key_seeded_load(const char *path, uint8_t mask_seed[32], uint64_t *bodies)
{
    return aes_key_seeded_load(kAesFwd, path, mask_seed, bodies);
}

int cbs_lwe_list_load(const char *path, uint64_t **data, uint64_t *count, uint64_t *lwe_words)
{
    Reader r;
    if (!path || !data || !count || !lwe_words || !r.load(path)) {
        set_error(std::string("cannot read ") + (path ? path : "(null)"));
        return CBS_ERR_IO;
    }
    uint64_t n = r.u64();
    // n comes from the file: bound it by the bytes actually present before any multiplication can wrap
    if (!r.ok || r.buf.size() < r.off + 32 || n != (r.buf.size() - r.off - 32) / 8 || (r.buf.size() - r.off - 32) % 8) {
        set_error(std::string(path) + ": not an LweCiphertextList<u64>");
        return CBS_ERR_FORMAT;
    }
    uint64_t *p = (uint64_t *)malloc(8 * (n ? n : 1));
    memcpy(p, r.buf.data() + r.off, 8 * n);
    r.off += 8 * n;
    uint64_t lw = r.u64();
    r.modulus();
    if (!r.done() || lw == 0 || n % lw) {
        free(p);
        set_error(std::string(path) + ": malformed LweCiphertextList trailer");
        return CBS_ERR_FORMAT;
    }
    *data = p;
    *count = n / lw;
    *lwe_words = lw;
    return CBS_OK;
}

int cbs_lwe_list_save(const char *path, const uint64_t *data, uint64_t count, uint64_t lwe_words)
{
    if (!path || (!data && count)) return CBS_ERR_ARG;
    Writer w;
    w.vec(data, count * lwe_words);
    w.u64(lwe_words);
    w.modulus();
    std::string p(path);
    size_t slash = p.find_last_of('/');
    if (slash != std::string::npos) mkdirs(p.substr(0, slash));
    if (!w.save(p)) {
        set_error("cannot write " + p);
        return CBS_ERR_IO;
    }
    return CBS_OK;
}

// decrypt_decode_lwe_list / decrypt, submission/src/help_fun.rs:12-42 (delta = 2^63)
int cbs_lwe_decrypt_bits(const uint64_t *sk, int n, const uint64_t *lwe, uint64_t count, uint64_t *bits_out)
{
    if (!sk || !lwe || !bits_out || n <= 0) return CBS_ERR_ARG;
    const uint64_t delta = 1ull << 63;
    for (uint64_t c = 0; c < count; c++) {
        const uint64_t *ct = lwe + c * (uint64_t)(n + 1);
        uint64_t phase = ct[n];
        for (int i = 0; i < n; i++)
            if (sk[i]) phase -= ct[i];
        const uint64_t rounding = (phase & (delta >> 1)) << 1;
        bits_out[c] = (phase + rounding) / delta;
    }
    return CBS_OK;
}

// The GLWE twin of cbs_lwe_decrypt_bits: coefficient j of GLWE g is bit g * 1024 + j.
// phase[j] = body[j] - sum_c sum_k s_c[k] m_c[j - k], negated where j - k wraps (X^1024 = -1); only the non-zero key
// words take part, so a binary key costs about 1024 additions per bit.
int cbs_glwe_decrypt_bits(const uint64_t *glwe_sk, const uint64_t *glwe, uint64_t nglwe, uint64_t nbits, uint64_t *bits_out)
{
    if (!glwe_sk || !glwe || !bits_out || nbits > nglwe * 1024) return CBS_ERR_ARG;
    std::vector<int> nz[2];
    for (int c = 0; c < 2; c++)
        for (int k = 0; k < 1024; k++)
            if (glwe_sk[c * 1024 + k]) nz[c].push_back(k);
    const uint64_t delta = 1ull << 63;
    for (uint64_t b = 0; b < nbits; b++) {
        const uint64_t *g = glwe + (b / 1024) * 3072;
        const int j = (int)(b % 1024);
        uint64_t phase = g[2048 + j];
        for (int c = 0; c < 2; c++)
            for (int k : nz[c]) {
                const uint64_t m = j >= k ? g[c * 1024 + j - k] : 0ull - g[c * 1024 + j - k + 1024];
                phase -= m * glwe_sk[c * 1024 + k];
            }
        const uint64_t rounding = (phase & (delta >> 1)) << 1;
        bits_out[b] = (phase + rounding) / delta;
    }
    return CBS_OK;
}

// GlweCiphertextList<Vec<u64>> {data, glwe_size = 3, polynomial_size = 1024, modulus}: the shape trans_key.bin holds its
// first-round LUTs in (all_rd_keys_walk), here for the output of cbs_pack_lwes
int cbs_glwe_list_save(const char *path, const uint64_t *data, uint64_t nglwe)
{
    if (!path || (!data && nglwe)) return CBS_ERR_ARG;
    Writer w;
    w.vec(data, nglwe * 3072);
    w.u64(3);
    w.u64(1024);
    w.modulus();
    std::string p(path);
    size_t slash = p.find_last_of('/');
    if (slash != std::string::npos) mkdirs(p.substr(0, slash));
    if (!w.save(p)) {
        set_error("cannot write " + p);
        return CBS_ERR_IO;
    }
    return CBS_OK;
}

int cbs_glwe_list_load(const char *path, uint64_t **data, uint64_t *nglwe)
{
    Reader r;
    if (!path || !data || !nglwe || !r.load(path)) {
        set_error(std::string("cannot read ") + (path ? path : "(null)"));
        return CBS_ERR_IO;
    }
    uint64_t n = r.u64();
    // n comes from the file: bound it by the bytes present (40 trailer bytes: sizes and modulus) before using it
    if (!r.ok || r.buf.size() < r.off + 40 || n != (r.buf.size() - r.off - 40) / 8 || (r.buf.size() - r.off - 40) % 8 || n % 3072) {
        set_error(std::string(path) + ": not a GlweCiphertextList<u64> of GLWE(2, 1024)");
        return CBS_ERR_FORMAT;
    }
    uint64_t *p = (uint64_t *)malloc(8 * (n ? n : 1));
    memcpy(p, r.buf.data() + r.off, 8 * n);
    r.off += 8 * n;
    r.expect(3);
    r.expect(1024);
    r.modulus();
    if (!r.done()) {
        free(p);
        set_error(std::string(path) + ": malformed GlweCiphertextList trailer (need glwe_size 3, polynomial_size 1024)");
        return CBS_ERR_FORMAT;
    }
    *data = p;
    *nglwe = n / 3072;
    return CBS_OK;
}

// bincode Vec<u64> (the intermediate/decoded_result*.txt files of the client stages)
int cbs_u64_vec_save(const char *path, const uint64_t *data, uint64_t n)
{
    if (!path || (!data && n)) return CBS_ERR_ARG;
    Writer w;
    w.vec(data, n);
    std::string p(path);
    size_t slash = p.find_last_of('/');
    if (slash != std::string::npos) mkdirs(p.substr(0, slash));
    if (!w.save(p)) {
        set_error("cannot write " + p);
        return CBS_ERR_IO;
    }
    return CBS_OK;
}

int cbs_u64_vec_load(const char *path, uint64_t **data, uint64_t *n)
{
    Reader r;
    if (!path || !data || !n || !r.load(path)) {
        set_error(std::string("cannot read ") + (path ? path : "(null)"));
        return CBS_ERR_IO;
    }
    uint64_t len = r.u64();
    if (!r.ok || r.off + 8 * len != r.buf.size()) {
        set_error(std::string(path) + ": not a bincode Vec<u64>");
        return CBS_ERR_FORMAT;
    }
    uint64_t *p = (uint64_t *)malloc(8 * (len ? len : 1));
    memcpy(p, r.buf.data() + r.off, 8 * len);
    *data = p;
    *n = len;
    return CBS_OK;
}

// dry run of the inner-product circuit plan on cleartext values (test hook of host/ip_plan.h)
int cbs_inner_product_plan_check(const uint16_t *vals, int nvals, uint16_t *result, int64_t *circuit_bootstraps, int *layers,
                                 int64_t *lut_ladders)
{
    if (nvals <= 0 || (nvals & 1) || (!vals && result)) {
        set_error("cbs_inner_product_plan_check: bad argument (need an even number of values)");
        return CBS_ERR_ARG;
    }
    const IpPlan plan = ip_make_plan(nvals);
    if (result) *result = ip_eval_clear(plan, vals);
    if (circuit_bootstraps) *circuit_bootstraps = plan.total_cbs();
    if (layers) *layers = (int)plan.layers.size();
    if (lut_ladders) {
        int64_t n = 0;
        for (const IpLayer &l : plan.layers) n += (int64_t)l.jobs.size();
        *lut_ladders = n;
    }
    return CBS_OK;
}

int cbs_max_plan_check(const uint16_t *vals, int nvals, uint16_t *result, int64_t *circuit_bootstraps, int *layers,
                       int64_t *lut_ladders)
{
    if (nvals <= 0 || (!vals && result)) {
        set_error("cbs_max_plan_check: bad argument");
        return CBS_ERR_ARG;
    }
    const IpPlan plan = max_make_plan(nvals);
    if (result) *result = ip_eval_clear(plan, vals);
    if (circuit_bootstraps) *circuit_bootstraps = plan.total_cbs();
    if (layers) *layers = (int)plan.layers.size();
    if (lut_ladders) {
        int64_t n = 0;
        for (const IpLayer &l : plan.layers) n += (int64_t)l.jobs.size();
        *lut_ladders = n;
    }
    return CBS_OK;
}

static int encrypt_bits(const uint64_t *sk, int n, double std, const uint8_t *bits, int count, uint64_t seed, uint64_t *out)
{
    const RngSource src(seed);
    for (int c = 0; c < count; c++) {
        Rng rng(src, 20000 + (uint64_t)c);
        uint64_t *ct = out + (size_t)c * (n + 1);
        uint64_t b = rng.noise(std) + ((uint64_t)(bits[c] & 1) << 63);
        for (int i = 0; i < n; i++) {
            ct[i] = rng.next();
            if (sk[i]) b += ct[i];
        }
        ct[n] = b;
    }
    return CBS_OK;
}

int cbs_encrypt_bits_big(const cbs_keyset *ks, const uint8_t *bits, int count, uint64_t seed, uint64_t *out)
{
    if (!ks || ks->glwe_sk.empty() || !bits || !out) {
        set_error("cbs_encrypt_bits_big: needs a keyset with secret keys");
        return CBS_ERR_ARG;
    }
    return encrypt_bits(ks->glwe_sk.data(), 2048, kStdGlwe, bits, count, seed, out);
}

int cbs_encrypt_bits_small(const cbs_keyset *ks, const uint8_t *bits, int count, uint64_t seed, uint64_t *out)
{
    if (!ks || ks->lwe_sk_small.empty() || !bits || !out) {
        set_error("cbs_encrypt_bits_small: needs a keyset with secret keys");
        return CBS_ERR_ARG;
    }
    return encrypt_bits(ks->lwe_sk_small.data(), 768, kStdLwe, bits, count, seed, out);
}

}  // extern "C"
