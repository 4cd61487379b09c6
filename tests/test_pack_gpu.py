"""LWE-to-GLWE packing on the GPU (cbs_pack_lwes, cbs_pack_lwes_dev, k_pack_level).

(a) Small keys (tests/test_exact_ref_cpu.py): every FP64 product is an exact integer, so the packed GLWEs must equal the
    exact reference tests/exact_pack_ref.py pack_lwes bit for bit, at counts that cover one slot, a partial group, a full group,
    and one, two and three groups.
(b) The seeded keys: the distance to the exact reference stays within a budget measured on one B200.
(c) Chained behind a device-resident CTR transcipher: the packed bits are the AES-CTR plaintext bits and the bits of the
    unpacked rows, with the rows' noise.
(d) Invariance (host == device, zero padding, group position, 1024 blocks), asynchrony and argument errors."""
import numpy as np
import pytest
import torch

import exact_pack_ref as ex
from conftest import NoiseFailure, glwe_phase, log2max, retry_on_noise, sdiff
from test_exact_ref_cpu import small_keys

pytestmark = pytest.mark.gpu

N = 1024
LWE = 2049


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()


def _host(t, words):
    return t.cpu().numpy().view(np.uint64).reshape(-1, words)


def _glwe_out(count):
    return torch.empty(((count + N - 1) // N, 3 * N), dtype=torch.int64, device="cuda")


@pytest.fixture(scope="module")
def small_ctx(cbs):
    c = cbs.Context(cbs.KeySet.from_arrays(*small_keys()), 0)
    yield c
    c.close()


@pytest.fixture
def sctx(ctx):
    """The session context issuing on a torch stream that is also torch's current stream (ordering without syncs)."""
    s = torch.cuda.Stream()
    ctx.set_stream(s.cuda_stream)
    with torch.cuda.stream(s):
        yield ctx
    ctx.set_stream(None)


# ---- (a) small keys: bit-exact ------------------------------------------------------------------------------------

def test_small_keys_bit_exact(small_ctx):
    """One group G of 1024 random rows whose last row is zero, repeated: count 1023 and 1024 are the same group (the zero
    slot against the skipped one), 1025 and 2055 repeat it and add a group of 1 and 7 rows, so the exact full group (about
    1023 keyswitches on the CPU) is computed once."""
    auto = small_keys()[2]
    rng = np.random.default_rng(61)
    g = rng.integers(0, 2 ** 64, (N, LWE), dtype=np.uint64)
    g[N - 1] = 0
    rows = np.concatenate([g, g, g[:7]])
    full = ex.pack_lwes(auto, g)[0]
    part = {k: ex.pack_lwes(auto, g[:k])[0] for k in (1, 2, 3, 7)}
    want = {1: [part[1]], 2: [part[2]], 3: [part[3]], 1023: [full], 1024: [full], 1025: [full, part[1]],
            2055: [full, full, part[7]]}
    for count, w in want.items():
        got = small_ctx.pack_lwes(rows[:count])
        assert got.shape == (len(w), 3 * N), count
        for i in range(len(w)):
            assert (got[i] == w[i]).all(), (count, i, int(np.flatnonzero(got[i] != w[i])[0]))


# ---- (b) seeded keys: FP64 error budget -----------------------------------------------------------------------------

def test_real_keys_error_budget(ctx, keyset):
    """Word distance and phase distance to the exact tree at 1, 3 and 64 fresh encryptions."""
    bits = np.random.default_rng(62).integers(0, 2, 64).astype(np.uint8)
    lwe = keyset.encrypt_bits_big(bits, 63)
    sk = keyset.glwe_sk
    e_word, e_phase = {}, {}
    for count in (1, 3, 64):
        got = ctx.pack_lwes(lwe[:count])
        want = ex.pack_lwes(keyset.auto_std, lwe[:count])
        e_word[count] = log2max(sdiff(got, want))
        e_phase[count] = log2max(sdiff(glwe_phase(got, sk), glwe_phase(want, sk)))
    print("packing - exact, words:", {k: round(v, 2) for k, v in e_word.items()},
          "phases:", {k: round(v, 2) for k, v in e_phase.items()})
    # measured on one B200 (1000 W, 1965 MHz): words 15.99 / 15.99 / 16.55 (no digit flip along the ten levels, like the
    # 10-step trace's 15.66), phases 17.24 / 18.33 / 18.64 at counts 1 / 3 / 64; the packed bits' own noise is 2^40.5
    # at count 64 (exact tree), so the FP64 error is 2^-22 of it.  Budgets: measured + 1 bit.
    assert max(e_word.values()) < 17.6, e_word
    assert max(e_phase.values()) < 19.7, e_phase


# ---- (c) chained behind the device-resident CTR transcipher ---------------------------------------------------------

def _ctr_dev(ctx, keyset, aes_key, nb, seed):
    """device-resident CTR transcipher of nb random blocks -> (plaintext bytes, d_rows [nb][128][2049])"""
    import aes_clear
    iv = bytes(range(16))
    pt = bytes(np.random.default_rng(seed).integers(0, 256, 16 * nb, dtype=np.uint8))
    ct = aes_clear.ctr_crypt(aes_key, iv, pt)
    counters = b"".join(((int.from_bytes(iv, "big") + b) % (1 << 128)).to_bytes(16, "big") for b in range(nb))
    d_ctr = torch.frombuffer(bytearray(counters), dtype=torch.uint8).cuda()
    d_ct = torch.frombuffer(bytearray(ct), dtype=torch.uint8).cuda()
    d_rows = torch.empty((nb, 128, LWE), dtype=torch.int64, device="cuda")
    ctx.ctr_transcipher_dev(d_ctr.data_ptr(), d_ct.data_ptr(), nb, d_rows.data_ptr())
    return pt, d_rows


def _noise(phase, bits):
    return sdiff(phase, np.asarray(bits, dtype=np.uint64) << np.uint64(63))


def _rows_and_packed(cbs, keyset, rows, packed):
    """(bits of the rows, bits of the packed GLWEs, log2 noise std of both) for the first len(rows) slots"""
    import ref_io
    sk = keyset.glwe_sk
    n = len(rows)
    p_rows = ref_io.lwe_phase(rows, sk)
    b_rows = ref_io.decode_bit(p_rows).astype(np.uint64)
    b_pack = cbs.glwe_decrypt_bits(sk, packed, n)
    p_pack = glwe_phase(packed, sk).reshape(-1)[:n]
    return b_rows, b_pack, np.log2(_noise(p_rows, b_rows).std()), np.log2(_noise(p_pack, b_rows).std())


@pytest.mark.parametrize("nb", [8, 9])
def test_chained_after_ctr_transcipher(sctx, cbs, keyset, aes_key, nb):
    ctx = sctx

    def run(attempt):
        ctx.upload_fwd_trans_key(*keyset.gen_forward_transciphering_keys(aes_key, 70 + attempt))
        pt, d_rows = _ctr_dev(ctx, keyset, aes_key, nb, 71 + nb)
        count = nb * 128
        d_out = _glwe_out(count)
        ctx.pack_lwes_dev(d_rows.data_ptr(), count, d_out.data_ptr())  # no synchronise or download in between
        packed = _host(d_out, 3 * N)
        rows = _host(d_rows, LWE)
        b_rows, b_pack, s_rows, s_pack = _rows_and_packed(cbs, keyset, rows, packed)
        print(f"{nb} blocks: noise std rows 2^{s_rows:.3f}, packed 2^{s_pack:.3f}")
        assert (b_pack == b_rows).all(), np.flatnonzero(b_pack != b_rows)[:16]
        assert abs(s_pack - s_rows) < 0.1, (s_rows, s_pack)
        assert (cbs.glwe_decrypt_bits(keyset.glwe_sk, packed)[count:] == 0).all()
        want = np.unpackbits(np.frombuffer(pt, dtype=np.uint8)).astype(np.uint64)  # MSB first inside each byte
        if (b_rows != want).any():
            raise NoiseFailure(f"transciphered rows differ from the plaintext in blocks "
                               f"{sorted(set((np.flatnonzero(b_rows != want) // 128).tolist()))}")
        assert (b_pack == want).all()

    retry_on_noise(run)


# ---- (d) invariance, asynchrony, arguments ------------------------------------------------------------------------

def test_host_device_padding_and_group_position(sctx, keyset):
    ctx = sctx
    rng = np.random.default_rng(64)
    bits = rng.integers(0, 2, 2 * N + 7).astype(np.uint8)
    lwe = keyset.encrypt_bits_big(bits, 65)
    g, h = lwe[:N], lwe[N:2 * N]
    alone = ctx.pack_lwes(g)
    # host call == device call
    for count in (1, 1025, 2 * N + 7):
        d_in, d_out = _dev(lwe[:count]), _glwe_out(count)
        ctx.pack_lwes_dev(d_in.data_ptr(), count, d_out.data_ptr())
        assert (_host(d_out, 3 * N) == ctx.pack_lwes(lwe[:count])).all(), count
    # 1025 == 2048 with zero rows 1025..: the skipped subtrees equal the computed zero ones
    padded = np.concatenate([lwe[:N + 1], np.zeros((N - 1, LWE), dtype=np.uint64)])
    assert (ctx.pack_lwes(lwe[:N + 1]) == ctx.pack_lwes(padded)).all()
    # one group alone, as group 0 and as group 1
    assert (ctx.pack_lwes(np.concatenate([g, h]))[0] == alone[0]).all()
    assert (ctx.pack_lwes(np.concatenate([h, g, lwe[2 * N:]]))[1] == alone[0]).all()
    from temp_fhe_transciphering_b200 import glwe_decrypt_bits
    assert (glwe_decrypt_bits(keyset.glwe_sk, ctx.pack_lwes(lwe), len(bits)) == bits).all()


def test_1024_blocks_decrypt_like_the_rows(sctx, cbs, keyset, aes_key):
    """BASELINE config 5's size: 1024 CTR blocks, 131,072 rows -> 128 GLWEs, every bit and the noise as the rows."""
    ctx = sctx
    ctx.upload_fwd_trans_key(*keyset.gen_forward_transciphering_keys(aes_key, 81))
    _, d_rows = _ctr_dev(ctx, keyset, aes_key, 1024, 82)
    count = 1024 * 128
    d_out = _glwe_out(count)
    ctx.pack_lwes_dev(d_rows.data_ptr(), count, d_out.data_ptr())
    packed = _host(d_out, 3 * N)
    assert packed.shape == (128, 3 * N)
    b_rows, b_pack, s_rows, s_pack = _rows_and_packed(cbs, keyset, _host(d_rows, LWE), packed)
    print(f"1024 blocks: noise std rows 2^{s_rows:.3f}, packed 2^{s_pack:.3f}")
    assert (b_pack == b_rows).all(), np.flatnonzero(b_pack != b_rows)[:16]
    assert abs(s_pack - s_rows) < 0.1, (s_rows, s_pack)


def test_pack_dev_is_asynchronous(sctx, keyset):
    ctx = sctx
    stream = torch.cuda.current_stream()
    count = 128 * N
    d_in, d_out = _dev(keyset.encrypt_bits_big(np.ones(count, dtype=np.uint8), 66)), _glwe_out(count)
    ctx.pack_lwes_dev(d_in.data_ptr(), count, d_out.data_ptr())  # warm: workspace
    stream.synchronize()
    ctx.pack_lwes_dev(d_in.data_ptr(), count, d_out.data_ptr())
    assert stream.query() is False
    from temp_fhe_transciphering_b200 import glwe_decrypt_bits
    assert (glwe_decrypt_bits(keyset.glwe_sk, _host(d_out, 3 * N)) == 1).all()


def test_pack_argument_errors(sctx, cbs):
    ctx = sctx
    d_in = torch.zeros((2 * N, LWE), dtype=torch.int64, device="cuda")
    d_out = _glwe_out(2 * N)
    p, o = d_in.data_ptr(), d_out.data_ptr()
    calls = [lambda: ctx.pack_lwes_dev(p, 0, o), lambda: ctx.pack_lwes_dev(p, -1, o), lambda: ctx.pack_lwes_dev(0, 4, o),
             lambda: ctx.pack_lwes_dev(p, 4, 0), lambda: ctx.pack_lwes_dev(p, 4, p),
             lambda: ctx.pack_lwes_dev(p, 2 * N, p + (2 * N * LWE - 8) * 8), lambda: ctx.pack_lwes_dev(p + 8, 4, p)]
    for call in calls:
        with pytest.raises(cbs.CbsError, match=r"\(code 1\)"):
            call()
    # an output that ends where the input starts, or starts where it ends, is accepted
    ctx.pack_lwes_dev(p + 3 * N * 8, 4, p)
    ctx.pack_lwes_dev(p, 4, p + 4 * LWE * 8)
    assert ctx.pack_lwes(np.zeros((0, LWE), dtype=np.uint64)).shape == (0, 3 * N)
