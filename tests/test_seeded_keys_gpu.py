"""Seeded transciphering keys on the GPU: cbs_{,fwd_}trans_key_seeded_upload (bodies copied, masks expanded by
k_expand_lut_masks) against the host expansion, end to end in both modes, noise, switching key forms in one context, chaining
into the packing, and argument errors."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import NoiseFailure, retry_on_noise, sdiff

pytestmark = pytest.mark.gpu

LWE = 2049


@pytest.fixture(scope="module")
def sctx(cbs, keyset):
    """A context of its own (the key uploads here leave the session context alone), issuing on a torch stream that is also
    torch's current stream, so tensor copies and the context's work are ordered without synchronising."""
    c = cbs.Context(keyset, 0)
    s = torch.cuda.Stream()
    c.set_stream(s.cuda_stream)
    with torch.cuda.stream(s):
        yield c
    c.set_stream(None)
    c.close()


def _host(t):
    return t.cpu().numpy().view(np.uint64).reshape(-1, LWE)


def _inputs(aes_key, mode, nb, seed):
    """(plaintext, the public inputs of the _dev call as device tensors)"""
    import aes_clear
    pt = bytes(np.random.default_rng(seed).integers(0, 256, 16 * nb, dtype=np.uint8))
    if mode == "ecb":
        return pt, (torch.frombuffer(bytearray(aes_clear.ecb_encrypt(aes_key, pt)), dtype=torch.uint8).cuda(),)
    iv = bytes(range(16))
    counters = b"".join(((int.from_bytes(iv, "big") + b) % (1 << 128)).to_bytes(16, "big") for b in range(nb))
    return pt, (torch.frombuffer(bytearray(counters), dtype=torch.uint8).cuda(),
                torch.frombuffer(bytearray(aes_clear.ctr_crypt(aes_key, iv, pt)), dtype=torch.uint8).cuda())


def _run(ctx, mode, d_in, nb):
    d_out = torch.empty((nb, 128, LWE), dtype=torch.int64, device="cuda")
    if mode == "ecb":
        ctx.transcipher_dev(d_in[0].data_ptr(), nb, d_out.data_ptr())
    else:
        ctx.ctr_transcipher_dev(d_in[0].data_ptr(), d_in[1].data_ptr(), nb, d_out.data_ptr())
    return d_out


def _keys(cbs, keyset, aes_key, mode, seed):
    """seeded key of the mode's direction, its host expansion, and the upload calls of both forms"""
    if mode == "ecb":
        ms, bodies = keyset.gen_seeded_transciphering_keys(aes_key, seed)
        return ms, bodies, cbs.expand_seeded_trans_key(ms, bodies)
    ms, bodies = keyset.gen_seeded_forward_transciphering_keys(aes_key, seed)
    return ms, bodies, cbs.expand_seeded_fwd_trans_key(ms, bodies)


def _upload_seeded(ctx, mode, ms, bodies):
    (ctx.upload_seeded_trans_key if mode == "ecb" else ctx.upload_seeded_fwd_trans_key)(ms, bodies)


def _upload_full(ctx, mode, arrays):
    (ctx.upload_trans_key if mode == "ecb" else ctx.upload_fwd_trans_key)(*arrays)


def _bits_and_noise(keyset, rows):
    import ref_io
    phase = ref_io.lwe_phase(rows, keyset.glwe_sk)
    bits = ref_io.decode_bit(phase).astype(np.uint64)
    return bits, sdiff(phase, bits << np.uint64(63))


def _check_plaintext(bits, pt):
    want = np.unpackbits(np.frombuffer(pt, dtype=np.uint8)).astype(np.uint64)  # MSB first inside each byte
    bad = sorted(set((np.flatnonzero(bits != want) // 128).tolist()))
    nb = len(pt) // 16
    if bad and len(bad) <= max(1, nb // 4):
        raise NoiseFailure(f"blocks {bad[:8]} of {nb} decrypt wrongly")
    assert not bad, f"{len(bad)} of {nb} blocks wrong"


@pytest.mark.parametrize("mode", ["ecb", "ctr"])
def test_device_expansion_equals_host_expansion(sctx, cbs, keyset, aes_key, mode):
    """9 blocks = two lanes, so every LUT is read: the rows after the seeded upload are the rows after uploading the
    host-expanded arrays, bit for bit."""
    ms, bodies, full = _keys(cbs, keyset, aes_key, mode, 501)
    _, d_in = _inputs(aes_key, mode, 9, 502)
    _upload_seeded(sctx, mode, ms, bodies)
    seeded_rows = _host(_run(sctx, mode, d_in, 9))
    _upload_full(sctx, mode, full)
    full_rows = _host(_run(sctx, mode, d_in, 9))
    assert (seeded_rows == full_rows).all(), np.flatnonzero((seeded_rows != full_rows).any(axis=1))[:16]


@pytest.mark.parametrize("nb", [1, 8, 64])
@pytest.mark.parametrize("mode", ["ecb", "ctr"])
def test_end_to_end(sctx, cbs, keyset, aes_key, mode, nb):
    def run(attempt):
        ms, bodies = _keys(cbs, keyset, aes_key, mode, 600 + 10 * nb + attempt)[:2]
        _upload_seeded(sctx, mode, ms, bodies)
        pt, d_in = _inputs(aes_key, mode, nb, 700 + nb)
        bits, _ = _bits_and_noise(keyset, _host(_run(sctx, mode, d_in, nb)))
        _check_plaintext(bits, pt)

    retry_on_noise(run)


def test_noise_matches_the_reference_format_key(sctx, cbs, keyset, aes_key):
    """64 CTR blocks with a seeded key and with a reference-format key (trivial middle and last LUTs) of the same AES key:
    the LUTs' fresh GLWE noise (about 2^12) disappears under the ladder's, so the output noise agrees within 0.15 bits."""
    def run(attempt):
        pt, d_in = _inputs(aes_key, "ctr", 64, 801)
        ms, bodies = keyset.gen_seeded_forward_transciphering_keys(aes_key, 802 + attempt)
        sctx.upload_seeded_fwd_trans_key(ms, bodies)
        b_s, n_s = _bits_and_noise(keyset, _host(_run(sctx, "ctr", d_in, 64)))
        sctx.upload_fwd_trans_key(*keyset.gen_forward_transciphering_keys(aes_key, 803 + attempt))
        b_r, n_r = _bits_and_noise(keyset, _host(_run(sctx, "ctr", d_in, 64)))
        _check_plaintext(b_s, pt)
        _check_plaintext(b_r, pt)
        s_s, s_r = np.log2(n_s.std()), np.log2(n_r.std())
        print(f"64 CTR blocks: output noise std seeded 2^{s_s:.3f}, reference format 2^{s_r:.3f}")
        assert abs(s_s - s_r) < 0.15, (s_s, s_r)

    retry_on_noise(run)


def test_switching_key_forms_in_one_context(sctx, cbs, keyset, aes_key):
    """reference format -> seeded -> reference format: all decrypt, and the two reference-format runs are bit-identical
    (the trivial-LUT flag is set back by the second upload)."""
    def run(attempt):
        pt, d_in = _inputs(aes_key, "ecb", 9, 901)
        full = keyset.gen_transciphering_keys(aes_key, 902 + attempt)
        ms, bodies = keyset.gen_seeded_transciphering_keys(aes_key, 903 + attempt)
        sctx.upload_trans_key(*full)
        first = _host(_run(sctx, "ecb", d_in, 9))
        sctx.upload_seeded_trans_key(ms, bodies)
        seeded = _host(_run(sctx, "ecb", d_in, 9))
        sctx.upload_trans_key(*full)
        again = _host(_run(sctx, "ecb", d_in, 9))
        assert (first == again).all()
        for rows in (first, seeded):
            _check_plaintext(_bits_and_noise(keyset, rows)[0], pt)

    retry_on_noise(run)


def test_seeded_ctr_into_packing(sctx, cbs, keyset, aes_key):
    def run(attempt):
        ms, bodies = keyset.gen_seeded_forward_transciphering_keys(aes_key, 1001 + attempt)
        sctx.upload_seeded_fwd_trans_key(ms, bodies)
        pt, d_in = _inputs(aes_key, "ctr", 8, 1002)
        d_rows = _run(sctx, "ctr", d_in, 8)
        d_packed = torch.empty((1, 3072), dtype=torch.int64, device="cuda")
        sctx.pack_lwes_dev(d_rows.data_ptr(), 8 * 128, d_packed.data_ptr())
        bits = cbs.glwe_decrypt_bits(keyset.glwe_sk, d_packed.cpu().numpy().view(np.uint64), 8 * 128)
        _check_plaintext(bits, pt)

    retry_on_noise(run)


def test_seeded_upload_argument_errors(sctx, cbs):
    L = cbs.lib()
    seed = (ctypes.c_uint8 * 32)()
    bodies = np.zeros(cbs.TRANS_KEY_SEEDED_GLWES * 1024, dtype=np.uint64)
    pb = bodies.ctypes.data_as(ctypes.c_void_p)
    for fn in (L.cbs_trans_key_seeded_upload, L.cbs_fwd_trans_key_seeded_upload):
        assert fn(sctx._h, None, pb) == 1
        assert fn(sctx._h, seed, None) == 1
        assert fn(None, seed, pb) == 1
