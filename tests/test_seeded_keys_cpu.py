"""Seeded transciphering keys on the host (no GPU): every LUT encrypted, masks from a public ChaCha20 stream.

The mask stream is checked against a numpy ChaCha20 written here from RFC 8439 (itself checked against the RFC's test vector),
the LUT contents against the reference-format generator's keyed tables, and the leak the seeded form closes is shown on the
reference-format key."""
import ctypes

import numpy as np
import pytest

from conftest import glwe_phase, sdiff

G = {"inv": 1184, "fwd": 896}
DIR = {"inv": 0, "fwd": 1}
NFIRST = {"inv": 128, "fwd": 96}


# ---- numpy ChaCha20 (RFC 8439 section 2.3) ---------------------------------------------------------------------------

def chacha20_blocks(key, counters, nonces):
    """key: 32 bytes; counters: (n,) u32; nonces: (n, 3) u32 -> (n, 16) u32, the serialized blocks as little-endian words"""
    counters = np.asarray(counters, dtype=np.uint32)
    n = counters.size
    state = np.empty((16, n), dtype=np.uint32)
    state[:4] = np.array([0x61707865, 0x3320646e, 0x79622d32, 0x6b206574], dtype=np.uint32)[:, None]
    state[4:12] = np.frombuffer(bytes(key), dtype="<u4")[:, None]
    state[12] = counters
    state[13:16] = np.asarray(nonces, dtype=np.uint32).reshape(n, 3).T
    x = state.copy()

    def rotl(v, k):
        return (v << np.uint32(k)) | (v >> np.uint32(32 - k))

    def qr(a, b, c, d):
        x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 16)  # noqa: E702
        x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 12)  # noqa: E702
        x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 8)  # noqa: E702
        x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 7)  # noqa: E702

    for _ in range(10):
        qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15)  # noqa: E702
        qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14)  # noqa: E702
    return (x + state).T.copy()


def mask_stream(mask_seed, direction, nglwe):
    """The masks of a seeded key as specified: [nglwe][2048] u64, word w of GLWE g from block (counter w/8, nonce (g, dir,
    "mask")), word i = out[2i] | out[2i+1] << 32"""
    g = np.repeat(np.arange(nglwe, dtype=np.uint32), 256)
    blk = np.tile(np.arange(256, dtype=np.uint32), nglwe)
    nonces = np.stack([g, np.full_like(g, direction), np.full_like(g, 0x6b73616d)], axis=1)
    out = chacha20_blocks(mask_seed, blk, nonces).astype(np.uint64)
    words = out[:, 0::2] | (out[:, 1::2] << np.uint64(32))
    return words.reshape(nglwe, 2048)


def test_chacha20_rfc8439_vector():
    key = bytes(range(32))
    nonce = bytes.fromhex("000000090000004a00000000")
    want = bytes.fromhex("10f1e7e4d13b5915500fdd1fa32071c4c7d1f4c733c068030422aa9ac3d46c4e"
                         "d2826446079faa0914c2d705d98b02a2b5129cd1de164eb9cbd083e8a2503c4e")
    got = chacha20_blocks(key, [1], np.frombuffer(nonce, dtype="<u4")[None]).astype("<u4").tobytes()
    assert got == want
    try:
        from cryptography.hazmat.primitives.ciphers import Cipher, algorithms
    except ImportError:
        return
    enc = Cipher(algorithms.ChaCha20(key, (1).to_bytes(4, "little") + nonce), mode=None).encryptor()
    assert enc.update(bytes(64)) == want


# ---- fixtures ---------------------------------------------------------------------------------------------------------

def _flat(arrays):
    return np.concatenate([np.asarray(a).reshape(-1, 3, 1024) for a in arrays])


@pytest.fixture(scope="module")
def seeded(keyset, aes_key):
    """per direction: (mask_seed, bodies, expanded GLWE [G][3][1024] in AllRdKeys order)"""
    from temp_fhe_transciphering_b200 import expand_seeded_fwd_trans_key, expand_seeded_trans_key
    out = {}
    for d, gen, expand in (("inv", keyset.gen_seeded_transciphering_keys, expand_seeded_trans_key),
                           ("fwd", keyset.gen_seeded_forward_transciphering_keys, expand_seeded_fwd_trans_key)):
        ms, bodies = gen(aes_key, 4711)
        out[d] = (ms, bodies, _flat(expand(ms, bodies)))
    return out


@pytest.fixture(scope="module")
def reference_format(keyset, aes_key):
    """per direction: the reference-format key as GLWE [G][3][1024] (first rounds encrypted, the rest trivial)"""
    return {"inv": _flat(keyset.gen_transciphering_keys(aes_key, 4712)),
            "fwd": _flat(keyset.gen_forward_transciphering_keys(aes_key, 4712))}


@pytest.fixture(scope="module")
def seeded_phases(seeded, keyset):
    return {d: glwe_phase(seeded[d][2], keyset.glwe_sk) for d in seeded}


def _check_tables(phase, ref, glwe_sk, nfirst):
    """phases of a fully encrypted key against the reference-format key: middle/last rounds within 2^20 of the trivial
    LUT's body, first rounds within 2^21 of the encrypted LUT's phase"""
    assert phase.shape[0] == ref.shape[0]
    first = np.abs(sdiff(phase[:nfirst], glwe_phase(ref[:nfirst], glwe_sk))).max()
    rest = np.abs(sdiff(phase[nfirst:], ref[nfirst:, 2])).max()
    assert first < 2.0 ** 21, np.log2(first)
    assert rest < 2.0 ** 20, np.log2(rest)


# ---- expansion ----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("d", ["inv", "fwd"])
def test_expansion_is_the_specified_stream(seeded, d):
    ms, bodies, glwe = seeded[d]
    assert len(ms) == 32 and bodies.shape == (G[d], 1024) and glwe.shape == (G[d], 3, 1024)
    assert (glwe[:, :2].reshape(G[d], 2048) == mask_stream(ms, DIR[d], G[d])).all()
    assert (glwe[:, 2] == bodies).all()  # words 2048..3071 of every GLWE


@pytest.mark.parametrize("d", ["inv", "fwd"])
def test_same_tables_as_the_reference_format_key(seeded_phases, reference_format, keyset, d):
    _check_tables(seeded_phases[d], reference_format[d], keyset.glwe_sk, NFIRST[d])


# ---- the leak ----------------------------------------------------------------------------------------------------------

def test_reference_format_bodies_show_the_round_keys(reference_format, aes_key):
    """The leak: in the reference-format forward key, middle block i, multiple 1, byte b is the table S(x ^ rk_{i+1}[b]) with
    bit 4a + t of entry x in the top bit of body coefficient 256 t + x of accumulator a.  Reading it back gives every round
    key rk1..rk8, and the whole table, exactly."""
    import aes_clear
    rk = aes_clear.expand_key(aes_key)
    mid = reference_format["fwd"][96:96 + 8 * 96].reshape(8, 3, 16, 2, 3, 1024)
    top = (mid[:, 0, :, :, 2] >> np.uint64(63)).astype(np.uint32).reshape(8, 16, 2, 4, 256)  # [round][byte][a][t][x]
    tables = sum(top[:, :, a, t] << (4 * a + t) for a in range(2) for t in range(4))  # [round][byte][x]
    for i in range(8):
        for b in range(16):
            x = int(np.flatnonzero(tables[i, b] == aes_clear.SBOX[0])[0])  # S(x ^ k) = S(0) at x = k
            assert x == rk[i + 1][b]
            assert tables[i, b].tolist() == [aes_clear.SBOX[v ^ x] for v in range(256)]


def test_seeded_bodies_hide_the_tables(seeded, reference_format):
    """The top bits of the seeded middle bodies agree with the table bits at chance, over all 2^20 middle coefficients."""
    table_bits = reference_format["inv"][128:128 + 1024, 2] >> np.uint64(63)
    body_bits = seeded["inv"][1][128:128 + 1024] >> np.uint64(63)
    assert table_bits.size == 1 << 20
    assert abs((table_bits == body_bits).mean() - 0.5) < 0.01


# ---- fresh and distinct masks ------------------------------------------------------------------------------------------

def test_masks_fresh_and_distinct(seeded):
    blocks = []
    for d in ("inv", "fwd"):
        masks = seeded[d][2][:, :2]
        assert (masks != 0).all()
        blocks.append(masks.reshape(-1, 8))
    assert seeded["inv"][0] == seeded["fwd"][0]  # one seed: only the direction in the nonce keeps the two streams apart
    rows = np.ascontiguousarray(np.concatenate(blocks)).view(np.dtype((np.void, 64)))
    assert np.unique(rows).size == rows.size == (G["inv"] + G["fwd"]) * 256


def test_os_entropy_keys_differ_and_decrypt(keyset, aes_key, reference_format):
    from temp_fhe_transciphering_b200 import expand_seeded_fwd_trans_key
    (s1, b1), (s2, b2) = (keyset.gen_seeded_forward_transciphering_keys(aes_key) for _ in range(2))
    assert s1 != s2 and len(s1) == len(s2) == 32
    assert (b1 != b2).mean() > 0.99
    for s, b in ((s1, b1), (s2, b2)):
        phase = glwe_phase(_flat(expand_seeded_fwd_trans_key(s, b)), keyset.glwe_sk)
        _check_tables(phase, reference_format["fwd"], keyset.glwe_sk, NFIRST["fwd"])


def test_deterministic_variant_is_reproducible(keyset, aes_key, seeded):
    ms, bodies = keyset.gen_seeded_transciphering_keys(aes_key, 4711)
    assert ms == seeded["inv"][0] and (bodies == seeded["inv"][1]).all()
    assert keyset.gen_seeded_transciphering_keys(aes_key, 4713)[0] != ms


# ---- files ---------------------------------------------------------------------------------------------------------------

def test_files(tmp_path, cbs, seeded):
    ms_i, b_i = seeded["inv"][:2]
    ms_f, b_f = seeded["fwd"][:2]
    pi, pf = tmp_path / "inv.seeded", tmp_path / "sub" / "fwd.seeded"
    cbs.save_seeded_trans_key(pi, ms_i, b_i)
    cbs.save_seeded_fwd_trans_key(pf, ms_f, b_f)
    assert pi.stat().st_size == 56 + 8192 * G["inv"]
    assert pf.stat().st_size == 56 + 8192 * G["fwd"]
    raw = pi.read_bytes()
    assert raw[:8] == b"CBSSEED1" and raw[16:48] == ms_i
    ms, b = cbs.load_seeded_trans_key(pi)
    assert ms == ms_i and (b == b_i).all()
    ms, b = cbs.load_seeded_fwd_trans_key(pf)
    assert ms == ms_f and (b == b_f).all()
    bad = {"other direction": None, "truncated": raw[:-8], "trailing": raw + b"\0", "magic": b"CBSSEED2" + raw[8:],
           "count": raw[:48] + (G["inv"] * 1024 + 1).to_bytes(8, "little") + raw[56:]}
    for name, data in bad.items():
        path = pf if data is None else tmp_path / (name + ".seeded")
        if data is not None:
            path.write_bytes(data)
        with pytest.raises(cbs.CbsError, match=r"\(code 3\)"):
            cbs.load_seeded_trans_key(path)
    with pytest.raises(cbs.CbsError, match=r"\(code 3\)"):
        cbs.load_seeded_fwd_trans_key(pi)


# ---- errors ----------------------------------------------------------------------------------------------------------------

def test_null_arguments(cbs, keyset, aes_key):
    L = cbs.lib()
    seed = (ctypes.c_uint8 * 32)()
    bodies = np.zeros(G["inv"] * 1024, dtype=np.uint64)
    pb = bodies.ctypes.data_as(ctypes.c_void_p)
    key = (ctypes.c_uint8 * 16).from_buffer_copy(aes_key)
    out = np.zeros(8 * 4 * 16 * 2 * 3072, dtype=np.uint64)
    po = out.ctypes.data_as(ctypes.c_void_p)
    calls = []
    for fn in ("cbs_trans_key_seeded_generate", "cbs_fwd_trans_key_seeded_generate"):
        f = getattr(L, fn)
        calls += [lambda f=f: f(None, key, ctypes.c_uint64(1), seed, pb), lambda f=f: f(keyset._h, None, ctypes.c_uint64(1), seed, pb),
                  lambda f=f: f(keyset._h, key, ctypes.c_uint64(1), None, pb), lambda f=f: f(keyset._h, key, ctypes.c_uint64(1), seed, None)]
        f = getattr(L, fn + "_os_entropy")
        calls += [lambda f=f: f(None, key, seed, pb), lambda f=f: f(keyset._h, key, None, pb), lambda f=f: f(keyset._h, key, seed, None)]
    for fn in ("cbs_trans_key_seeded_expand", "cbs_fwd_trans_key_seeded_expand"):
        f = getattr(L, fn)
        calls += [lambda f=f: f(None, pb, po, po, po), lambda f=f: f(seed, None, po, po, po), lambda f=f: f(seed, pb, None, po, po),
                  lambda f=f: f(seed, pb, po, None, po), lambda f=f: f(seed, pb, po, po, None)]
    for fn in ("cbs_trans_key_seeded_save", "cbs_fwd_trans_key_seeded_save"):
        f = getattr(L, fn)
        calls += [lambda f=f: f(None, seed, pb), lambda f=f: f(b"/nonexistent/x", None, pb), lambda f=f: f(b"/nonexistent/x", seed, None)]
    for i, call in enumerate(calls):
        assert call() == 1, i
    # a keyset without the secret key cannot generate
    pub = cbs.KeySet.from_arrays(keyset.bsk, keyset.ksk, keyset.auto_std, keyset.ss)
    with pytest.raises(cbs.CbsError, match=r"\(code 1\)"):
        pub.gen_seeded_transciphering_keys(aes_key, 1)
