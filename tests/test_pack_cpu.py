"""LWE-to-GLWE packing on the CPU: the exact reference tests/exact_pack_ref.py pack_lwes decrypts to the packed bits, padding
with zero rows changes nothing, and the client helpers (cbs_glwe_decrypt_bits, cbs_glwe_list_save/load) agree with numpy
and with the bincode layout.  The GPU kernel is checked against the same reference in tests/test_pack_gpu.py."""
import numpy as np
import pytest

import exact_pack_ref as ex
from conftest import glwe_phase, sdiff

N = 1024


def lwe_noise(lwe, sk, bits):
    """signed phase - bit * 2^63 of big LWE rows"""
    lwe = np.asarray(lwe, dtype=np.uint64).reshape(-1, 2049)
    with np.errstate(over="ignore"):
        phase = lwe[:, 2048] - (lwe[:, :2048] * np.asarray(sk, dtype=np.uint64)).sum(axis=1)
    return sdiff(phase, np.asarray(bits, dtype=np.uint64) << np.uint64(63))


def packed_noise(glwe, sk, bits):
    """signed phase - bit * 2^63 of every coefficient of the packed GLWEs (bits padded with 0 to whole GLWEs)"""
    phase = glwe_phase(glwe, sk).reshape(-1)
    want = np.zeros(phase.size, dtype=np.uint64)
    want[: len(bits)] = np.asarray(bits, dtype=np.uint64) << np.uint64(63)
    return sdiff(phase, want)


@pytest.fixture(scope="module")
def inputs(keyset):
    bits = np.random.default_rng(51).integers(0, 2, 64).astype(np.uint8)
    return bits, keyset.encrypt_bits_big(bits, 52)


@pytest.mark.parametrize("count", [1, 2, 3, 17, 64])
def test_exact_pack_decrypts_to_the_bits(keyset, inputs, count):
    bits, lwe = inputs
    sk = keyset.glwe_sk
    glwe = ex.pack_lwes(keyset.auto_std, lwe[:count])
    assert glwe.shape == (1, 3 * N)
    e_in = lwe_noise(lwe[:count], sk, bits[:count])
    e_out = packed_noise(glwe, sk, bits[:count])
    print(f"count {count}: input noise max 2^{np.log2(np.abs(e_in).max()):.1f}, packed 2^{np.log2(np.abs(e_out).max()):.1f}, "
          f"packed - input 2^{np.log2(np.abs(e_out[:count] - e_in).max() + 1):.1f}, empty slots 2^{np.log2(np.abs(e_out[count:]).max() + 1):.1f}")
    assert (np.abs(e_out[:count]) <= np.abs(e_in) + 2.0 ** 42).all()
    assert (np.abs(e_out[count:]) <= 2.0 ** 42).all()
    from temp_fhe_transciphering_b200 import glwe_decrypt_bits
    assert (glwe_decrypt_bits(sk, glwe) == np.concatenate([bits[:count], np.zeros(N - count, np.uint8)])).all()


@pytest.mark.parametrize("count", [3, 17])
def test_exact_pack_zero_padding_changes_no_word(keyset, inputs, count):
    lwe = inputs[1][:count]
    padded = np.concatenate([lwe, np.zeros((N - count, 2049), dtype=np.uint64)])
    assert (ex.pack_lwes(keyset.auto_std, lwe) == ex.pack_lwes(keyset.auto_std, padded)).all()


def test_glwe_decrypt_bits_matches_numpy(cbs, keyset):
    rng = np.random.default_rng(53)
    sk = keyset.glwe_sk
    glwe = rng.integers(0, 2 ** 64, (3, 3 * N), dtype=np.uint64)
    want = (glwe_phase(glwe, sk).reshape(-1) + np.uint64(1 << 62)) >> np.uint64(63)
    assert (cbs.glwe_decrypt_bits(sk, glwe) == want).all()
    assert (cbs.glwe_decrypt_bits(sk, glwe, 2049) == want[:2049]).all()
    with pytest.raises(cbs.CbsError):
        cbs.glwe_decrypt_bits(sk, glwe, 3 * N + 1)


def test_glwe_list_save_load_layout(cbs, tmp_path):
    rng = np.random.default_rng(54)
    glwe = rng.integers(0, 2 ** 64, (2, 3 * N), dtype=np.uint64)
    path = tmp_path / "packed" / "result.bin"
    cbs.save_glwe_list(path, glwe)
    words = np.fromfile(path, dtype="<u8")
    assert words.size == 1 + 2 * 3 * N + 5
    assert words[0] == 2 * 3 * N and (words[1:1 + 2 * 3 * N] == glwe.reshape(-1)).all()
    assert words[-5:].tolist() == [3, 1024, 0, 0, 64]  # glwe_size, polynomial_size, modulus (u128 0, scalar bits 64)
    assert (cbs.load_glwe_list(path) == glwe).all()
    cbs.save_glwe_list(tmp_path / "empty.bin", np.zeros((0, 3 * N), dtype=np.uint64))
    assert cbs.load_glwe_list(tmp_path / "empty.bin").shape == (0, 3 * N)
    bad = words.copy()
    bad[-4] = 2048  # another polynomial size
    bad.tofile(tmp_path / "bad.bin")
    with pytest.raises(cbs.CbsError):
        cbs.load_glwe_list(tmp_path / "bad.bin")
    words[:-1].tofile(tmp_path / "short.bin")
    with pytest.raises(cbs.CbsError):
        cbs.load_glwe_list(tmp_path / "short.bin")
