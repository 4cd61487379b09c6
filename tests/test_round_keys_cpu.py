"""Transciphering keys of both directions (ECB: inverse AES, 4 multiples per byte; CTR: forward AES, 3 multiples) come from
one generator and one walk of the AllRdKeys file shape.  Seeded keys and the files written from them stay byte for byte
what they were before the two directions shared that code."""
import hashlib
import os

import pytest

# keyset seed 20261018 (conftest), the harness AES key, transciphering-key seed 99:
# sha256 of the generated arrays, sha256 and size of the key file
PINS = {
    "ecb": ("da4dc3ce346ed4b981bd917b6831ccc441399d13bb6ccf7a1456b5116b49bbeb",
            "02f7b0b0a3310352985408901b1f57a9e02fb0f8f4cbef778aa12a4420ab2cc3", 29_147_824),
    "ctr": ("bad63d335dbd4938f05824e52e449354332689fbf23dd5cd1273775ef98b8513",
            "469a006e09b03925feb2979d39bd29f8f34f9b4a16e818a1f2a8e26cf97d76bd", 22_057_832),
}


@pytest.fixture(scope="module")
def fwd_key(keyset, aes_key):
    return keyset.gen_forward_transciphering_keys(aes_key, 99)


def _io(cbs, direction):
    return (cbs.save_trans_key, cbs.load_trans_key) if direction == "ecb" else (cbs.save_fwd_trans_key, cbs.load_fwd_trans_key)


@pytest.mark.parametrize("direction", ["ecb", "ctr"])
def test_seeded_key_and_file_bytes_and_round_trip(cbs, trans_key, fwd_key, direction, tmp_path):
    key = trans_key if direction == "ecb" else fwd_key
    save, load = _io(cbs, direction)
    arrays_sha, file_sha, size = PINS[direction]
    assert hashlib.sha256(b"".join(a.tobytes() for a in key)).hexdigest() == arrays_sha
    path = tmp_path / "trans_key.bin"
    save(path, *key)
    assert os.path.getsize(path) == size
    assert hashlib.sha256(path.read_bytes()).hexdigest() == file_sha
    for a, b in zip(load(path), key):
        assert a.shape == b.shape and (a == b).all()


def test_key_file_of_one_direction_is_rejected_by_the_other(cbs, trans_key, fwd_key, tmp_path):
    cbs.save_trans_key(tmp_path / "ecb.bin", *trans_key)
    cbs.save_fwd_trans_key(tmp_path / "ctr.bin", *fwd_key)
    with pytest.raises(cbs.CbsError, match="not a forward"):
        cbs.load_fwd_trans_key(tmp_path / "ecb.bin")
    with pytest.raises(cbs.CbsError, match="not an AllRdKeys file"):
        cbs.load_trans_key(tmp_path / "ctr.bin")
