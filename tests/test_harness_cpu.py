"""CPU checks of the harness plumbing (tests/harness_run.py, tests/shims/pyaes.py): the pyaes stand-in against FIPS-197
and the oracle's own cleartext AES, and the submission/target/release layout the harness hard-codes."""
import hashlib
import os
import sys

import pytest

import harness_run

sys.path.insert(0, harness_run.SHIMS)


def test_pyaes_shim_matches_fips197_and_oracle_aes():
    import aes_clear
    import pyaes
    key = bytes(range(16))
    pt = bytes.fromhex("00112233445566778899aabbccddeeff")
    ct = bytes(pyaes.AES(key).encrypt(pt))
    assert ct.hex() == "69c4e0d86a7b0430d8cdb78070b4c55a"  # FIPS-197 appendix C.1
    assert bytes(pyaes.AES(key).decrypt(ct)) == pt
    with pytest.raises(ValueError):
        pyaes.AES(key).encrypt(pt + pt)
    data = bytes(range(256)) * 4
    for iv in (hashlib.sha256(b"ivNone").digest()[:16], b"\xff" * 16, b"\x00" * 15 + b"\xfe"):
        ctr = pyaes.AESModeOfOperationCTR(key, counter=pyaes.Counter(int.from_bytes(iv, "big")))
        out = ctr.encrypt(data[:100]) + ctr.encrypt(data[100:])  # streaming, like pyaes
        assert out == aes_clear.ctr_crypt(key, iv, data)
        assert pyaes.AESModeOfOperationCTR(key, counter=pyaes.Counter(int.from_bytes(iv, "big"))).decrypt(out) == data


HARNESS_FILES = ("run_submission.py", "utils.py", "params.py", "cleartext_impl.py", "verify_result.py")


def _stand_in_reference(d):
    """A tree shaped like oracle/_ref (the reference's harness, scripts and client executables, which this repository does
    not contain) with placeholder files: enough to check what layout() builds where oracle/_ref is absent."""
    (d / "harness").mkdir(parents=True)
    (d / "scripts").mkdir()
    for f in HARNESS_FILES:
        (d / "harness" / f).write_text(f"# stand-in for the reference's harness/{f}\n")
    for st in harness_run.STAGES:
        (d / st).write_text("#!/bin/sh\nexit 0\n")
        (d / st).chmod(0o755)
    return str(d)


@pytest.mark.parametrize("size", [0, 1])
def test_layout_is_what_run_submission_expects(tmp_path, size):
    ref = harness_run.REF if harness_run.available() else _stand_in_reference(tmp_path / "ref")
    work = tmp_path / "work"
    origin = harness_run.layout(str(work), size, ref=ref)
    rel = work / "submission" / "target" / "release"
    for st in harness_run.STAGES:
        assert os.access(rel / st, os.X_OK), st
        src = os.path.join(harness_run.BIN if origin[st] == "ours" else ref, st)
        assert os.path.realpath(rel / st) == os.path.realpath(src), st
    assert origin["server_encrypted_aes_decryption"] == origin["server_encrypted_compute"] == "ours"
    assert origin["client_encode_encrypt"] == ("ours" if size >= 1 else "reference")
    for f in HARNESS_FILES:
        assert (work / "harness" / f).is_file()
    assert (work / "scripts").is_dir()
    # the harness is copied byte for byte
    assert open(os.path.join(ref, "harness", "run_submission.py"), "rb").read() == (work / "harness" / "run_submission.py").read_bytes()


@pytest.mark.parametrize("nblocks,cvd,gpus,want", [(1, "3,5,6", None, "3"), (64, "0,1,2,3,4,5,6,7", None, "0"),
                                                   (1024, "0,1,2,3,4,5,6,7", None, "0,1,2,3"), (8, "4,5", "2", "4,5"),
                                                   (4000, "0,1,2,3,4,5,6,7", None, "0,1,2,3,4,5,6,7")])
def test_stage_executable_plans_its_gpu_count_before_cuda_starts(tmp_path, nblocks, cvd, gpus, want):
    """stage_common.h plan_visible_gpus: driver start-up dominates a one-shot stage process (0.8 s with one GPU visible,
    5-9 s with eight), so stage 7 narrows CUDA_VISIBLE_DEVICES to sqrt(blocks / 53) devices before its first CUDA call."""
    import subprocess
    (tmp_path / "datasets" / "toy").mkdir(parents=True)
    (tmp_path / "datasets" / "toy" / "db.hex").write_text("00" * 16 * nblocks)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES=cvd, CBS_PLAN_DEBUG="1")
    env.pop("CBS_GPUS", None)
    if gpus:
        env["CBS_GPUS"] = gpus
    exe = os.path.join(harness_run.BIN, "server_encrypted_aes_decryption")
    p = subprocess.run([exe, "0"], cwd=tmp_path, env=env, capture_output=True, text=True, timeout=60)
    assert p.returncode != 0  # no keys in this directory: it stops right after the plan
    assert f"CUDA_VISIBLE_DEVICES={want}\n" in p.stderr, p.stderr
