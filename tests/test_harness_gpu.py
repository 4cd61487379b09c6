"""The reference's UNMODIFIED harness/run_submission.py (copied verbatim to oracle/_ref/harness by `make -C oracle ref`)
drives the stage executables: reference client binaries + OUR server_encrypted_aes_decryption / server_encrypted_compute
(+ our client_encode_encrypt for the CTR instances), laid out under submission/target/release as
harness/run_submission.py:39 hard-codes.  Both verifiers (verify_aes_decryption.py, verify_result.py) must print PASS,
at every instance size and for both mini-workloads (north star: "drops into run_submission.py unchanged").
Where oracle/_ref has no harness copy, harness_run.replay runs the same stage sequence, datasets and checks with this
repository's ten executables.
The per-stage wall times the harness records (utils.py:85-141 -> measurements/<size>/results.json) are printed; the
builder's copies live in profiles/r02_harness_*.jsonl and DESIGN.md section 5."""
import json

import pytest

import harness_run
from conftest import NoiseFailure, retry_on_noise

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("size", [0, 1, 2])
@pytest.mark.parametrize("mini_workload", [0, 1])
def test_run_submission_unchanged(tmp_path, size, mini_workload):
    harness = harness_run.available()
    drive = harness_run.run if harness else harness_run.replay

    def attempt(k):
        res = drive(str(tmp_path / f"try{k}"), size, mini_workload)
        print(json.dumps(harness_run.summary(res)))
        assert res["rc"] == 0, res["stdout"][-4000:]
        assert res["stage_origin"]["server_encrypted_aes_decryption"] == "ours"
        assert res["stage_origin"]["server_encrypted_compute"] == "ours"
        assert res["stage_origin"]["client_key_generation"] == ("reference" if harness else "ours")
        per_stage = res["results_json"]["per_stage"]
        assert "Encrypted aes decryption" in per_stage and "Encrypted computation of mini workload" in per_stage
        if not (res["pass_aes"] and res["pass_result"]):
            # a FAIL of the harness's verifiers with exit code 0 everywhere: AES_TIGHT's own failure probability
            # (conftest.NoiseFailure) - the keys are fresh on every run, so run the harness again
            raise NoiseFailure("harness verifier printed FAIL: " + " | ".join(
                l for l in res["stdout"].splitlines() if "FAIL" in l)[:400] if harness else
                f"decrypted results differ from the cleartext (values {res['values'][:16]}...)")
        return res

    retry_on_noise(attempt)
