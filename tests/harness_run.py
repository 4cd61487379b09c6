"""Drive the reference's UNMODIFIED harness (harness/run_submission.py) against this repository's stage executables.

Test / measurement infrastructure, not product code.  The harness hard-codes where it finds things
(harness/run_submission.py:37-39: cwd/harness, cwd/submission/target/release; utils.py:58-66 also wants cwd/scripts), so
`layout()` builds exactly that tree in a scratch directory out of

  * oracle/_ref/harness, oracle/_ref/scripts  - the reference's own Python files, copied verbatim by `make -C oracle ref`
  * oracle/_ref/<client stage>                - the reference's own prebuilt client executables (key generation,
                                                encode/encrypt for the toy instance, decrypt, postprocess, the two no-op
                                                preprocess stages)
  * temp_fhe_transciphering_b200/bin/server_encrypted_aes_decryption, .../server_encrypted_compute - OURS (the GPU path)
  * temp_fhe_transciphering_b200/bin/client_encode_encrypt for sizes 1 and 2: the harness encrypts those in CTR mode
    (harness/aes_keygen_and_encrypt.py:49-55) and the reference's encoder only emits ECB-decryption keys

and `run()` executes `python3 harness/run_submission.py <size> [--mini_workload 1]` there with tests/shims (the pyaes
stand-in) on PYTHONPATH.  The harness does not forward --mini_workload to stage 8 (run_submission.py:97), so the
selection reaches our server_encrypted_compute through CBS_MINI_WORKLOAD.

CLI (builder runs, e.g. under gpurun):  python tests/harness_run.py --sizes 0 1 2 --out gpurun_out/r02_harness.json
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")
BIN = os.path.join(ROOT, "temp_fhe_transciphering_b200", "bin")
SHIMS = os.path.join(ROOT, "tests", "shims")

STAGES = ["client_preprocess", "client_key_generation", "client_encode_encrypt", "server_preprocess_dataset",
          "server_encrypted_aes_decryption", "server_encrypted_compute", "client_decrypt_decode_aes_decryption",
          "client_postprocess_aes_decryption", "client_decrypt_decode", "client_postprocess"]
SIZE_NAME = ["toy", "small", "medium"]


def available():
    return os.path.isfile(os.path.join(REF, "harness", "run_submission.py")) and os.path.isfile(os.path.join(REF, "client_key_generation"))


def layout(workdir, size, servers="ours", ref=REF):
    """Create harness/, scripts/, submission/target/release/ under workdir out of `ref` (a tree shaped like oracle/_ref)
    and bin/.  servers = "ours" | "reference"."""
    os.makedirs(workdir, exist_ok=True)
    for d in ("harness", "scripts"):
        dst = os.path.join(workdir, d)
        if os.path.exists(dst):
            shutil.rmtree(dst)
        shutil.copytree(os.path.join(ref, d), dst)
    rel = os.path.join(workdir, "submission", "target", "release")
    if os.path.exists(rel):
        shutil.rmtree(rel)
    os.makedirs(rel)
    origin = {}
    for st in STAGES:
        ours = servers == "ours" and (st.startswith("server_encrypted") or (st == "client_encode_encrypt" and size >= 1))
        src = os.path.join(BIN if ours else ref, st)
        if not os.path.isfile(src):
            raise FileNotFoundError(src)
        os.symlink(src, os.path.join(rel, st))  # $ORIGIN of our executables resolves through the link to bin/
        origin[st] = "ours" if ours else "reference"
    return origin


def run(workdir, size, mini_workload=0, seed=None, servers="ours", env_extra=None, timeout=3600):
    origin = layout(workdir, size, servers)
    env = dict(os.environ)
    env["PYTHONPATH"] = SHIMS + os.pathsep + env.get("PYTHONPATH", "")
    env["CBS_MINI_WORKLOAD"] = str(mini_workload)
    env["LD_LIBRARY_PATH"] = os.path.dirname(BIN) + os.pathsep + env.get("LD_LIBRARY_PATH", "")
    timing_file = os.path.join(workdir, "stage_timing.jsonl")
    env.setdefault("CBS_STAGE_TIMING", timing_file)  # per-phase breakdown of OUR stage processes (stage_common.h StageClock)
    if env_extra:
        env.update(env_extra)
    cmd = ["python3", os.path.join("harness", "run_submission.py"), str(size)]
    if mini_workload:
        cmd += ["--mini_workload", str(mini_workload)]
    if seed is not None:
        cmd += ["--seed", str(seed)]
    t0 = time.time()
    p = subprocess.run(cmd, cwd=workdir, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout)
    wall = time.time() - t0
    name = SIZE_NAME[size]
    res = {"size": size, "instance": name, "mini_workload": mini_workload, "servers": servers, "rc": p.returncode,
           "wall_s": round(wall, 3), "stage_origin": origin, "stdout": p.stdout,
           "pass_aes": "[harness] PASS AES Decryption" in p.stdout,
           "pass_result": any(l.startswith("[harness] PASS  (") for l in p.stdout.splitlines())}
    rj = os.path.join(workdir, "measurements", name, "results.json")
    if os.path.isfile(rj):
        res["results_json"] = json.load(open(rj))
    if os.path.isfile(timing_file):
        res["stage_timing"] = [json.loads(l) for l in open(timing_file) if l.strip()]
    return res


VALUES = [8, 64, 512]  # u16 values of the toy / small / medium instance (harness/params.py:39)
STAGE_LABEL = {"client_key_generation": "FHE Key Generation", "client_encode_encrypt": "AES key encoding and encryption",
               "server_encrypted_aes_decryption": "Encrypted aes decryption",
               "server_encrypted_compute": "Encrypted computation of mini workload"}


def replay(workdir, size, mini_workload=0, seed=None, timeout=3600):
    """Where oracle/_ref has no harness copy: the driver of harness/run_submission.py (SURVEY.md 3.1) replayed here with this
    repository's ten stage executables.  Dataset as harness/generate_dataset.py + aes_keygen_and_encrypt.py make it (random
    u16 values, AES key sha256("None")[:16], ECB for size 0 and CTR for sizes 1/2), the stages in the harness's order with
    argv[1] = size in cwd = workdir, then the verifiers' exact list equality against harness/cleartext_impl.py:52-70.
    Returns the same dict as run()."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import aes_clear
    name = SIZE_NAME[size]
    vals = np.random.default_rng(seed).integers(0, 65536, VALUES[size]).tolist()
    key = aes_clear.harness_aes_key(None)
    ds = os.path.join(workdir, "datasets", name)
    os.makedirs(ds)
    open(os.path.join(ds, "aes_key.hex"), "w").write(key.hex())
    if size == 0:
        ct = aes_clear.ecb_encrypt(key, aes_clear.pack_u16_be(vals))
    else:
        iv = aes_clear.harness_iv(None)
        open(os.path.join(ds, "aes_iv.hex"), "w").write(iv.hex())
        ct = aes_clear.ctr_crypt(key, iv, aes_clear.pack_u16_be(vals))
    open(os.path.join(ds, "db.hex"), "w").write(ct.hex())
    env = dict(os.environ)
    env["CBS_MINI_WORKLOAD"] = str(mini_workload)
    timing_file = os.path.join(workdir, "stage_timing.jsonl")
    env.setdefault("CBS_STAGE_TIMING", timing_file)
    per_stage, out, rc = {}, [], 0
    t0 = time.time()
    for st in STAGES:
        t = time.time()
        p = subprocess.run([os.path.join(BIN, st), str(size)], cwd=workdir, env=env, stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, text=True, timeout=timeout)
        per_stage[STAGE_LABEL.get(st, st)] = "%.4fs" % (time.time() - t)
        out.append(p.stdout)
        if p.returncode != 0:
            rc = p.returncode
            break
    wall = time.time() - t0

    def ints(f):
        path = os.path.join(workdir, "io", name, f)
        return [int(x) for x in open(path).read().split()] if os.path.isfile(path) else None

    h = len(vals) // 2
    want = sum((x * y) % 65536 for x, y in zip(vals[:h], vals[h:])) % 65536 if mini_workload else max(vals)
    res = {"size": size, "instance": name, "mini_workload": mini_workload, "servers": "ours", "rc": rc, "wall_s": round(wall, 3),
           "stage_origin": {st: "ours" for st in STAGES}, "stdout": "".join(out), "values": vals,
           "pass_aes": rc == 0 and ints("result_aes.txt") == vals, "pass_result": rc == 0 and ints("result.txt") == [want],
           "results_json": {"per_stage": per_stage, "total_latency_s": round(wall, 4)}}
    if os.path.isfile(timing_file):
        res["stage_timing"] = [json.loads(l) for l in open(timing_file) if l.strip()]
    return res


def summary(res):
    ps = res.get("results_json", {}).get("per_stage", {})
    return {"instance": res["instance"], "mini_workload": "inner_product" if res["mini_workload"] else "max", "servers": res["servers"],
            "pass_aes": res["pass_aes"], "pass_result": res["pass_result"], "rc": res["rc"],
            "stage7_s": ps.get("Encrypted aes decryption"), "stage8_s": ps.get("Encrypted computation of mini workload"),
            "keygen_s": ps.get("FHE Key Generation"), "encode_s": ps.get("AES key encoding and encryption"),
            "total_latency_s": res.get("results_json", {}).get("total_latency_s"), "wall_s": res["wall_s"],
            "stage_timing": res.get("stage_timing")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[0, 1, 2])
    ap.add_argument("--mini", type=int, nargs="+", default=[0, 1])
    ap.add_argument("--servers", default="ours")
    ap.add_argument("--out", default=None)
    ap.add_argument("--keep", action="store_true")
    a = ap.parse_args()
    if not available():
        sys.exit("oracle/_ref has no harness copy: run `make -C oracle ref` where /root/reference exists")
    rows = []
    for size in a.sizes:
        for mw in a.mini:
            d = tempfile.mkdtemp(prefix="harness_%s_" % SIZE_NAME[size])
            r = run(d, size, mw, servers=a.servers)
            s = summary(r)
            try:
                import torch
                s["gpus_visible"] = torch.cuda.device_count()
            except Exception:
                pass
            s["gpus_env"] = os.environ.get("CBS_GPUS")
            rows.append(s)
            print(json.dumps(s), flush=True)
            if not (r["pass_aes"] and r["pass_result"]):
                print(r["stdout"][-3000:], flush=True)
            if not a.keep:
                shutil.rmtree(d, ignore_errors=True)
    if a.out:
        with open(a.out, "w") as f:
            for s in rows:
                f.write(json.dumps(s) + "\n")
    sys.exit(0 if all(s["pass_aes"] and s["pass_result"] for s in rows) else 1)


if __name__ == "__main__":
    main()
