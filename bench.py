#!/usr/bin/env python
"""bench.py — AES-128 blocks transciphered per second on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (ours; N>1 under torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...   (the reference's own CPU path, rank 0 only)
  python bench.py ... --dump-outputs DIR                    (also save the last step's outputs: compare two builds)

A step = one pass of the hot path (aes_to_lwe_trasnciphering, stage 7 of the reference) over one
batch of synthetic AES blocks: BLOCKS_PER_GPU = 8 blocks per GPU = the block count of the small
instance (BASELINE.json configs[1], 64 u16 values); at N GPUs every rank transciphers its own 8
blocks (weak scaling; N = 8 is the block count of the medium instance, 64).  The headline leg runs
ECB block DECRYPTION, the one mode the reference's stage 7 implements (so the reference arm times the
same operation); the harness encrypts sizes 1/2 in CTR mode (harness/aes_keygen_and_encrypt.py:49-55),
which needs forward AES on the counters - that path (cbs_aes128_ctr_transcipher_dev, what our stage 7
runs for sizes 1/2) is timed on the same 8 blocks and reported under "ctr".  Inputs: seeded FHE keys
(binary secrets, AES_TIGHT Gaussian noise), AES key sha256("None")[:16] as in the harness.  After the
timed region the last result is decrypted with the secret key and compared with the plaintext
("verified"; AES_TIGHT itself leaves ~0.05 % of blocks wrong, DESIGN.md section 2).
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLOCKS_PER_GPU = 8
CBS_PER_BLOCK = 1152           # 9 bootstrapped rounds x 128 state bits (SURVEY.md 3.2)
BR_MFLOP = 148.6               # FP64 MFLOP per blind rotation (SURVEY.md 8(d))
BSK_BYTES = 56_623_104         # Fourier bootstrapping key streamed once per launch
BR_IO_BYTES = 30_728           # LWE in + accumulator out per blind rotation
RF_WORDS_PER_WARP_STEP = 10_555  # register source words per warp and step of k_blind_rotate_v4 (csrc/tools/sass_rf_model.py)
NCU_BR_CSV = "r02_blind_rotate_ncu_full.csv"   # ncu --set full of k_blind_rotate_v4 on the 512-ciphertext lane shape the step launches
METRIC = "AES-128 blocks transciphered/sec"
UNIT = "blocks/s"
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, name, lwe, limit_bytes):
    """Write u64 LWE ciphertexts [..., 2049] to out_dir/name.npy as float64 torus values in [-1/2, 1/2) (the top 53 of the
    64 bits; noise sits at 2^58).  Above limit_bytes, a fixed seeded sample of whole ciphertexts in row order."""
    import numpy as np
    a = np.ascontiguousarray(lwe).view(np.int64)
    budget = limit_bytes - 4096  # room for the .npy header
    if a.nbytes > budget:
        rows = a.reshape(-1, a.shape[-1])
        keep = np.sort(np.random.default_rng(0).choice(rows.shape[0], budget // rows[0].nbytes, replace=False))
        a = rows[keep]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64) * 2.0 ** -64)


def read_ncu_traffic():
    """DRAM bytes per blind-rotation launch from the committed ncu --set full capture (profiles/)."""
    p = os.path.join(ROOT, "profiles", NCU_BR_CSV)
    try:
        rd = wr = None
        for line in open(p):
            f = line.strip().split(",")
            if f[0] == "dram__bytes_read.sum":
                rd = float(f[2]) * (1e6 if f[1] == "Mbyte" else 1e9 if f[1] == "Gbyte" else 1e3 if f[1] == "Kbyte" else 1)
            if f[0] == "dram__bytes_write.sum":
                wr = float(f[2]) * (1e6 if f[1] == "Mbyte" else 1e9 if f[1] == "Gbyte" else 1e3 if f[1] == "Kbyte" else 1)
        return None if rd is None or wr is None else rd + wr
    except Exception:
        return None


def read_ncu_metric(name):
    """One metric of the throughput blind-rotation kernel from the committed ncu --set full summary (profiles/)."""
    p = os.path.join(ROOT, "profiles", NCU_BR_CSV)
    try:
        for line in open(p):
            f = line.strip().split(",")
            if f[0] == name:
                return float(f[2])
    except Exception:
        pass
    return None


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.proc = None
        self.lines = []
        self.index = index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------------
# reference arm: the reference's own prebuilt, unmodified stage-7 binary on the host cores
def make_reference_workdirs(base, copies):
    """io/ + datasets/ for the toy instance (1 block, ECB).  Keys and transciphering key come from the REFERENCE's own
    prebuilt client binaries (oracle/_ref/client_key_generation, client_encode_encrypt), the AES ciphertext from the
    pure-Python oracle/aes_clear.py: nothing of this repository's library is loaded by the reference arm.
    One cwd per concurrent copy, sharing the read-only inputs."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import aes_clear
    ref = os.path.join(ROOT, "oracle", "_ref")
    shared = os.path.join(base, "shared")
    aes_key = aes_clear.harness_aes_key(None)
    vals = np.random.default_rng(5).integers(0, 65536, 8).tolist()
    ct = aes_clear.ecb_encrypt(aes_key, aes_clear.pack_u16_be(vals))
    os.makedirs(os.path.join(shared, "datasets", "toy"), exist_ok=True)
    open(os.path.join(shared, "datasets", "toy", "aes_key.hex"), "w").write(aes_key.hex())
    open(os.path.join(shared, "datasets", "toy", "db.hex"), "w").write(ct.hex())
    for exe in ("client_key_generation", "client_encode_encrypt"):
        subprocess.run([os.path.join(ref, exe), "0"], cwd=shared, check=True, stdout=subprocess.DEVNULL)
    dirs = []
    for c in range(copies):
        d = os.path.join(base, f"copy{c}")
        os.makedirs(os.path.join(d, "io", "toy"))
        os.symlink(os.path.join(shared, "datasets"), os.path.join(d, "datasets"))
        for sub in ("public_keys", "ciphertexts_upload", "secret_keys"):
            os.symlink(os.path.join(shared, "io", "toy", sub), os.path.join(d, "io", "toy", sub))
        dirs.append(d)
    return dirs, vals


def reference_decrypts_to(d, vals):
    """decrypt stage 7's result.bin with the reference's own client binaries and compare with the expected values."""
    ref = os.path.join(ROOT, "oracle", "_ref")
    for exe in ("client_decrypt_decode_aes_decryption", "client_postprocess_aes_decryption"):
        subprocess.run([os.path.join(ref, exe), "0"], cwd=d, check=True, stdout=subprocess.DEVNULL)
    got = [int(x) for x in open(os.path.join(d, "io", "toy", "result_aes.txt")).read().split()]
    return got == vals


def run_reference_wave(dirs, binary):
    t0 = time.perf_counter()
    procs = [subprocess.Popen([binary, "0"], cwd=d, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE) for d in dirs]
    for p in procs:
        _, err = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"reference binary failed: {err.decode()[:200]}")
    return time.perf_counter() - t0


def reference_blocks_per_s(copies, waves):
    """Returns (blocks/s, seconds per wave, kind, verified)."""
    binary = os.path.join(ROOT, "oracle", "_ref", "server_encrypted_aes_decryption")
    base = tempfile.mkdtemp(prefix="cbs_ref_")
    try:
        if os.path.exists(binary):
            dirs, vals = make_reference_workdirs(base, copies)
            times = [run_reference_wave(dirs, binary) for _ in range(waves)]
            ok = reference_decrypts_to(dirs[0], vals)
            t = sum(times) / len(times)
            return copies / t, t, "reference", bool(ok)
        # fallback: the C oracle port (OpenMP over all host threads), one block per "wave"
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import numpy as np
        import aes_clear
        import oracle
        import ref_io
        import temp_fhe_transciphering_b200 as cbs
        ks = cbs.KeySet.generate(777)
        aes_key = aes_clear.harness_aes_key(None)
        pt = bytes(range(16))
        ct = aes_clear.ecb_encrypt(aes_key, pt)
        tk = ks.gen_transciphering_keys(aes_key, 778)
        K = oracle.Keys(ks.bsk, ks.ksk, ks.auto_std, ks.ss)
        times = []
        for _ in range(waves):
            t0 = time.perf_counter()
            out = oracle.aes128_transcipher(K, ct, *tk)
            times.append(time.perf_counter() - t0)
        ok = np.packbits(ref_io.decode_bit(ref_io.lwe_phase(out[0], ks.glwe_sk))).tobytes() == pt
        t = sum(times) / len(times)
        return 1.0 / t, t, "port", bool(ok)
    finally:
        shutil.rmtree(base, ignore_errors=True)


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    # one wave = `cores` independent copies of the single-threaded reference binary, one AES block
    # each (~50 s); bounded to 2 timed waves so the arm ends within a few minutes whatever K is.
    waves = max(1, min(args.steps, 2))
    value, t_wave, kind, ok = reference_blocks_per_s(cores, waves)
    used = cores if kind == "reference" else None
    if kind == "port":
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle
        used = oracle.num_threads()
    sample = (f"{waves} wave(s) of {cores} concurrent single-threaded runs of the prebuilt reference "
              f"server_encrypted_aes_decryption, 1 AES block (1152 circuit bootstraps) each" if kind == "reference"
              else f"{waves} x 1 AES block through the OpenMP oracle port")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": waves, "warmup": 0, "requested_steps": args.steps, "requested_warmup": args.warmup,
        "ms_per_step": t_wave * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "AES-128 ECB block transciphering, AES_TIGHT, 1 block per process (the reference "
                               "cannot batch); throughput = concurrent copies / wall time"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "verified": ok,
    }
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------------------------------
def main_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import temp_fhe_transciphering_b200 as cbs
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import aes_clear

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        # keep stdout to the one JSON line: this image exports NCCL_DEBUG=VERSION, whose banner goes to stdout
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            del os.environ["NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    nblocks = args.blocks
    # --- untimed setup: client side (keys, transciphering key, AES ciphertext), replicated per GPU ---
    ks = cbs.KeySet.generate(20261018)
    aes_key = aes_clear.harness_aes_key(None)
    rng = np.random.default_rng(1000 + rank)
    pt = bytes(rng.integers(0, 256, 16 * nblocks, dtype=np.uint8))
    ct = aes_clear.ecb_encrypt(aes_key, pt)
    k10_9, k8_1, k0 = ks.gen_transciphering_keys(aes_key, 31337)
    ctx = cbs.Context(ks, local)
    # a dedicated non-default stream: the library launches on it and torch's events are recorded on it
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    ctx.upload_trans_key(k10_9, k8_1, k0)
    d_ct = torch.frombuffer(bytearray(ct), dtype=torch.uint8).cuda()
    d_out = torch.empty((nblocks, 128, 2049), dtype=torch.int64, device="cuda")
    # pinned host buffers for the end-to-end leg
    def pin(a):
        t = torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).pin_memory()
        return t, t.numpy().view(np.uint64)
    keep = []
    hk = []
    for a in (k10_9, k8_1, k0):
        t, v = pin(a)
        keep.append(t)
        hk.append(v)
    h_ct_t = torch.frombuffer(bytearray(ct), dtype=torch.uint8).pin_memory()
    h_out_t = torch.empty((nblocks, 128, 2049), dtype=torch.int64).pin_memory()
    lib = cbs.lib()
    import ctypes
    u64p = ctypes.POINTER(ctypes.c_uint64)
    u8p = ctypes.POINTER(ctypes.c_uint8)

    def e2e_call():
        rc = lib.cbs_aes128_transcipher(ctx._h, ctypes.cast(h_ct_t.data_ptr(), u8p), nblocks,
                                        hk[0].ctypes.data_as(u64p), hk[1].ctypes.data_as(u64p), hk[2].ctypes.data_as(u64p),
                                        ctypes.cast(h_out_t.data_ptr(), u64p))
        if rc != 0:
            raise RuntimeError(lib.cbs_last_error().decode())

    def dev_step():
        ctx.transcipher_dev(d_ct.data_ptr(), nblocks, d_out.data_ptr())

    # --- device-resident leg ---
    for _ in range(args.warmup):
        dev_step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        dev_step()
    e1.record(stream)
    barrier()
    launches = ctx.launch_count - l0
    clocks = sampler.stop() if rank == 0 else None
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    value = world * nblocks * args.steps / (ms_total * 1e-3)

    # --- CTR leg: the mode the harness uses for sizes 1/2 (forward AES of the public counters, 3 LUT multiples per byte,
    #     forward linear layer, XOR with the ciphertext bits); same blocks, device-resident, same timing rules ---
    iv = aes_clear.harness_iv(None)
    ctr_ct = aes_clear.ctr_crypt(aes_key, iv, pt)
    ctx.upload_fwd_trans_key(*ks.gen_forward_transciphering_keys(aes_key, 31338))
    counters = b"".join(((int.from_bytes(iv, "big") + b) % (1 << 128)).to_bytes(16, "big") for b in range(nblocks))
    d_ctr = torch.frombuffer(bytearray(counters), dtype=torch.uint8).cuda()
    d_cct = torch.frombuffer(bytearray(ctr_ct), dtype=torch.uint8).cuda()
    d_cout = torch.empty((nblocks, 128, 2049), dtype=torch.int64, device="cuda")
    ctr_steps = args.steps
    for _ in range(min(args.warmup, 3)):
        ctx.ctr_transcipher_dev(d_ctr.data_ptr(), d_cct.data_ptr(), nblocks, d_cout.data_ptr())
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record(stream)
    for _ in range(ctr_steps):
        ctx.ctr_transcipher_dev(d_ctr.data_ptr(), d_cct.data_ptr(), nblocks, d_cout.data_ptr())
    c1.record(stream)
    barrier()
    cms = torch.tensor([c0.elapsed_time(c1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(cms, op=dist.ReduceOp.MAX)
    ctr_value = world * nblocks * ctr_steps / (float(cms.item()) * 1e-3)

    # verify the last device-resident result (untimed)
    import ref_io
    ctr_ok = np.packbits(ref_io.decode_bit(ref_io.lwe_phase(d_cout.cpu().numpy().view(np.uint64).reshape(-1, 2049),
                                                            ks.glwe_sk))).tobytes() == pt
    out = d_out.cpu().numpy().view(np.uint64)
    bits, std, mx = ref_io.noise_stats(out.reshape(-1, 2049), ks.glwe_sk)
    verified = np.packbits(bits).tobytes() == pt

    # --- end-to-end leg: host buffers through the C ABI, H2D + D2H inside the timed region ---
    e2e_steps = args.steps
    for _ in range(min(args.warmup, 2)):
        e2e_call()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record(stream)
    for _ in range(e2e_steps):
        e2e_call()
    f1.record(stream)
    barrier()
    ems = torch.tensor([f0.elapsed_time(f1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ems, op=dist.ReduceOp.MAX)
    e2e_value = world * nblocks * e2e_steps / (float(ems.item()) * 1e-3)
    e2e_ok = np.packbits(ref_io.decode_bit(ref_io.lwe_phase(h_out_t.numpy().view(np.uint64).reshape(-1, 2049),
                                                            ks.glwe_sk))).tobytes() == pt
    h2d = 16 * nblocks + 8 * (cbs.K10_9_WORDS + cbs.K8_1_WORDS + cbs.K0_WORDS)
    d2h = nblocks * 128 * 2049 * 8

    # --- mini-workload of the small instance: encrypted max over the 8*nblocks transciphered u16 values
    #     (stage 8, server_encrypted_compute.rs), host buffers through the C ABI; reported, not part of `value` ---
    maxw = None
    ipw = None
    if rank == 0:
        res = h_out_t.numpy().view(np.uint64).reshape(-1, 2049)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ctx.max_u16(res)  # first call allocates the workspaces
        t_max_first = time.perf_counter() - t0
        t0 = time.perf_counter()
        mx_ct = ctx.max_u16(res)
        t_max = time.perf_counter() - t0
        got = ref_io.bits_to_u16(ref_io.decode_bit(ref_io.lwe_phase(mx_ct, ks.glwe_sk)))[0]
        want = max(aes_clear.unpack_u16_be(pt))
        maxw = {"values": 8 * nblocks, "seconds": t_max, "first_call_seconds": t_max_first, "verified": bool(got == want)}
        # mini-workload #2 (harness/cleartext_impl.py:65-70): inner product mod 2^16 of the two halves
        vals = aes_clear.unpack_u16_be(pt)
        t0 = time.perf_counter()
        ctx.inner_product_u16(res)
        t_ip_first = time.perf_counter() - t0
        t0 = time.perf_counter()
        ip_ct = ctx.inner_product_u16(res)
        t_ip = time.perf_counter() - t0
        got = ref_io.bits_to_u16(ref_io.decode_bit(ref_io.lwe_phase(ip_ct, ks.glwe_sk)))[0]
        h = len(vals) // 2
        want = sum((x * y) % 65536 for x, y in zip(vals[:h], vals[h:])) % 65536
        _, n_cbs, n_layers, n_ladders = cbs.inner_product_plan_check(np.array(vals, dtype=np.uint16))
        ipw = {"values": 8 * nblocks, "seconds": t_ip, "first_call_seconds": t_ip_first, "verified": bool(got == want), "circuit_bootstraps": n_cbs,
               "layers": n_layers, "lut_ladders": n_ladders}

    # --- roofline of the dominant kernel (blind rotation), timed alone with CUDA events ---
    roof = None
    cpu = None
    if rank == 0:
        # same launch shape as inside the step: the chunk runs as CBS_LANES (default 2) block-aligned lanes,
        # so one blind-rotation launch covers nblocks/lanes blocks
        lanes = max(1, min(int(os.environ.get("CBS_LANES", "2")), nblocks))
        B = (nblocks // lanes) * 128
        small = torch.from_numpy(ks.encrypt_bits_small(rng.integers(0, 2, B, dtype=np.uint8), 5).view(np.int64)).cuda()
        acc = torch.empty((B, 3072), dtype=torch.int64, device="cuda")
        for _ in range(2):
            ctx.blind_rotate_dev(small.data_ptr(), acc.data_ptr(), B)
        torch.cuda.synchronize()
        reps = 5
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        for _ in range(reps):
            ctx.blind_rotate_dev(small.data_ptr(), acc.data_ptr(), B)
        g1.record(stream)
        torch.cuda.synchronize()
        br_ms = g0.elapsed_time(g1) / reps
        fp64_peak = ctx.measure_fp64_tflops()
        hbm_peak, hbm_src = read_peaks()
        achieved = BR_MFLOP * 1e6 * B / (br_ms * 1e-3) * 1e-12
        props = torch.cuda.get_device_properties(0)
        sm_count = props.multi_processor_count
        sm_clock_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6 if isinstance(clocks, dict) else 1965.0e6
        br_bytes = BSK_BYTES + B * BR_IO_BYTES
        roof = {
            "kernel": "k_blind_rotate_v4", "bound": "fp64", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
            "frac": achieved / fp64_peak, "traffic": read_ncu_traffic(),
            "traffic_source": f"profiles/{NCU_BR_CSV} (ncu --set full, same kernel, same 512-ciphertext launch shape)",
            "peak_source": "FP64 FMA probe kernel, same run",
            # why frac cannot reach 1: the FMA probe counts 2 flop per issue slot, the transform mixes DADD/DMUL (1 flop)
            # with DFMA (2): 148.6 MFLOP per blind rotation are ~98.3 M FP64 instructions, so a saturated FP64 pipe would
            # read frac = 0.755; ncu's pipe-active figure of the same kernel (profiles/) is the like-for-like utilisation
            "frac_at_saturated_fp64_pipe": 148.6e6 / (768 * 64 * 2000.0 * 2.0),
            "ncu_fp64_pipe_active_pct_of_elapsed": read_ncu_metric("sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_elapsed"),
            "ncu_shared_pipe_pct_of_peak": read_ncu_metric("l1tex__data_pipe_lsu_wavefronts_mem_shared.sum.pct_of_peak_sustained_elapsed"),
            # the resource that actually binds (DESIGN.md section 4, profiles/r02_rf_microbench.txt): a scheduler reads two 32-bit
            # register words per cycle (a DFMA with three fresh sources issues every 3 cycles, not 2); the kernel's SASS reads
            # RF_WORDS_PER_WARP_STEP words per warp and step (csrc/tools/sass_rf_model.py)
            "register_file": {
                "bound": "register-file read bandwidth", "unit": "32-bit register words per clock per SM",
                "achieved": RF_WORDS_PER_WARP_STEP * 2 * 768 * B / (br_ms * 1e-3 * sm_clock_hz * sm_count),
                "peak": 8.0, "peak_source": "csrc/tools/bench_rf.cu on B200: 2 words per clock per scheduler",
                "frac": RF_WORDS_PER_WARP_STEP * 2 * 768 * B / (br_ms * 1e-3 * sm_clock_hz * sm_count) / 8.0,
                "sm_clock_mhz": sm_clock_hz * 1e-6,
                "words_per_blind_rotation": RF_WORDS_PER_WARP_STEP * 2 * 768,
            },
            "launch_ms": br_ms, "ciphertexts_per_launch": B, "launches_per_step": 9 * lanes,
            "share_of_step": br_ms * 9 * lanes / (ms_total / args.steps),
            "share_note": "lanes overlap on the device, so kernel shares of the step sum to more than 1; "
                          "ncu's serialised launch list (profiles/r02_launch_summary.csv) gives the share of the serialised sum",
            "hbm": {"bound": "hbm", "achieved": br_bytes / (br_ms * 1e-3) * 1e-9, "peak": hbm_peak, "unit": "GB/s",
                    "frac": br_bytes / (br_ms * 1e-3) * 1e-9 / hbm_peak, "peak_source": hbm_src + " MEASURED_PEAKS.json",
                    "algorithmic_bytes_per_launch": br_bytes},
        }
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            v, t_wave, kind, ok = reference_blocks_per_s(cores, 1)
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "verified": ok,
                   "sample": f"1 wave of {cores} concurrent single-threaded runs of the prebuilt reference stage-7 binary, "
                             f"1 AES block each ({t_wave:.1f} s)" if kind == "reference" else
                             f"1 AES block through the OpenMP oracle port ({t_wave:.1f} s)"}
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{nblocks} AES-128 ECB blocks per GPU (the block count of the small instance, size 1) = "
                                   f"{nblocks * 128} bit-ciphertexts x 9 bootstrapped rounds, AES_TIGHT; CTR mode of the same "
                                   f"blocks under 'ctr'",
                       "blocks_per_gpu": nblocks, "parallelism": f"blocks sharded over {world} GPU(s), replicated keys, "
                                                                   "no collective in the data path",
                       "l2": "per-step working set ~0.7 GB (Fourier GGSW 528 MB) exceeds the 126 MB L2"},
            "circuit_bootstraps_per_s": value * CBS_PER_BLOCK,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "verified": bool(e2e_ok)},
            "ctr": {"value": ctr_value, "unit": UNIT, "ms_per_step": float(cms.item()) / ctr_steps, "steps": ctr_steps,
                    "verified": bool(ctr_ok), "what": "cbs_aes128_ctr_transcipher_dev on the same blocks (harness sizes 1/2 mode)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "verified": bool(verified), "output_noise_log2_std": std, "output_noise_log2_max": mx,
            "roofline": roof,
            "max_u16_miniworkload": maxw,
            "inner_product_u16_miniworkload": ipw,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    if args.dump_outputs:
        # what the timed device-resident path returned in its last step (d_out is not written after the timed loop)
        dump_outputs(args.dump_outputs, "transcipher_out" if world == 1 else f"transcipher_out_rank{rank}", out,
                     DUMP_LIMIT_BYTES // world)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--blocks", type=int, default=BLOCKS_PER_GPU, help="AES blocks per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's output ciphertexts to DIR/transcipher_out.npy "
                         "(transcipher_out_rank<r>.npy per rank under torchrun; float64 torus values in [-1/2, 1/2); "
                         "at most 64 MB in all, a seeded sample of ciphertexts beyond)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        return main_reference(args)
    return main_ours(args)


if __name__ == "__main__":
    sys.exit(main())
