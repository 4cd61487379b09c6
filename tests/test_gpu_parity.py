"""GPU parity tests: every CUDA stage, called through the C ABI, against the CPU oracle on the same
seeded inputs.  Integer/byte work is bit-exact; stages that go through the FP64 FFT differ from the
oracle only by floating-point summation order, so they are compared with a tolerance far below
the ciphertext noise (stated per test, in log2 of the torus scale 2^64) AND by decrypting with the
secret key.  Tolerances follow SURVEY.md Appendix A's measured per-stage noise levels."""
import numpy as np
import pytest

from conftest import glwe_phase, log2max, sdiff

pytestmark = pytest.mark.gpu

N = 1024


def _bits(n, seed):
    return np.random.default_rng(seed).integers(0, 2, n, dtype=np.uint8)


def test_lwe_keyswitch_matches_oracle(ctx, orc, orc_keys, keyset):
    import ref_io
    bits = _bits(24, 1)
    big = keyset.encrypt_bits_big(bits, 11)
    got = ctx.keyswitch_lwe_ciphertext_by_glwe_keyswitch(big)
    want = orc.lwe_keyswitch(orc_keys, big)
    # FFT round-off of a B=2^4, l=3 product against 64-bit key words: ~2^20; LWE noise is ~2^47
    assert log2max(sdiff(got, want)) < 30
    ph = ref_io.lwe_phase(got, keyset.lwe_sk_small)
    assert (ref_io.decode_bit(ph) == bits).all()
    # keyswitch noise: 12 decomposed bits of 2048 mask words -> ~2^(64-12-1) * sqrt(2048/2) ~ 2^56.5
    assert log2max(ref_io.bit_error(ph, bits)) < 58.5


def test_blind_rotate_single_step_matches_oracle(ctx, orc, orc_keys):
    """One non-zero mask element = one external product: the ciphertexts themselves must agree up to
    FP64 round-off (B = 2^23 digits x 64-bit key words over 3072 terms: ~2^41)."""
    rng = np.random.default_rng(21)
    lwe = np.zeros((4, 769), dtype=np.uint64)
    for i in range(4):
        lwe[i, 100 * i + 7] = rng.integers(1 << 56, 1 << 63, dtype=np.uint64)
        lwe[i, 768] = rng.integers(0, 1 << 63, dtype=np.uint64)
    got = ctx.blind_rotate(lwe)
    want = orc.blind_rotate(orc_keys, lwe)
    assert log2max(sdiff(got, want)) < 44, log2max(sdiff(got, want))


def test_blind_rotate_matches_oracle(ctx, orc, orc_keys, keyset):
    bits = _bits(6, 2)
    small = keyset.encrypt_bits_small(bits, 12)
    got = ctx.blind_rotate(small)
    want = orc.blind_rotate(orc_keys, small)
    # After the first of the 768 external products the two FP64 evaluations round a few digits
    # differently, which re-randomises the masks, so from then on they are two INDEPENDENT samples of
    # the same noisy result: their phases differ by sqrt(2) x the blind-rotation noise (2^48.5 std,
    # dominated by the B = 2^23 decomposition rounding; SURVEY.md Appendix A), i.e. ~2^49 std / 2^51 max.
    # Bit-level agreement of the arithmetic is pinned by the single-step test above.
    pg, pw = glwe_phase(got, keyset.glwe_sk), glwe_phase(want, keyset.glwe_sk)
    d = sdiff(pg, pw)
    assert log2max(d) < 52.0, log2max(d)
    assert np.log2(d.std() + 1) < 49.7, np.log2(d.std() + 1)
    # decrypt: coefficient lvl of the accumulator holds bit*2^(64-2(lvl+1)) - 2^(63-2(lvl+1))
    ph = pg
    for i, b in enumerate(bits):
        for lvl in range(7):
            val = int(ph[i, lvl]) + (1 << (63 - 2 * (lvl + 1)))
            val &= (1 << 64) - 1
            want_val = (int(b) << (64 - 2 * (lvl + 1))) & ((1 << 64) - 1)
            err = (val - want_val + (1 << 63)) % (1 << 64) - (1 << 63)
            assert abs(err) < 2 ** 52, (i, lvl, np.log2(abs(err) + 1))


def test_blind_rotate_throughput_and_team_kernels(ctx, orc, orc_keys, keyset):
    """Batches of at most 2 ciphertexts per SM run the 192-thread-team kernel (the tests above), larger ones the
    4-groups-per-CTA throughput kernel: a 300-ciphertext batch must decrypt correctly, match the oracle in its single-step
    arithmetic, and agree in phase with the team kernel on the same inputs."""
    bits = _bits(300, 31)
    small = keyset.encrypt_bits_small(bits, 33)
    big = ctx.blind_rotate(small)            # throughput kernel
    team = ctx.blind_rotate(small[:6])       # team kernel
    ph = glwe_phase(big, keyset.glwe_sk)
    for lvl in range(7):
        val = (ph[:, lvl] + np.uint64(1 << (63 - 2 * (lvl + 1))))
        want = bits.astype(np.uint64) << np.uint64(64 - 2 * (lvl + 1))
        assert log2max(sdiff(val, want)) < 52
    d = sdiff(ph[:6], glwe_phase(team, keyset.glwe_sk))
    assert log2max(d) < 52.0, log2max(d)
    # one full wave through the throughput kernel + the remainder through the team kernel (mixed launch)
    nsm = __import__("torch").cuda.get_device_properties(0).multi_processor_count
    bits2 = _bits(4 * nsm + 5, 35)
    ph2 = glwe_phase(ctx.blind_rotate(keyset.encrypt_bits_small(bits2, 36)), keyset.glwe_sk)
    val = ph2[:, 0] + np.uint64(1 << 61)
    assert log2max(sdiff(val, bits2.astype(np.uint64) << np.uint64(62))) < 52
    # single external product through the throughput kernel: ciphertext-level agreement with the oracle
    rng = np.random.default_rng(22)
    lwe = np.zeros((300, 769), dtype=np.uint64)
    for i in range(300):
        lwe[i, (37 * i + 5) % 768] = rng.integers(1 << 56, 1 << 63, dtype=np.uint64)
        lwe[i, 768] = rng.integers(0, 1 << 63, dtype=np.uint64)
    got = ctx.blind_rotate(lwe)
    want = orc.blind_rotate(orc_keys, lwe[:4])
    assert log2max(sdiff(got[:4], want)) < 44


def test_glev_from_acc_bit_exact(ctx, orc):
    acc = np.random.default_rng(3).integers(0, 2 ** 64, (5, 3072), dtype=np.uint64)
    got = ctx.glev_from_acc(acc)
    want = orc.glev_from_acc(acc)
    assert (got == want).all()


def test_trace_matches_oracle(ctx, orc, orc_keys, keyset):
    rng = np.random.default_rng(4)
    acc = ctx.blind_rotate(keyset.encrypt_bits_small(_bits(2, 5), 13))
    pre = orc.glev_from_acc(acc).reshape(-1, 3072)[:5]
    got = ctx.trace_assign(pre)
    want = orc.trace(orc_keys, pre)
    d = sdiff(got, want)
    # split-FFT keyswitch round-off ~2^13 per step (SURVEY.md 7 "FFT precision"), 10 steps doubling
    assert log2max(d) < 30, log2max(d)
    # the trace kills every non-constant coefficient: phase[j != 0] is pure noise <= 2^40
    ph = glwe_phase(got, keyset.glwe_sk).astype(np.int64).astype(np.float64)
    assert log2max(ph[:, 1:]) < 42


def test_scheme_switch_matches_oracle(ctx, orc, orc_keys, keyset):
    small = keyset.encrypt_bits_small(_bits(2, 6), 14)
    glev = ctx.lwe_msb_bit_to_glev_by_trace_with_preprocessing(small)
    got = ctx.switch_scheme(glev)
    want = orc.scheme_switch(orc_keys, glev)
    d = sdiff(got, want)
    assert log2max(d) < 40, log2max(d)
    # rows k (copies of the GLEV) are bit-exact
    g = got.reshape(-1, 7, 3, 3072)
    assert (g[:, :, 2] == glev.reshape(-1, 7, 3072)).all()


def test_circuit_bootstrap_decrypts(ctx, orc, orc_keys, keyset):
    bits = _bits(8, 7)
    small = keyset.encrypt_bits_small(bits, 15)
    ggsw = ctx.circuit_bootstrap_lwe_ciphertext_by_trace_with_preprocessing(small).reshape(-1, 7, 3, 3, 1024)
    sk = keyset.glwe_sk.reshape(2, 1024)
    worst = 0.0
    for i, b in enumerate(bits):
        for lvl in range(7):
            scale = 64 - 2 * (lvl + 1)
            ph = glwe_phase(ggsw[i, lvl].reshape(3, 3072), keyset.glwe_sk)  # [3 rows][1024]
            for row in range(3):
                want = np.zeros(1024, dtype=np.uint64)
                if b:
                    if row < 2:
                        want = (np.uint64(0) - sk[row]) << np.uint64(scale)
                    else:
                        want[0] = np.uint64(1) << np.uint64(scale)
                worst = max(worst, log2max(sdiff(ph[row], want)))
    # SURVEY.md Appendix A: CBS GGSW rows max error 2^49.8 .. 2^50.8
    assert worst < 52.5, worst
    # and the whole pipeline agrees with the oracle in PHASE (ciphertexts re-randomise, see above)
    want = orc.circuit_bootstrap(orc_keys, small[:2]).reshape(2, 7, 3, 3072)
    for i in range(2):
        for lvl in range(7):
            d = sdiff(glwe_phase(ggsw[i, lvl].reshape(3, 3072), keyset.glwe_sk), glwe_phase(want[i, lvl], keyset.glwe_sk))
            assert log2max(d) < 51.5, (i, lvl, log2max(d))


def test_lut8_matches_oracle(ctx, orc, orc_keys, keyset, trans_key):
    import ref_io
    k10_9, k8_1, k0 = trans_key
    value = 0xA7
    bits = np.array([(value >> i) & 1 for i in range(8)], dtype=np.uint8)  # LSB first
    small = keyset.encrypt_bits_small(bits, 16)
    ggsw = ctx.circuit_bootstrap_lwe_ciphertext_by_trace_with_preprocessing(small)
    luts = np.stack([k8_1[3, m, 5] for m in range(4)])  # round 4, byte 5, 4 multiples
    got = ctx.evaluate_8_to_8_cipher_lut(ggsw[None], luts[None])[0]  # [4][8][2049]
    gf = orc.ggsw_to_fourier(ggsw)
    for m in range(4):
        want = orc.lut8_eval(gf, luts[m])
        assert log2max(sdiff(got[m], want)) < 52
        ph = ref_io.lwe_phase(got[m], keyset.glwe_sk)
        dec = ref_io.decode_bit(ph)
        table_bits = [int(luts[m][a, 2048 + 256 * t + value] >> np.uint64(63)) for a in range(2) for t in range(4)]
        assert dec.tolist() == table_bits
        assert log2max(ref_io.bit_error(ph, dec)) < 60.5


def test_first_rounds_bit_exact(ctx, orc, trans_key):
    k10_9, _, _ = trans_key
    ct = bytes(np.random.default_rng(8).integers(0, 256, 32, dtype=np.uint8))
    got = ctx.aes_first_rounds(ct, k10_9)
    for blk in range(2):
        c = ct[16 * blk:16 * blk + 16]
        c2 = bytes(c[4 * ((col - row) % 4) + row] for col in range(4) for row in range(4))
        t = [orc.known_rotate(c2, k10_9[m]) for m in range(4)]
        want = orc.inv_shift_rows(orc.inv_mix_columns_precomp(*t))
        assert (got[blk] == want).all()


def test_inv_linear_bit_exact(ctx, orc):
    t4 = np.random.default_rng(9).integers(0, 2 ** 64, (4, 3, 128, 2049), dtype=np.uint64)
    got = ctx.he_inv_mix_columns_and_shift_rows(t4)
    for blk in range(3):
        want = orc.inv_shift_rows(orc.inv_mix_columns_precomp(t4[0, blk], t4[1, blk], t4[2, blk], t4[3, blk]))
        assert (got[blk] == want).all()


def test_aes_transcipher_two_blocks(ctx, orc, orc_keys, keyset, aes_key, trans_key):
    import aes_clear
    import ref_io
    pt = bytes(np.random.default_rng(10).integers(0, 256, 32, dtype=np.uint8))
    ct = aes_clear.ecb_encrypt(aes_key, pt)
    got = ctx.aes_to_lwe_transciphering(ct, *trans_key)
    bits, std, mx = ref_io.noise_stats(got.reshape(-1, 2049), keyset.glwe_sk)
    assert np.packbits(bits).tobytes() == pt
    # reference measured 2^57.9-2^58.2 std / <= 2^60.1 max on this stage (BASELINE.md); tolerance +0.3 bit
    assert std < 58.5 and mx < 61.0, (std, mx)
    want = orc.aes128_transcipher(orc_keys, ct[:16], *trans_key)
    obits, ostd, omx = ref_io.noise_stats(want[0], keyset.glwe_sk)
    assert (obits == bits[:128]).all()
    assert abs(std - ostd) < 0.5


def test_aes_transcipher_medium_instance_size(ctx, keyset, aes_key, trans_key):
    """BASELINE.json configs[2] at its full size on one GPU: 64 blocks = 8192 bit-ciphertexts per round (one chunk, two
    lanes, throughput blind-rotation kernel).  Size-independent checks: bit-exact decryption of all 8192 output bits
    against the cleartext and the output-noise tolerance of the reference (+0.3 bit)."""
    import aes_clear
    import ref_io
    pt = bytes(np.random.default_rng(64).integers(0, 256, 16 * 64, dtype=np.uint8))
    ct = aes_clear.ecb_encrypt(aes_key, pt)
    got = ctx.aes_to_lwe_transciphering(ct, *trans_key)
    bits, std, mx = ref_io.noise_stats(got.reshape(-1, 2049), keyset.glwe_sk)
    assert np.packbits(bits).tobytes() == pt
    assert std < 58.5 and mx < 61.5, (std, mx)


def test_aes_ctr_transcipher(ctx, orc, orc_keys, keyset, aes_key):
    """CTR mode (harness sizes 1/2): forward AES of the public counters xor the ciphertext."""
    import aes_clear
    import ref_io
    iv = bytes([0xFF] * 15 + [0xFE])  # exercises the 128-bit big-endian carry on the 3rd block
    pt = bytes(np.random.default_rng(12).integers(0, 256, 48, dtype=np.uint8))
    ct = aes_clear.ctr_crypt(aes_key, iv, pt)
    kf = keyset.gen_forward_transciphering_keys(aes_key, 55)
    got = ctx.aes_ctr_to_lwe_transciphering(ct, iv, *kf)
    bits, std, mx = ref_io.noise_stats(got.reshape(-1, 2049), keyset.glwe_sk)
    assert np.packbits(bits).tobytes() == pt
    assert std < 58.5 and mx < 61.0, (std, mx)
    want = orc.aes128_ctr_transcipher(orc_keys, ct[:16], iv, *kf)
    obits, ostd, _ = ref_io.noise_stats(want[0], keyset.glwe_sk)
    assert (obits == bits[:128]).all() and abs(std - ostd) < 0.5


def test_max_u16(ctx, keyset):
    import ref_io
    vals = [20962, 11749, 64797, 2177, 19876, 44457, 4094, 20862]
    bits = np.array([(v >> (15 - i)) & 1 for v in vals for i in range(16)], dtype=np.uint8)
    lwe = keyset.encrypt_bits_big(bits, 17)
    got = ctx.max_u16(lwe)
    dec, std, mx = ref_io.noise_stats(got, keyset.glwe_sk)
    assert ref_io.bits_to_u16(dec) == [max(vals)]
    assert mx < 61.5
    # above the reference's 8 values cbs_max_u16 runs the LUT circuit (csrc/host/ip_plan.h max_make_plan): odd counts
    # exercise the carried value, near-equal values the case where the CMux ladder's noise is largest (2^60.2)
    for n in (33, 200):
        vals = np.random.default_rng(n).integers(0, 65536, n).tolist()
        vals[3] = max(vals) ^ 1  # a close runner-up
        bits = np.array([(v >> (15 - i)) & 1 for v in vals for i in range(16)], dtype=np.uint8)
        got = ctx.max_u16(keyset.encrypt_bits_big(bits, n))
        dec, std, mx = ref_io.noise_stats(got, keyset.glwe_sk)
        assert ref_io.bits_to_u16(dec) == [max(vals)], n
        assert mx < 60.5, (n, std, mx)
    # both variants on the same 8 values
    vals = [513, 512, 65535, 65534, 7, 7, 40000, 1]
    bits = np.array([(v >> (15 - i)) & 1 for v in vals for i in range(16)], dtype=np.uint8)
    lwe = keyset.encrypt_bits_big(bits, 9)
    for fn in (ctx.max_u16, ctx.max_u16_lut):
        dec, std, mx = ref_io.noise_stats(fn(lwe), keyset.glwe_sk)
        assert ref_io.bits_to_u16(dec) == [65535]


def test_inner_product_u16(ctx, keyset):
    """mini-workload #2: decrypted result bit-exact against harness/cleartext_impl.py:65-70 (toy = 8 values)."""
    import ref_io
    for seed, n in ((1, 8), (2, 2), (3, 20)):
        vals = np.random.default_rng(seed).integers(0, 65536, n).tolist()
        if seed == 2:
            vals = [65535, 65535]
        bits = np.array([(v >> (15 - i)) & 1 for v in vals for i in range(16)], dtype=np.uint8)
        lwe = keyset.encrypt_bits_big(bits, 40 + seed)
        got = ctx.inner_product_u16(lwe)
        dec, std, mx = ref_io.noise_stats(got, keyset.glwe_sk)
        want = sum((x * y) % 65536 for x, y in zip(vals[: n // 2], vals[n // 2:])) % 65536
        assert ref_io.bits_to_u16(dec) == [want], (n, vals)
        assert mx < 61.5


def test_sum_u16_and_sharded_inner_product(ctx, keyset):
    """cbs_sum_u16 (the combine step of the multi-GPU inner product) and the shard -> partial -> sum route on one GPU."""
    import ref_io
    from temp_fhe_transciphering_b200 import sharding
    vals = np.random.default_rng(77).integers(0, 65536, 20).tolist()
    bits = np.array([(v >> (15 - i)) & 1 for v in vals for i in range(16)], dtype=np.uint8)
    lwe = keyset.encrypt_bits_big(bits, 78)
    dec = ref_io.decode_bit(ref_io.lwe_phase(ctx.sum_u16(lwe[:5 * 16]), keyset.glwe_sk))
    assert ref_io.bits_to_u16(dec) == [sum(vals[:5]) % 65536]
    parts = [ctx.inner_product_u16(sharding.shard_inner_product_values(lwe, r, 3)) for r in range(3)]
    dec = ref_io.decode_bit(ref_io.lwe_phase(ctx.sum_u16(np.concatenate(parts)), keyset.glwe_sk))
    assert ref_io.bits_to_u16(dec) == [sum((x * y) % 65536 for x, y in zip(vals[:10], vals[10:])) % 65536]


def test_max_u16_against_oracle_max_of_two(ctx, orc, orc_keys, keyset):
    """a10 parity (VERDICT r01): the CUDA max beside the oracle's restatement of the reference's stage 8
    (oracle.max_u16 = server_encrypted_compute.rs:34-98,213-350, pinned against the reference binary in
    tests/golden/reference_pin.json A).  The CUDA path changes the algorithm on purpose (balanced tree, operands refreshed
    from the level-1 GLEV, e reset per output bit: DESIGN.md 4a), so ciphertexts differ; what must agree is the
    decryption and the output noise: over 3 x 16 output bits log2 std(GPU) <= log2 std(oracle) + 0.75 bit and at most 2^59.4
    (the reference's worst measured stage-8 run, 2^59.1, + 0.3 bit).  The bound is one-sided because the refreshed operands
    make the CUDA ladder QUIETER than the reference's (measured on B200: 2^58.3 against the oracle's 2^59.2 on these
    inputs; the reference binary itself: 2^58.1 - 2^59.1); the floor is one LUT-ladder output, 2^56."""
    import ref_io
    sets = ([20962, 11749, 64797, 2177, 19876, 44457, 4094, 20862],  # the values of golden pin A
            [513, 512, 65535, 65534, 7, 9, 40000, 1],
            np.random.default_rng(8).integers(0, 65536, 8).tolist())
    g_err, o_err = [], []
    for k, vals in enumerate(sets):
        bits = np.array([(v >> (15 - i)) & 1 for v in vals for i in range(16)], dtype=np.uint8)
        lwe = keyset.encrypt_bits_big(bits, 170 + k)
        got = ctx.max_u16(lwe)
        want = orc.max_u16(orc_keys, lwe)
        gd = ref_io.decode_bit(ref_io.lwe_phase(got, keyset.glwe_sk))
        od = ref_io.decode_bit(ref_io.lwe_phase(want, keyset.glwe_sk))
        assert ref_io.bits_to_u16(gd) == ref_io.bits_to_u16(od) == [max(vals)], vals
        g_err.append(ref_io.bit_error(ref_io.lwe_phase(got, keyset.glwe_sk), gd))
        o_err.append(ref_io.bit_error(ref_io.lwe_phase(want, keyset.glwe_sk), od))
    g = np.log2(np.sqrt(np.mean(np.concatenate(g_err) ** 2)))
    o = np.log2(np.sqrt(np.mean(np.concatenate(o_err) ** 2)))
    assert g <= o + 0.75, (g, o)
    assert 56.0 < g <= 59.4, g
    assert 57.0 < o <= 59.6, o  # the oracle itself stays where the reference binary was measured


def test_golden_pin_b_on_gpu(cbs):
    """Golden pin B (oracle/pin_against_reference.py): the UNMODIFIED reference stage-7 binary was run on inputs that are a
    pure function of two seeds; its decrypted bytes and per-bit phase errors are committed in
    tests/golden/reference_pin.json.  Regenerate the same inputs here, run cbs_aes128_transcipher on them and compare
    with what the reference produced: same bytes, output noise std at most 0.5 bit above the reference's (and not more than
    1 bit below: 128 samples, and the CUDA path's FP64 transforms are a little quieter than concrete-fft's), worst bit
    within 1 bit."""
    import json
    import os
    import aes_clear
    import ref_io
    from conftest import ROOT
    pin = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_pin.json")))["B_seeded_keys"]
    ks = cbs.KeySet.generate(pin["seed_keys"])
    chk = int(np.bitwise_xor.reduce(ks.bsk.reshape(-1))) ^ int(np.bitwise_xor.reduce(ks.auto_std.reshape(-1)))
    assert chk == pin["keyset_checksum"]  # same key material the reference binary was given
    aes_key = bytes.fromhex(pin["aes_key_hex"])
    tk = ks.gen_transciphering_keys(aes_key, pin["seed_trans_key"])
    ct = bytes.fromhex(pin["ciphertext_hex"])
    c = cbs.Context(ks, 0)
    try:
        got = c.aes_to_lwe_transciphering(ct, *tk).reshape(-1, 2049)
    finally:
        c.close()
    bits, std, mx = ref_io.noise_stats(got, ks.glwe_sk)
    ref = pin["reference_stage7"]
    assert np.packbits(bits).tobytes().hex() == ref["bytes_hex"] == pin["plaintext_hex"]
    assert ref["noise_log2_std"] - 1.0 < std < ref["noise_log2_std"] + 0.5, (std, ref["noise_log2_std"])
    assert mx < ref["noise_log2_max"] + 1.0, (mx, ref["noise_log2_max"])
    # the reference's own per-bit errors: same scale, no bit of ours further out than the reference's worst by 2x
    ref_err = np.array(ref["phase_error_int64"], dtype=np.float64)
    assert abs(np.log2(np.sqrt(np.mean(ref_err ** 2))) - ref["noise_log2_std"]) < 0.01
    err = ref_io.bit_error(ref_io.lwe_phase(got, ks.glwe_sk), bits).astype(np.float64)
    assert np.abs(err).max() < 2.0 * np.abs(ref_err).max()


def _check_non_trivial_luts(keyset, gen, key, run, pt):
    """Adds a GLWE encryption of zero (difference of two encryptions of the same first-round table, from `gen` with another
    seed) to one middle-round accumulator of every round of `key`; run(key) must still decrypt to pt."""
    import ref_io
    first, mid, last = key
    other = gen(424242)[0]
    if (other == first).all():  # same seed as the key: take another one
        other = gen(424243)[0]
    zero = (first[0, 0, 0].astype(np.uint64) - other[0, 0, 0].astype(np.uint64))
    assert zero[:2048].any()
    mid = mid.copy()
    with np.errstate(over="ignore"):
        for r in range(8):
            mid[r, 0, 0, 0] = mid[r, 0, 0, 0] + zero
    assert mid[0, 0, 0, 0, :2048].any()
    got = run((first, mid, last))
    bits, std, mx = ref_io.noise_stats(got.reshape(-1, 2049), keyset.glwe_sk)
    assert np.packbits(bits).tobytes() == pt
    assert std < 58.6 and mx < 61.2, (std, mx)
    # and back to the trivial LUTs of the key (later tests share the context)
    got = run(key)
    bits, _, _ = ref_io.noise_stats(got.reshape(-1, 2049), keyset.glwe_sk)
    assert np.packbits(bits).tobytes() == pt


def test_aes_transcipher_with_non_trivial_luts(ctx, keyset, aes_key, trans_key):
    """The reference always writes the round 8..0 LUTs as trivial GLWE (zero masks, data_struct.rs:145-151) and the ladder
    skips the mask transforms of its first CMux when the device-side check (k_masks_nonzero) says so.  Here one accumulator
    gets a real mask: a GLWE encryption of zero (difference of two encryptions of the same table) is added to it, which
    leaves every decryption unchanged - provided the check notices and the full first CMux runs."""
    import aes_clear
    pt = bytes(np.random.default_rng(11).integers(0, 256, 16, dtype=np.uint8))
    ct = aes_clear.ecb_encrypt(aes_key, pt)
    _check_non_trivial_luts(keyset, lambda seed: keyset.gen_transciphering_keys(aes_key, seed), trans_key,
                            lambda k: ctx.aes_to_lwe_transciphering(ct, *k), pt)


def test_aes_ctr_transcipher_with_non_trivial_luts(ctx, keyset, aes_key):
    """The same for CTR mode, whose forward LUTs have their own device-side mask flag."""
    import aes_clear
    pt = bytes(np.random.default_rng(11).integers(0, 256, 16, dtype=np.uint8))
    iv = bytes(range(16))
    ct = aes_clear.ctr_crypt(aes_key, iv, pt)
    _check_non_trivial_luts(keyset, lambda seed: keyset.gen_forward_transciphering_keys(aes_key, seed),
                            keyset.gen_forward_transciphering_keys(aes_key, 55),
                            lambda k: ctx.aes_ctr_to_lwe_transciphering(ct, iv, *k), pt)
