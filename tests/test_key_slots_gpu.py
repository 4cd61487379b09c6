"""Key slots on the GPU: many transciphering keys resident at once, one call over blocks of many keys
(cbs_*trans_key_slots_reserve, cbs_*trans_key_*slot_upload, cbs_aes128_*transcipher_slots{,_dev}).

The workers pin the blind-rotation kernel with CBS_BR_LOWLAT=0 (read once per process), as test_partitions_gpu.py does, so
the comparisons do not depend on which kernel a part size selects by default.  Three AES keys, slots 0 and
2 seeded and slot 1 in the reference format (trivial middle and last LUTs), over 11 blocks with interleaved slots, so both lanes
mix keys and a part that holds the reference-format key runs the full first CMux on its trivial LUTs.  Every block must equal,
bit for bit, that key's blocks transciphered alone through the single-key upload and decrypt to its own key's plaintext."""
import ctypes
import hashlib
import os
import traceback

import numpy as np
import pytest

from conftest import NoiseFailure, retry_on_noise
from test_partitions_gpu import _counters, _run_worker, _setup_worker

pytestmark = pytest.mark.gpu

LWE = 2049
SLOTS = [2, 0, 1, 1, 0, 2, 2, 1, 0, 0, 2]
SPLITS = [(64, 2), (3, 2), (1, 1), (2, 3), (4, 4)]  # (CBS_CHUNK_BLOCKS, CBS_LANES)
SEEDED = (True, False, True)  # key form of slots 0, 1, 2
IVS = [bytes([0x10 * s] * 15 + [0xFE]) for s in range(3)]  # slot 0's counter carries through all 128 bits


def _digests(rows):
    rows = np.ascontiguousarray(rows).view(np.uint64).reshape(-1, 128 * LWE)
    return [hashlib.sha256(b.tobytes()).hexdigest() for b in rows]


def _batch(aes_keys, slots, seed):
    """public inputs of a batch whose block b is under key slots[b]: (ECB ciphertext, CTR counters, CTR ciphertext, plaintext),
    each sender's CTR blocks counting up from its own IV in the order they appear"""
    import aes_clear
    pt = bytes(np.random.default_rng(seed).integers(0, 256, 16 * len(slots), dtype=np.uint8))
    ecb, ctr, ct = bytearray(), bytearray(), bytearray()
    seen = [0, 0, 0]
    for b, s in enumerate(slots):
        blk = pt[16 * b:16 * b + 16]
        ecb += aes_clear.ecb_encrypt(aes_keys[s], blk)
        c = _counters(IVS[s], seen[s] + 1)[-16:]
        ctr += c
        ct += aes_clear.ctr_crypt(aes_keys[s], c, blk)
        seen[s] += 1
    return bytes(ecb), bytes(ctr), bytes(ct), pt


class _Keys:
    """three AES keys and their transciphering keys in both directions (slots 0 and 2 seeded, slot 1 reference format)"""

    def __init__(self, cbs, ks, attempt):
        import aes_clear
        self.aes = [aes_clear.harness_aes_key(f"sender-{s}") for s in range(3)]
        self.forms = {}
        for mode in ("ecb", "ctr"):
            for s in range(3):
                self.forms[mode, s] = self.make(ks, mode, s, 100 * attempt + 10 * s)

    def make(self, ks, mode, s, seed, aes_key=None):
        aes_key = aes_key or self.aes[s]
        if SEEDED[s]:
            gen = ks.gen_seeded_transciphering_keys if mode == "ecb" else ks.gen_seeded_forward_transciphering_keys
            return "seeded", gen(aes_key, 5000 + seed)
        gen = ks.gen_transciphering_keys if mode == "ecb" else ks.gen_forward_transciphering_keys
        return "full", gen(aes_key, 6000 + seed)


def _upload_single(ctx, mode, form):
    kind, arrays = form
    if kind == "seeded":
        (ctx.upload_seeded_trans_key if mode == "ecb" else ctx.upload_seeded_fwd_trans_key)(*arrays)
    else:
        (ctx.upload_trans_key if mode == "ecb" else ctx.upload_fwd_trans_key)(*arrays)


def _upload_slot(ctx, mode, slot, form):
    kind, arrays = form
    if kind == "seeded":
        (ctx.upload_seeded_trans_key_slot if mode == "ecb" else ctx.upload_seeded_fwd_trans_key_slot)(slot, *arrays)
    else:
        (ctx.upload_trans_key_slot if mode == "ecb" else ctx.upload_fwd_trans_key_slot)(slot, *arrays)


def _dev(ctx, mode, batch, slots=None):
    """the _dev call (single key if slots is None) on device copies of the batch's inputs -> host rows"""
    import torch
    ecb, ctr, ct, _ = batch
    nb = len(ecb) // 16
    t = lambda b: torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()  # noqa: E731
    d_out = torch.zeros((nb, 128, LWE), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    if mode == "ecb":
        d_ct = t(ecb)
        if slots is None:
            ctx.transcipher_dev(d_ct.data_ptr(), nb, d_out.data_ptr())
        else:
            ctx.transcipher_slots_dev(d_ct.data_ptr(), slots, nb, d_out.data_ptr())
    else:
        d_ctr, d_ct = t(ctr), t(ct)
        if slots is None:
            ctx.ctr_transcipher_dev(d_ctr.data_ptr(), d_ct.data_ptr(), nb, d_out.data_ptr())
        else:
            ctx.ctr_transcipher_slots_dev(d_ctr.data_ptr(), d_ct.data_ptr(), slots, nb, d_out.data_ptr())
    ctx.synchronize()
    return d_out.cpu().numpy().view(np.uint64)


def _sub(batch, blocks):
    return tuple(b"".join(x[16 * i:16 * i + 16] for i in blocks) for x in batch)


def _context(cbs, ks, chunk=64, lanes=2):
    os.environ["CBS_CHUNK_BLOCKS"], os.environ["CBS_LANES"] = str(chunk), str(lanes)
    return cbs.Context(ks, 0)


def _slots_worker(q, attempt=0):
    try:
        _setup_worker(0)
        import ref_io
        import temp_fhe_transciphering_b200 as cbs
        ks = cbs.KeySet.generate(20261018 + attempt)
        keys = _Keys(cbs, ks, attempt)
        batch = _batch(keys.aes, SLOTS, 77 + attempt)
        res = {"pt": batch[3]}
        for mode in ("ecb", "ctr"):
            c = _context(cbs, ks)
            # each key's blocks alone under the single key, then the mixed batch under the slots (dev and host calls)
            for s in range(3):
                blocks = [b for b, x in enumerate(SLOTS) if x == s]
                _upload_single(c, mode, keys.forms[mode, s])
                res[mode, "alone", s] = _digests(_dev(c, mode, _sub(batch, blocks)))
            c.reserve_trans_key_slots(3) if mode == "ecb" else c.reserve_fwd_trans_key_slots(3)
            for s in range(3):
                _upload_slot(c, mode, s, keys.forms[mode, s])
            rows = _dev(c, mode, batch, SLOTS)
            res[mode, "slots"] = _digests(rows)
            bits = ref_io.decode_bit(ref_io.lwe_phase(rows.reshape(-1, LWE), ks.glwe_sk))
            res[mode, "bytes"] = np.packbits(bits).tobytes()
            ecb, ctr, ct, _ = batch
            host = c.transcipher_slots(ecb, SLOTS) if mode == "ecb" else c.ctr_transcipher_slots(ctr, ct, SLOTS)
            res[mode, "host"] = _digests(host)
            # slot calls and uploads leave the single key alone, and the other way round
            sub2 = _sub(batch, [b for b, x in enumerate(SLOTS) if x == 2])
            res[mode, "single_after_slots"] = _digests(_dev(c, mode, sub2))
            _upload_single(c, mode, keys.forms[mode, 0])
            _dev(c, mode, _sub(batch, [0, 1]))
            res[mode, "slots_after_single"] = _digests(_dev(c, mode, batch, SLOTS))
            # one slot for every block, one block and 65 (a second chunk)
            for nb in (1, 65):
                big = _batch(keys.aes, [2] * nb, 300 + nb)
                _upload_single(c, mode, keys.forms[mode, 2])
                res[mode, "one_slot", nb] = (_digests(_dev(c, mode, big)), _digests(_dev(c, mode, big, [2] * nb)))
            c.close()
            # the mixed batch under every chunk and lane split, fresh contexts
            for split in SPLITS[1:]:
                c = _context(cbs, ks, *split)
                c.reserve_trans_key_slots(3) if mode == "ecb" else c.reserve_fwd_trans_key_slots(3)
                for s in range(3):
                    _upload_slot(c, mode, s, keys.forms[mode, s])
                res[mode, "split", split] = _digests(_dev(c, mode, batch, SLOTS))
                c.close()
            # growing the pool keeps the slots; a new key in slot 0 gives that key's single-key rows
            c = _context(cbs, ks)
            grow = [0, 1, 1, 0]
            gb = _batch(keys.aes, grow, 400)
            c.reserve_trans_key_slots(2) if mode == "ecb" else c.reserve_fwd_trans_key_slots(2)
            for s in range(2):
                _upload_slot(c, mode, s, keys.forms[mode, s])
            res[mode, "grow", 2] = _digests(_dev(c, mode, gb, grow))
            c.reserve_trans_key_slots(5) if mode == "ecb" else c.reserve_fwd_trans_key_slots(5)
            res[mode, "grow", 5] = _digests(_dev(c, mode, gb, grow))
            new_key = keys.make(ks, mode, 0, 900 + attempt, aes_key=keys.aes[2])  # seeded, AES key of sender 2
            _upload_slot(c, mode, 0, new_key)
            nb3 = _batch(keys.aes, [2, 2, 2], 401)
            res[mode, "replaced"] = _digests(_dev(c, mode, nb3, [0, 0, 0]))
            _upload_single(c, mode, new_key)
            res[mode, "replaced_single"] = _digests(_dev(c, mode, nb3))
            c.close()
        q.put(("ok", res))
    except BaseException:
        q.put(("error", traceback.format_exc()))
        raise


def _worker_attempt(attempt):
    import functools
    return _run_worker(functools.partial(_slots_worker, attempt=attempt))


@pytest.fixture(scope="module")
def slots_run():
    return _worker_attempt(0)


@pytest.mark.parametrize("mode", ["ecb", "ctr"])
def test_mixed_keys_equal_each_key_alone(slots_run, mode):
    alone = [iter(slots_run[mode, "alone", s]) for s in range(3)]
    want = [next(alone[s]) for s in SLOTS]
    got = slots_run[mode, "slots"]
    bad = [b for b in range(len(SLOTS)) if got[b] != want[b]]
    assert not bad, f"{mode}: blocks {bad} (slots {[SLOTS[b] for b in bad]}) differ from their key alone"
    assert slots_run[mode, "host"] == got, "host-buffer call differs from the _dev call"


@pytest.mark.parametrize("mode", ["ecb", "ctr"])
def test_mixed_keys_decrypt_to_each_senders_plaintext(slots_run, mode):
    def run(attempt):
        r = slots_run if attempt == 0 else _worker_attempt(attempt)
        got, pt = r[mode, "bytes"], r["pt"]
        bad = [b for b in range(len(SLOTS)) if got[16 * b:16 * b + 16] != pt[16 * b:16 * b + 16]]
        if bad and len(bad) <= 2:
            raise NoiseFailure(f"{mode}: blocks {bad} decrypt wrongly")
        assert not bad, f"{mode}: blocks {bad} of {len(SLOTS)} wrong"

    retry_on_noise(run)


@pytest.mark.parametrize("mode", ["ecb", "ctr"])
def test_mixed_keys_every_chunk_and_lane_split(slots_run, mode):
    """one chunk of two lanes (5 + 6 blocks), chunks of 3 (1 + 2 lanes), one block per chunk, chunks of 2 over three lanes,
    chunks of 4 over four lanes: every block bit-identical"""
    base = slots_run[mode, "slots"]
    for split in SPLITS[1:]:
        got = slots_run[mode, "split", split]
        bad = [b for b in range(len(SLOTS)) if got[b] != base[b]]
        assert not bad, f"{mode} {split}: blocks {bad} differ"


@pytest.mark.parametrize("nb", [1, 65])
@pytest.mark.parametrize("mode", ["ecb", "ctr"])
def test_one_slot_for_every_block_equals_single_key(slots_run, mode, nb):
    single, slots = slots_run[mode, "one_slot", nb]
    assert single == slots, [b for b in range(nb) if single[b] != slots[b]]


@pytest.mark.parametrize("mode", ["ecb", "ctr"])
def test_growing_the_pool_keeps_slots_and_replacing_a_slot(slots_run, mode):
    assert slots_run[mode, "grow", 2] == slots_run[mode, "grow", 5]
    assert slots_run[mode, "replaced"] == slots_run[mode, "replaced_single"]


@pytest.mark.parametrize("mode", ["ecb", "ctr"])
def test_slots_and_single_key_are_independent(slots_run, mode):
    assert slots_run[mode, "single_after_slots"] == slots_run[mode, "alone", 2]
    assert slots_run[mode, "slots_after_single"] == slots_run[mode, "slots"]


def test_argument_errors_queue_nothing(cbs, keyset):
    import torch
    L = cbs.lib()
    c = cbs.Context(keyset, 0)
    try:
        h = c._h
        u64 = lambda n: np.zeros(n, dtype=np.uint64)  # noqa: E731
        inv = [u64(cbs.K10_9_WORDS), u64(cbs.K8_1_WORDS), u64(cbs.K0_WORDS)]
        fwd = [u64(cbs.KF_FIRST_WORDS), u64(cbs.KF_MID_WORDS), u64(cbs.KF_LAST_WORDS)]
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
        seed = (ctypes.c_uint8 * 32)()
        bodies = u64(cbs.TRANS_KEY_SEEDED_GLWES * 1024)
        fbodies = u64(cbs.FWD_TRANS_KEY_SEEDED_GLWES * 1024)
        n0 = c.launch_count
        # uploads before any reserve
        assert L.cbs_trans_key_slot_upload(h, 0, *map(p, inv)) == 1
        assert L.cbs_fwd_trans_key_slot_upload(h, 0, *map(p, fwd)) == 1
        assert L.cbs_trans_key_seeded_slot_upload(h, 0, seed, p(bodies)) == 1
        assert L.cbs_fwd_trans_key_seeded_slot_upload(h, 0, seed, p(fbodies)) == 1
        for fn in (L.cbs_trans_key_slots_reserve, L.cbs_fwd_trans_key_slots_reserve):
            assert fn(h, 0) == 1 and fn(h, -1) == 1
            assert fn(h, 3) == 0
            assert fn(h, 2) == 1  # a pool only grows
            assert fn(h, 3) == 0
            assert fn(None, 4) == 1
        assert c.launch_count == n0
        c.upload_trans_key_slot(0, *inv)       # inverse: slot 0 only
        c.upload_fwd_trans_key_slot(2, *fwd)   # forward: slot 2 only
        n1 = c.launch_count
        for bad_slot in (-1, 3, 7):
            assert L.cbs_trans_key_slot_upload(h, bad_slot, *map(p, inv)) == 1
            assert L.cbs_trans_key_seeded_slot_upload(h, bad_slot, seed, p(bodies)) == 1
            assert L.cbs_fwd_trans_key_slot_upload(h, bad_slot, *map(p, fwd)) == 1
            assert L.cbs_fwd_trans_key_seeded_slot_upload(h, bad_slot, seed, p(fbodies)) == 1
        assert L.cbs_trans_key_slot_upload(h, 1, None, p(inv[1]), p(inv[2])) == 1
        assert L.cbs_trans_key_seeded_slot_upload(h, 1, None, p(bodies)) == 1
        assert L.cbs_fwd_trans_key_seeded_slot_upload(h, 1, seed, None) == 1

        d_in = torch.zeros(16 * 2, dtype=torch.uint8, device="cuda")
        d_ct = torch.zeros(16 * 2, dtype=torch.uint8, device="cuda")
        d_out = torch.zeros((2, 128, LWE), dtype=torch.int64, device="cuda")
        hin, hct, hout = np.zeros(32, np.uint8), np.zeros(32, np.uint8), u64(2 * 128 * LWE)
        P = ctypes.c_void_p

        def ecb_dev(sl, nb=None, a=P(d_in.data_ptr()), o=P(d_out.data_ptr())):
            s = np.asarray(sl, dtype=np.int32)
            return L.cbs_aes128_transcipher_slots_dev(h, a, p(s) if s.size else None, len(s) if nb is None else nb, o)

        def ctr_dev(sl, nb=None):
            s = np.asarray(sl, dtype=np.int32)
            return L.cbs_aes128_ctr_transcipher_slots_dev(h, P(d_in.data_ptr()), P(d_ct.data_ptr()), p(s) if s.size else None,
                                                          len(s) if nb is None else nb, P(d_out.data_ptr()))

        def ecb_host(sl):
            s = np.asarray(sl, dtype=np.int32)
            return L.cbs_aes128_transcipher_slots(h, p(hct), p(s), len(s), p(hout))

        def ctr_host(sl):
            s = np.asarray(sl, dtype=np.int32)
            return L.cbs_aes128_ctr_transcipher_slots(h, p(hin), p(hct), p(s), len(s), p(hout))

        # negative, >= reserved, reserved but never uploaded, uploaded only in the other direction; a good slot first
        for sl in ([0, -1], [0, 3], [0, 1], [0, 2]):
            assert ecb_dev(sl) == 1 and ecb_host(sl) == 1, sl
        for sl in ([2, -1], [2, 3], [2, 1], [2, 0]):
            assert ctr_dev(sl) == 1 and ctr_host(sl) == 1, sl
        assert ecb_dev([0], nb=0) == 1 and ecb_dev([0], nb=-1) == 1
        assert ctr_dev([2], nb=0) == 1
        assert ecb_dev([], nb=1) == 1 and ctr_dev([], nb=1) == 1  # null slot array
        assert ecb_dev([0], a=None) == 1 and ecb_dev([0], o=None) == 1
        assert L.cbs_aes128_ctr_transcipher_slots_dev(h, None, P(d_ct.data_ptr()), p(np.zeros(1, np.int32)), 1,
                                                      P(d_out.data_ptr())) == 1
        assert L.cbs_aes128_transcipher_slots(h, None, p(np.zeros(1, np.int32)), 1, p(hout)) == 1
        assert L.cbs_aes128_ctr_transcipher_slots(h, p(hin), p(hct), p(np.full(1, 2, np.int32)), 1, None) == 1
        assert L.cbs_aes128_transcipher_slots_dev(None, P(d_in.data_ptr()), p(np.zeros(1, np.int32)), 1,
                                                  P(d_out.data_ptr())) == 1
        assert c.launch_count == n1, (n1, c.launch_count)
        c.synchronize()
    finally:
        c.close()
