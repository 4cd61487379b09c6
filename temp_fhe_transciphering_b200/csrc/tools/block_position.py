"""Development tool: does a CTR block that decrypts wrongly in bigcheck.py do so because of its inputs or because of where
it sits in the launch?  Rebuilds bigcheck.py's CTR inputs and transciphers one block three ways through
cbs_aes128_ctr_transcipher_dev: alone, at its own position in its 64-block chunk, and moved to the chunk's first slot
(swapped with the block there).  Prints, per way, the block's wrong bits, its worst phase error and an output digest.
Same bits in all three = the failure belongs to the inputs (AES_TIGHT noise); different = a position-dependent defect.
The blind-rotation mode is whatever CBS_BR_LOWLAT says (read once per process).
usage: block_position.py [blocks] [block] [seed]"""
import hashlib
import os
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", "..", ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np
import torch
import aes_clear
import ref_io
import temp_fhe_transciphering_b200 as cbs

nb = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
blk = int(sys.argv[2]) if len(sys.argv) > 2 else 510
seed = int(sys.argv[3]) if len(sys.argv) > 3 else 1
chunk = 64
ks = cbs.KeySet.generate(seed)
ctx = cbs.Context(ks, 0)
key = aes_clear.harness_aes_key(None)
pt = bytes(np.random.default_rng(seed).integers(0, 256, 16 * nb, dtype=np.uint8))  # as bigcheck.py
iv = aes_clear.harness_iv(None)
ct = aes_clear.ctr_crypt(key, iv, pt)
ctx.upload_fwd_trans_key(*ks.gen_forward_transciphering_keys(key, seed + 1))
ctr = [((int.from_bytes(iv, "big") + b) % (1 << 128)).to_bytes(16, "big") for b in range(nb)]


def run(order):
    """transcipher the blocks `order` (indices into the run) as one call -> [len(order)][128][2049]"""
    d_ctr = torch.frombuffer(bytearray(b"".join(ctr[b] for b in order)), dtype=torch.uint8).cuda()
    d_ct = torch.frombuffer(bytearray(b"".join(ct[16 * b:16 * b + 16] for b in order)), dtype=torch.uint8).cuda()
    d_out = torch.zeros((len(order), 128, 2049), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ctx.ctr_transcipher_dev(d_ctr.data_ptr(), d_ct.data_ptr(), len(order), d_out.data_ptr())
    ctx.synchronize()
    return d_out.cpu().numpy().view(np.uint64)


c0 = blk // chunk * chunk
home = list(range(c0, c0 + chunk))
moved = list(home)
moved[0], moved[blk - c0] = blk, c0
want = np.unpackbits(np.frombuffer(pt[16 * blk:16 * blk + 16], dtype=np.uint8))
print({"blocks": nb, "block": blk, "seed": seed, "CBS_BR_LOWLAT": os.environ.get("CBS_BR_LOWLAT", "1 (default)")})
digests = []
for name, order in (("alone", [blk]), (f"chunk {c0}..{c0 + chunk - 1}, slot {blk - c0}", home),
                    (f"chunk {c0}..{c0 + chunk - 1}, slot 0", moved)):
    out = run(order)[order.index(blk)]
    ph = ref_io.lwe_phase(out, ks.glwe_sk)
    bits = ref_io.decode_bit(ph)
    err = np.abs(ref_io.bit_error(ph, want))
    digests.append(hashlib.sha256(out.tobytes()).hexdigest()[:16])
    print({"way": name, "wrong_bits": int((bits != want).sum()), "wrong_bit_positions": np.flatnonzero(bits != want)[:12].tolist(),
           "log2_max_error": round(float(np.log2(err.max() + 1)), 3), "digest": digests[-1]})
print({"bit_identical_in_all_three": len(set(digests)) == 1})
ctx.close()
