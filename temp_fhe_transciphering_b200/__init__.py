"""temp_fhe_transciphering_b200 — host-side mirror of the reference's cbs_lib interface over
libcbs_b200.so (hand-written sm_100a kernels behind the C ABI of include/cbs_b200.h).

The function names and argument meaning follow the Rust functions they replace
(/root/reference/submission/cbs_lib/src/*.rs and the two server stage binaries); each wrapper
cites the function it mirrors.  All arrays are numpy uint64 in the flat layouts documented in
include/cbs_b200.h.  There is NO CPU fallback: importing works anywhere, but any compute call
raises CbsError when the shared library or a B200 is missing.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libcbs_b200.so")
_lib = None

LWE_SMALL = 769
LWE_BIG = 2049
GLWE_WORDS = 3072
GLEV_WORDS = 21504
GGSW_WORDS = 64512
BSK_WORDS = 768 * 9 * 1024
KSK_WORDS = 8 * 3 * 4 * 256
AUTO_WORDS = 10 * 2 * 3 * 3 * 1024
SS_WORDS = 2 * 2 * 3 * 3 * 1024
K10_9_WORDS = 4 * 16 * 2 * 3072
K8_1_WORDS = 8 * 4 * 16 * 2 * 3072
K0_WORDS = 16 * 2 * 3072
KF_FIRST_WORDS = 3 * 16 * 2 * 3072
KF_MID_WORDS = 8 * 3 * 16 * 2 * 3072
KF_LAST_WORDS = 16 * 2 * 3072
TRANS_KEY_SEEDED_GLWES = 1184  # seeded keys: one 1024-word body per LUT GLWE, AllRdKeys order (include/cbs_b200.h)
FWD_TRANS_KEY_SEEDED_GLWES = 896


class CbsError(RuntimeError):
    pass


def build(verbose=False):
    """Compile libcbs_b200.so and the stage executables in-tree for sm_100a (nvcc cross-compiles
    without a GPU)."""
    cmd = ["make", "-C", os.path.join(_HERE, "csrc"), "all"]
    if not verbose:
        cmd.insert(1, "-s")
    subprocess.check_call(cmd)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise CbsError(f"{_LIB_PATH} is missing: run __graft_entry__.build() (no CPU fallback exists)")
        L = ctypes.CDLL(_LIB_PATH)
        L.cbs_last_error.restype = ctypes.c_char_p
        L.cbs_version.restype = ctypes.c_char_p
        L.cbs_ctx_launch_count.restype = ctypes.c_uint64
        L.cbs_ctx_launch_count.argtypes = [ctypes.c_void_p]
        for name in ("cbs_keyset_bsk", "cbs_keyset_ksk", "cbs_keyset_auto", "cbs_keyset_ss",
                     "cbs_keyset_lwe_sk_small", "cbs_keyset_glwe_sk"):
            getattr(L, name).restype = ctypes.POINTER(ctypes.c_uint64)
            getattr(L, name).argtypes = [ctypes.c_void_p]
        _lib = L
    return _lib


def inner_product_plan_check(vals):
    """Host-only dry run of the inner-product circuit on cleartext u16 values -> (result, circuit bootstraps,
    layers, LUT ladders).  Checks the circuit plan, never touches the GPU."""
    v = np.ascontiguousarray(vals, dtype=np.uint16)
    res = ctypes.c_uint16()
    ncbs = ctypes.c_int64()
    layers = ctypes.c_int()
    ladders = ctypes.c_int64()
    _check(lib().cbs_inner_product_plan_check(v.ctypes.data_as(ctypes.c_void_p), int(v.size), ctypes.byref(res),
                                              ctypes.byref(ncbs), ctypes.byref(layers), ctypes.byref(ladders)),
           "cbs_inner_product_plan_check")
    return int(res.value), int(ncbs.value), int(layers.value), int(ladders.value)


def max_plan_check(vals):
    """Host-only dry run of the LUT-circuit maximum on cleartext u16 values -> (result, circuit bootstraps, layers, ladders)."""
    v = np.ascontiguousarray(vals, dtype=np.uint16)
    res = ctypes.c_uint16()
    ncbs = ctypes.c_int64()
    layers = ctypes.c_int()
    ladders = ctypes.c_int64()
    _check(lib().cbs_max_plan_check(v.ctypes.data_as(ctypes.c_void_p), int(v.size), ctypes.byref(res), ctypes.byref(ncbs),
                                    ctypes.byref(layers), ctypes.byref(ladders)), "cbs_max_plan_check")
    return int(res.value), int(ncbs.value), int(layers.value), int(ladders.value)


def _check(rc, what):
    if rc != 0:
        raise CbsError(f"{what} failed (code {rc}): {lib().cbs_last_error().decode()}")


def _u64(a):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a, a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64))


def _out(shape):
    a = np.zeros(shape, dtype=np.uint64)
    return a, a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64))


def _u8(b):
    a = np.frombuffer(bytes(b), dtype=np.uint8).copy()
    return a, a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))


def _i32(a):
    a = np.ascontiguousarray(a, dtype=np.int32).reshape(-1)
    return a, a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))


def _slots(slots, nblocks):
    a = np.ascontiguousarray(slots, dtype=np.int32).reshape(-1)
    if a.size != nblocks:
        raise ValueError(f"{a.size} slots for {nblocks} blocks")
    return a, a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))


class KeySet:
    """Host-side evaluation (and optionally secret) keys in the standard domain.

    Mirrors the tuple returned by generate_fhe_keys (src/bin/client_key_generation.rs:20-86) and the
    files it writes under io/<size>/{public_keys,secret_keys}/."""

    def __init__(self, handle):
        self._h = ctypes.c_void_p(handle)

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.cbs_keyset_free(self._h)
            self._h = None

    @classmethod
    def generate(cls, seed=None):
        """seed = None: ChaCha20 keyed by getrandom(2) (fresh keys, what the stage executable does without a seed);
        an integer: the deterministic, not cryptographically secure test generator."""
        h = ctypes.c_void_p()
        if seed is None:
            _check(lib().cbs_keyset_generate_os_entropy(ctypes.byref(h)), "cbs_keyset_generate_os_entropy")
        else:
            _check(lib().cbs_keyset_generate(ctypes.c_uint64(seed), ctypes.byref(h)), "cbs_keyset_generate")
        return cls(h.value)

    @classmethod
    def load_dir(cls, io_dir, with_secret=False):
        h = ctypes.c_void_p()
        _check(lib().cbs_keyset_load_dir(str(io_dir).encode(), int(with_secret), ctypes.byref(h)), "cbs_keyset_load_dir")
        return cls(h.value)

    @classmethod
    def from_arrays(cls, bsk, ksk, auto_std, ss, lwe_sk_small=None, glwe_sk=None):
        h = ctypes.c_void_p()
        keep = [_u64(x) for x in (bsk, ksk, auto_std, ss)]
        sk1 = _u64(lwe_sk_small) if lwe_sk_small is not None else (None, None)
        sk2 = _u64(glwe_sk) if glwe_sk is not None else (None, None)
        _check(lib().cbs_keyset_from_arrays(keep[0][1], keep[1][1], keep[2][1], keep[3][1], sk1[1], sk2[1],
                                            ctypes.byref(h)), "cbs_keyset_from_arrays")
        return cls(h.value)

    def save_dir(self, io_dir, with_secret=False):
        _check(lib().cbs_keyset_save_dir(self._h, str(io_dir).encode(), int(with_secret)), "cbs_keyset_save_dir")

    def _arr(self, fn, n, shape):
        p = getattr(lib(), fn)(self._h)
        if not p:
            return None
        return np.ctypeslib.as_array(p, shape=(n,)).reshape(shape).copy()

    @property
    def bsk(self):
        return self._arr("cbs_keyset_bsk", BSK_WORDS, (768, 1, 3, 3, 1024))

    @property
    def ksk(self):
        return self._arr("cbs_keyset_ksk", KSK_WORDS, (8, 3, 4, 256))

    @property
    def auto_std(self):
        return self._arr("cbs_keyset_auto", AUTO_WORDS, (10, 2, 3, 3, 1024))

    @property
    def ss(self):
        return self._arr("cbs_keyset_ss", SS_WORDS, (2, 2, 3, 3, 1024))

    @property
    def lwe_sk_small(self):
        return self._arr("cbs_keyset_lwe_sk_small", 768, (768,))

    @property
    def glwe_sk(self):
        return self._arr("cbs_keyset_glwe_sk", 2048, (2048,))

    # ---- client-side helpers (seeded; the reference's client binaries are unseeded) ----
    def gen_transciphering_keys(self, aes_key, seed):
        """gen_transciphering_keys, src/bin/client_encode_encrypt.rs:9-22 -> (k10_9, k8_1, k0)."""
        k10_9, p1 = _out((4, 16, 2, GLWE_WORDS))
        k8_1, p2 = _out((8, 4, 16, 2, GLWE_WORDS))
        k0, p3 = _out((16, 2, GLWE_WORDS))
        _, pk = _u8(aes_key)
        _check(lib().cbs_trans_key_generate(self._h, pk, ctypes.c_uint64(seed), p1, p2, p3), "cbs_trans_key_generate")
        return k10_9, k8_1, k0

    def gen_forward_transciphering_keys(self, aes_key, seed):
        """Forward-direction keyed-S-box LUTs for CTR mode (keyed tables cbs_lib/src/aes_ref.rs:334-380)
        -> (kf_first[3][16][2], kf_mid[8][3][16][2], kf_last[16][2]) GLWE."""
        a, p1 = _out((3, 16, 2, GLWE_WORDS))
        b, p2 = _out((8, 3, 16, 2, GLWE_WORDS))
        c, p3 = _out((16, 2, GLWE_WORDS))
        _, pk = _u8(aes_key)
        _check(lib().cbs_fwd_trans_key_generate(self._h, pk, ctypes.c_uint64(seed), p1, p2, p3), "cbs_fwd_trans_key_generate")
        return a, b, c

    def gen_seeded_transciphering_keys(self, aes_key, seed=None):
        """The transciphering key with EVERY LUT encrypted, in seeded form -> (mask_seed: 32 bytes, bodies [1184][1024]).
        gen_transciphering_keys writes rounds 8..0 as trivial LUTs whose bodies show the round keys; this one does not.
        seed = None: noise key and mask seed from getrandom(2); an integer: the deterministic, not secure test generator."""
        return self._gen_seeded("cbs_trans_key_seeded_generate", TRANS_KEY_SEEDED_GLWES, aes_key, seed)

    def gen_seeded_forward_transciphering_keys(self, aes_key, seed=None):
        """The forward (CTR) twin of gen_seeded_transciphering_keys -> (mask_seed, bodies [896][1024])."""
        return self._gen_seeded("cbs_fwd_trans_key_seeded_generate", FWD_TRANS_KEY_SEEDED_GLWES, aes_key, seed)

    def _gen_seeded(self, fn, nglwe, aes_key, seed):
        bodies, pb = _out((nglwe, 1024))
        ms = (ctypes.c_uint8 * 32)()
        _, pk = _u8(aes_key)
        if seed is None:
            _check(getattr(lib(), fn + "_os_entropy")(self._h, pk, ms, pb), fn + "_os_entropy")
        else:
            _check(getattr(lib(), fn)(self._h, pk, ctypes.c_uint64(seed), ms, pb), fn)
        return bytes(ms), bodies

    def encrypt_bits_big(self, bits, seed):
        bits = np.ascontiguousarray(bits, dtype=np.uint8)
        out, po = _out((bits.size, LWE_BIG))
        _check(lib().cbs_encrypt_bits_big(self._h, bits.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), bits.size,
                                          ctypes.c_uint64(seed), po), "cbs_encrypt_bits_big")
        return out

    def encrypt_bits_small(self, bits, seed):
        bits = np.ascontiguousarray(bits, dtype=np.uint8)
        out, po = _out((bits.size, LWE_SMALL))
        _check(lib().cbs_encrypt_bits_small(self._h, bits.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), bits.size,
                                            ctypes.c_uint64(seed), po), "cbs_encrypt_bits_small")
        return out


def load_trans_key(path):
    """bincode AllRdKeys (src/data_struct.rs:11-26) -> (k10_9, k8_1, k0)."""
    k10_9, p1 = _out((4, 16, 2, GLWE_WORDS))
    k8_1, p2 = _out((8, 4, 16, 2, GLWE_WORDS))
    k0, p3 = _out((16, 2, GLWE_WORDS))
    _check(lib().cbs_trans_key_load(str(path).encode(), p1, p2, p3), "cbs_trans_key_load")
    return k10_9, k8_1, k0


def save_trans_key(path, k10_9, k8_1, k0):
    a, p1 = _u64(k10_9)
    b, p2 = _u64(k8_1)
    c, p3 = _u64(k0)
    _check(lib().cbs_trans_key_save(str(path).encode(), p1, p2, p3), "cbs_trans_key_save")


def load_fwd_trans_key(path):
    a, p1 = _out((3, 16, 2, GLWE_WORDS))
    b, p2 = _out((8, 3, 16, 2, GLWE_WORDS))
    c, p3 = _out((16, 2, GLWE_WORDS))
    _check(lib().cbs_fwd_trans_key_load(str(path).encode(), p1, p2, p3), "cbs_fwd_trans_key_load")
    return a, b, c


def save_fwd_trans_key(path, kf_first, kf_mid, kf_last):
    a, p1 = _u64(kf_first)
    b, p2 = _u64(kf_mid)
    c, p3 = _u64(kf_last)
    _check(lib().cbs_fwd_trans_key_save(str(path).encode(), p1, p2, p3), "cbs_fwd_trans_key_save")


def _seed(mask_seed):
    if len(mask_seed) != 32:
        raise ValueError("a mask seed is 32 bytes")
    return (ctypes.c_uint8 * 32).from_buffer_copy(bytes(mask_seed))


def _bodies(bodies, nglwe):
    b, pb = _u64(bodies)
    if b.size != nglwe * 1024:
        raise ValueError(f"seeded key bodies must hold {nglwe} x 1024 words, got {b.size}")
    return b, pb


def expand_seeded_trans_key(mask_seed, bodies):
    """Seeded inverse key -> (k10_9, k8_1, k0) with the masks regenerated from mask_seed: the arrays every reference-format
    call takes (upload_trans_key, aes_to_lwe_transciphering, save_trans_key)."""
    a, p1 = _out((4, 16, 2, GLWE_WORDS))
    b, p2 = _out((8, 4, 16, 2, GLWE_WORDS))
    c, p3 = _out((16, 2, GLWE_WORDS))
    _, pb = _bodies(bodies, TRANS_KEY_SEEDED_GLWES)
    _check(lib().cbs_trans_key_seeded_expand(_seed(mask_seed), pb, p1, p2, p3), "cbs_trans_key_seeded_expand")
    return a, b, c


def expand_seeded_fwd_trans_key(mask_seed, bodies):
    """Seeded forward key -> (kf_first, kf_mid, kf_last)."""
    a, p1 = _out((3, 16, 2, GLWE_WORDS))
    b, p2 = _out((8, 3, 16, 2, GLWE_WORDS))
    c, p3 = _out((16, 2, GLWE_WORDS))
    _, pb = _bodies(bodies, FWD_TRANS_KEY_SEEDED_GLWES)
    _check(lib().cbs_fwd_trans_key_seeded_expand(_seed(mask_seed), pb, p1, p2, p3), "cbs_fwd_trans_key_seeded_expand")
    return a, b, c


def _load_seeded(fn, nglwe, path):
    bodies, pb = _out((nglwe, 1024))
    ms = (ctypes.c_uint8 * 32)()
    _check(getattr(lib(), fn)(str(path).encode(), ms, pb), fn)
    return bytes(ms), bodies


def load_seeded_trans_key(path):
    """seeded inverse key file ("CBSSEED1") -> (mask_seed, bodies [1184][1024])."""
    return _load_seeded("cbs_trans_key_seeded_load", TRANS_KEY_SEEDED_GLWES, path)


def save_seeded_trans_key(path, mask_seed, bodies):
    _, pb = _bodies(bodies, TRANS_KEY_SEEDED_GLWES)
    _check(lib().cbs_trans_key_seeded_save(str(path).encode(), _seed(mask_seed), pb), "cbs_trans_key_seeded_save")


def load_seeded_fwd_trans_key(path):
    """seeded forward key file -> (mask_seed, bodies [896][1024])."""
    return _load_seeded("cbs_fwd_trans_key_seeded_load", FWD_TRANS_KEY_SEEDED_GLWES, path)


def save_seeded_fwd_trans_key(path, mask_seed, bodies):
    _, pb = _bodies(bodies, FWD_TRANS_KEY_SEEDED_GLWES)
    _check(lib().cbs_fwd_trans_key_seeded_save(str(path).encode(), _seed(mask_seed), pb), "cbs_fwd_trans_key_seeded_save")


def load_lwe_list(path):
    data = ctypes.POINTER(ctypes.c_uint64)()
    count, words = ctypes.c_uint64(), ctypes.c_uint64()
    _check(lib().cbs_lwe_list_load(str(path).encode(), ctypes.byref(data), ctypes.byref(count), ctypes.byref(words)),
           "cbs_lwe_list_load")
    try:
        return np.ctypeslib.as_array(data, shape=(count.value * words.value,)).reshape(count.value, words.value).copy()
    finally:
        lib().cbs_free(data)


def save_lwe_list(path, arr):
    arr = np.ascontiguousarray(arr, dtype=np.uint64)
    a, p = _u64(arr)
    _check(lib().cbs_lwe_list_save(str(path).encode(), p, ctypes.c_uint64(arr.shape[0]), ctypes.c_uint64(arr.shape[1])),
           "cbs_lwe_list_save")


def glwe_decrypt_bits(glwe_sk, glwe, nbits=None):
    """Client side of Context.pack_lwes: coefficient j of GLWE g -> bit g*1024 + j (delta = 2^63) under glwe_sk [2048] (the
    big LWE key); glwe [nglwe][3072]; the first nbits bits (default all nglwe*1024) as uint64 0/1."""
    g, pg = _u64(np.reshape(glwe, (-1, GLWE_WORDS)))
    s, ps = _u64(np.reshape(glwe_sk, (2048,)))
    nbits = g.shape[0] * 1024 if nbits is None else int(nbits)
    out, po = _out((nbits,))
    _check(lib().cbs_glwe_decrypt_bits(ps, pg, ctypes.c_uint64(g.shape[0]), ctypes.c_uint64(nbits), po), "cbs_glwe_decrypt_bits")
    return out


def load_glwe_list(path):
    """bincode GlweCiphertextList {data, glwe_size = 3, polynomial_size = 1024, modulus} -> [nglwe][3072]."""
    data = ctypes.POINTER(ctypes.c_uint64)()
    n = ctypes.c_uint64()
    _check(lib().cbs_glwe_list_load(str(path).encode(), ctypes.byref(data), ctypes.byref(n)), "cbs_glwe_list_load")
    try:
        if n.value == 0:
            return np.zeros((0, GLWE_WORDS), dtype=np.uint64)
        return np.ctypeslib.as_array(data, shape=(n.value * GLWE_WORDS,)).reshape(n.value, GLWE_WORDS).copy()
    finally:
        lib().cbs_free(data)


def save_glwe_list(path, glwe):
    g, p = _u64(np.reshape(glwe, (-1, GLWE_WORDS)))
    _check(lib().cbs_glwe_list_save(str(path).encode(), p, ctypes.c_uint64(g.shape[0])), "cbs_glwe_list_save")


class Context:
    """One B200: Fourier-domain keys + workspaces (cbs_ctx).  Creation uploads the standard-domain
    keys and converts them on the GPU, replacing server_encrypted_aes_decryption.rs:645-687."""

    def __init__(self, keyset, device=0):
        h = ctypes.c_void_p()
        _check(lib().cbs_ctx_create(keyset._h, int(device), ctypes.byref(h)), "cbs_ctx_create")
        self._h = h
        self._keyset = keyset
        self._stream = None  # the cudaStream_t handle last given to set_stream; None: the context's own stream

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.cbs_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    @property
    def launch_count(self):
        return int(lib().cbs_ctx_launch_count(self._h))

    def set_stream(self, cuda_stream):
        _check(lib().cbs_ctx_set_stream(self._h, ctypes.c_void_p(cuda_stream)), "cbs_ctx_set_stream")
        self._stream = int(cuda_stream) if cuda_stream else None

    @property
    def stream(self):
        """The cudaStream_t handle (an int) the context issues its work on, as given to set_stream; None: its own stream."""
        return self._stream

    def synchronize(self):
        _check(lib().cbs_ctx_synchronize(self._h), "cbs_ctx_synchronize")

    # ---- cbs_lib stage mirrors (host buffers) ----
    def keyswitch_lwe_ciphertext_by_glwe_keyswitch(self, lwe_big):
        """cbs_lib/src/fourier_glwe_keyswitch.rs:344 — LWE(2048) -> LWE(768), batched."""
        a, pi = _u64(np.reshape(lwe_big, (-1, LWE_BIG)))
        out, po = _out((a.shape[0], LWE_SMALL))
        _check(lib().cbs_lwe_keyswitch(self._h, pi, po, a.shape[0]), "cbs_lwe_keyswitch")
        return out

    def blind_rotate(self, lwe_small):
        """accumulator (ggsw_conv.rs:250-268) + gen_blind_rotate_local_assign (pbs.rs:70)."""
        a, pi = _u64(np.reshape(lwe_small, (-1, LWE_SMALL)))
        out, po = _out((a.shape[0], GLWE_WORDS))
        _check(lib().cbs_blind_rotate(self._h, pi, po, a.shape[0]), "cbs_blind_rotate")
        return out

    def glev_from_acc(self, acc):
        """cbs_lib/src/ggsw_conv.rs:302-314."""
        a, pi = _u64(np.reshape(acc, (-1, GLWE_WORDS)))
        out, po = _out((a.shape[0], 7, GLWE_WORDS))
        _check(lib().cbs_glev_from_acc(self._h, pi, po, a.shape[0]), "cbs_glev_from_acc")
        return out

    def trace_assign(self, glwe):
        """trace_assign, cbs_lib/src/automorphism.rs:195 (returns the traced copy)."""
        a = np.array(np.reshape(glwe, (-1, GLWE_WORDS)), dtype=np.uint64, order="C", copy=True)
        _check(lib().cbs_trace(self._h, a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), a.shape[0]), "cbs_trace")
        return a

    def lwe_msb_bit_to_glev_by_trace_with_preprocessing(self, lwe_small):
        """cbs_lib/src/ggsw_conv.rs:231."""
        a, pi = _u64(np.reshape(lwe_small, (-1, LWE_SMALL)))
        out, po = _out((a.shape[0], 7, GLWE_WORDS))
        _check(lib().cbs_lwe_msb_bit_to_glev(self._h, pi, po, a.shape[0]), "cbs_lwe_msb_bit_to_glev")
        return out

    def switch_scheme(self, glev):
        """switch_scheme, cbs_lib/src/ggsw_conv.rs:163."""
        a, pi = _u64(np.reshape(glev, (-1, GLEV_WORDS)))
        out, po = _out((a.shape[0], GGSW_WORDS))
        _check(lib().cbs_scheme_switch(self._h, pi, po, a.shape[0]), "cbs_scheme_switch")
        return out

    def circuit_bootstrap_lwe_ciphertext_by_trace_with_preprocessing(self, lwe_small):
        """cbs_lib/src/ggsw_conv.rs:409 (GGSW returned in the standard domain)."""
        a, pi = _u64(np.reshape(lwe_small, (-1, LWE_SMALL)))
        out, po = _out((a.shape[0], GGSW_WORDS))
        _check(lib().cbs_circuit_bootstrap(self._h, pi, po, a.shape[0]), "cbs_circuit_bootstrap")
        return out

    def evaluate_8_to_8_cipher_lut(self, ggsw_bits, luts):
        """src/bin/server_encrypted_aes_decryption.rs:550.  ggsw_bits [nbytes][8][GGSW], luts
        [nbytes][nluts][2][GLWE] -> out [nbytes][nluts][8][2049]."""
        g, pg = _u64(np.reshape(ggsw_bits, (-1, 8, GGSW_WORDS)))
        nbytes = g.shape[0]
        l, pl = _u64(np.reshape(luts, (nbytes, -1, 2, GLWE_WORDS)))
        nluts = l.shape[1]
        out, po = _out((nbytes, nluts, 8, LWE_BIG))
        _check(lib().cbs_lut8_eval(self._h, pg, nbytes, pl, nluts, po), "cbs_lut8_eval")
        return out

    def max_of_two(self, ggsw, op, a_idx, b_idx):
        """max_of_two, src/bin/server_encrypted_compute.rs:34-98, one ladder per pair (a_idx[p], b_idx[p]): ggsw
        [nvals][16][GGSW] (standard domain, MSB first), op [nvals][16][GLWE] data operands -> [npairs][16][2049]."""
        g, pg = _u64(np.reshape(ggsw, (-1, 16, GGSW_WORDS)))
        o, po = _u64(np.reshape(op, (g.shape[0], 16, GLWE_WORDS)))
        (a, pa), (b, pb) = _i32(a_idx), _i32(b_idx)
        if a.size != b.size:
            raise ValueError(f"{a.size} a indices for {b.size} b indices")
        out, pout = _out((a.size, 16, LWE_BIG))
        _check(lib().cbs_max_of_two(self._h, pg, po, g.shape[0], pa, pb, a.size, pout), "cbs_max_of_two")
        return out

    def evaluate_gathered_luts(self, ggsw, sel, luts, lut_index, out_index, nout):
        """the gathered LUT ladder of the stage-8 circuits: ggsw [nbits][GGSW], sel [njobs][8] (-1: constant-0 selector),
        luts [nluts][GLWE] -> out [nout][2049]; job j writes rows out_index[j] .. + 3, the other rows are zero."""
        g, pg = _u64(np.reshape(ggsw, (-1, GGSW_WORDS)))
        l, pl = _u64(np.reshape(luts, (-1, GLWE_WORDS)))
        s, ps = _i32(sel)
        (li, pli), (oi, poi) = _i32(lut_index), _i32(out_index)
        if s.size != 8 * li.size or oi.size != li.size:
            raise ValueError(f"sel of {s.size} entries, {li.size} LUT indices and {oi.size} output indices")
        out, pout = _out((nout, LWE_BIG))
        _check(lib().cbs_lut8_gather_eval(self._h, pg, g.shape[0], ps, pl, l.shape[0], pli, poi, li.size, pout, int(nout)),
               "cbs_lut8_gather_eval")
        return out

    def aes_first_rounds(self, ct, k10_9):
        """known_rotate_keyed_lut x4 + he_inv_mix_columns_precomp + he_inv_shift_rows
        (server_encrypted_aes_decryption.rs:89-128)."""
        c, pc = _u8(ct)
        nblocks = c.size // 16
        k, pk = _u64(k10_9)
        out, po = _out((nblocks, 128, LWE_BIG))
        _check(lib().cbs_aes_first_rounds(self._h, pc, nblocks, pk, po), "cbs_aes_first_rounds")
        return out

    def he_inv_mix_columns_and_shift_rows(self, t4):
        """he_inv_mix_columns_precomp + he_inv_shift_rows (server_encrypted_aes_decryption.rs:195-265);
        t4 = [4 (x9,x11,x13,x14)][nblocks][128][2049]."""
        t, pt = _u64(t4)
        nblocks = t.shape[1]
        out, po = _out((nblocks, 128, LWE_BIG))
        _check(lib().cbs_aes_inv_linear(self._h, pt, nblocks, po), "cbs_aes_inv_linear")
        return out

    def aes_to_lwe_transciphering(self, ct, k10_9, k8_1, k0):
        """aes_to_lwe_trasnciphering, src/bin/server_encrypted_aes_decryption.rs:28-191, over all
        16-byte blocks of `ct` -> [nblocks][128][2049] (MSB first inside each byte)."""
        c, pc = _u8(ct)
        nblocks = c.size // 16
        a, p1 = _u64(k10_9)
        b, p2 = _u64(k8_1)
        d, p3 = _u64(k0)
        out, po = _out((nblocks, 128, LWE_BIG))
        _check(lib().cbs_aes128_transcipher(self._h, pc, nblocks, p1, p2, p3, po), "cbs_aes128_transcipher")
        return out

    def aes_ctr_to_lwe_transciphering(self, ct, iv, kf_first, kf_mid, kf_last):
        """CTR-mode transciphering: forward AES of the public counter blocks (he_sub_bytes_8_to_24,
        he_shift_rows, he_mix_columns_precomp; cbs_lib/src/aes_he.rs:285-474) xor the public ciphertext
        -> [nblocks][128][2049] plaintext bits, MSB first inside each byte."""
        c, pc = _u8(ct)
        nblocks = c.size // 16
        ivb, pi = _u8(iv)
        a, p1 = _u64(kf_first)
        b, p2 = _u64(kf_mid)
        d, p3 = _u64(kf_last)
        out, po = _out((nblocks, 128, LWE_BIG))
        _check(lib().cbs_aes128_ctr_transcipher(self._h, pc, nblocks, pi, p1, p2, p3, po), "cbs_aes128_ctr_transcipher")
        return out

    def max_u16(self, lwe_bits):
        """stage 8, src/bin/server_encrypted_compute.rs:99-359: [nvals*16][2049] -> [16][2049]."""
        a, pi = _u64(np.reshape(lwe_bits, (-1, LWE_BIG)))
        nvals = a.shape[0] // 16
        out, po = _out((16, LWE_BIG))
        _check(lib().cbs_max_u16(self._h, pi, nvals, po), "cbs_max_u16")
        return out

    def max_u16_lut(self, lwe_bits):
        """the maximum as a LUT circuit (noise independent of data and tree depth); same formats as max_u16."""
        a, pi = _u64(np.reshape(lwe_bits, (-1, LWE_BIG)))
        nvals = a.shape[0] // 16
        out, po = _out((16, LWE_BIG))
        _check(lib().cbs_max_u16_lut(self._h, pi, nvals, po), "cbs_max_u16_lut")
        return out

    def sum_u16(self, lwe_bits):
        """sum of the values mod 2^16 (combines per-GPU partial inner products); same formats as max_u16."""
        a, pi = _u64(np.reshape(lwe_bits, (-1, LWE_BIG)))
        nvals = a.shape[0] // 16
        out, po = _out((16, LWE_BIG))
        _check(lib().cbs_sum_u16(self._h, pi, nvals, po), "cbs_sum_u16")
        return out

    def inner_product_u16(self, lwe_bits):
        """mini-workload #2 (harness/cleartext_impl.py:65-70): [nvals*16][2049] -> [16][2049] encrypting
        sum_i (x_i * y_i mod 2^16) mod 2^16, x = first half of the values, y = second half."""
        a, pi = _u64(np.reshape(lwe_bits, (-1, LWE_BIG)))
        nvals = a.shape[0] // 16
        out, po = _out((16, LWE_BIG))
        _check(lib().cbs_inner_product_u16(self._h, pi, nvals, po), "cbs_inner_product_u16")
        return out

    def pack_lwes(self, lwe_bits):
        """LWE-to-GLWE packing (cbs_lib glwe_conv.rs pack_lwes): [count][2049] big LWE bits -> [ceil(count/1024)][3072] GLWE;
        coefficient i % 1024 of GLWE i // 1024 decrypts to bit i (glwe_decrypt_bits)."""
        a, pi = _u64(np.reshape(lwe_bits, (-1, LWE_BIG)))
        out, po = _out(((a.shape[0] + 1023) // 1024, GLWE_WORDS))
        _check(lib().cbs_pack_lwes(self._h, pi, a.shape[0], po), "cbs_pack_lwes")
        return out

    def measure_fp64_tflops(self):
        v = ctypes.c_double()
        _check(lib().cbs_measure_fp64_tflops(self._h, ctypes.byref(v)), "cbs_measure_fp64_tflops")
        return float(v.value)

    # ---- device-resident API (bench) ----
    def upload_trans_key(self, k10_9, k8_1, k0):
        a, p1 = _u64(k10_9)
        b, p2 = _u64(k8_1)
        d, p3 = _u64(k0)
        _check(lib().cbs_trans_key_upload(self._h, p1, p2, p3), "cbs_trans_key_upload")

    def upload_fwd_trans_key(self, kf_first, kf_mid, kf_last):
        """forward-direction (CTR) transciphering key -> device, once; then ctr_transcipher_dev can be called repeatedly."""
        (a, pa), (b, pb), (c, pc) = _u64(kf_first), _u64(kf_mid), _u64(kf_last)
        _check(lib().cbs_fwd_trans_key_upload(self._h, pa, pb, pc), "cbs_fwd_trans_key_upload")

    def upload_seeded_trans_key(self, mask_seed, bodies):
        """seeded inverse key -> device: the bodies are copied, the masks expanded on the GPU (k_expand_lut_masks)."""
        _, pb = _bodies(bodies, TRANS_KEY_SEEDED_GLWES)
        _check(lib().cbs_trans_key_seeded_upload(self._h, _seed(mask_seed), pb), "cbs_trans_key_seeded_upload")

    def upload_seeded_fwd_trans_key(self, mask_seed, bodies):
        """seeded forward (CTR) key -> device, as upload_seeded_trans_key."""
        _, pb = _bodies(bodies, FWD_TRANS_KEY_SEEDED_GLWES)
        _check(lib().cbs_fwd_trans_key_seeded_upload(self._h, _seed(mask_seed), pb), "cbs_fwd_trans_key_seeded_upload")

    # key slots: many transciphering keys resident at once, block b of a call under slot slots[b] (include/cbs_b200.h)
    def reserve_trans_key_slots(self, nslots):
        """grow the inverse (ECB) key pool to nslots slots (29.1 MB each); uploaded slots are kept."""
        _check(lib().cbs_trans_key_slots_reserve(self._h, int(nslots)), "cbs_trans_key_slots_reserve")

    def reserve_fwd_trans_key_slots(self, nslots):
        """grow the forward (CTR) key pool to nslots slots (22.0 MB each)."""
        _check(lib().cbs_fwd_trans_key_slots_reserve(self._h, int(nslots)), "cbs_fwd_trans_key_slots_reserve")

    def upload_trans_key_slot(self, slot, k10_9, k8_1, k0):
        (a, p1), (b, p2), (d, p3) = _u64(k10_9), _u64(k8_1), _u64(k0)
        _check(lib().cbs_trans_key_slot_upload(self._h, int(slot), p1, p2, p3), "cbs_trans_key_slot_upload")

    def upload_fwd_trans_key_slot(self, slot, kf_first, kf_mid, kf_last):
        (a, p1), (b, p2), (d, p3) = _u64(kf_first), _u64(kf_mid), _u64(kf_last)
        _check(lib().cbs_fwd_trans_key_slot_upload(self._h, int(slot), p1, p2, p3), "cbs_fwd_trans_key_slot_upload")

    def upload_seeded_trans_key_slot(self, slot, mask_seed, bodies):
        _, pb = _bodies(bodies, TRANS_KEY_SEEDED_GLWES)
        _check(lib().cbs_trans_key_seeded_slot_upload(self._h, int(slot), _seed(mask_seed), pb), "cbs_trans_key_seeded_slot_upload")

    def upload_seeded_fwd_trans_key_slot(self, slot, mask_seed, bodies):
        _, pb = _bodies(bodies, FWD_TRANS_KEY_SEEDED_GLWES)
        _check(lib().cbs_fwd_trans_key_seeded_slot_upload(self._h, int(slot), _seed(mask_seed), pb),
               "cbs_fwd_trans_key_seeded_slot_upload")

    def transcipher_slots_dev(self, d_ct_ptr, slots, nblocks, d_out_ptr):
        """device-resident ECB transciphering, block b under key slot slots[b] (a host sequence of nblocks ints)."""
        s, ps = _slots(slots, nblocks)
        _check(lib().cbs_aes128_transcipher_slots_dev(self._h, ctypes.c_void_p(d_ct_ptr), ps, int(nblocks),
                                                      ctypes.c_void_p(d_out_ptr)), "cbs_aes128_transcipher_slots_dev")

    def ctr_transcipher_slots_dev(self, d_ctr_ptr, d_ct_ptr, slots, nblocks, d_out_ptr):
        """device-resident CTR transciphering, block b under key slot slots[b]; d_ctr = the public counter blocks."""
        s, ps = _slots(slots, nblocks)
        _check(lib().cbs_aes128_ctr_transcipher_slots_dev(self._h, ctypes.c_void_p(d_ctr_ptr), ctypes.c_void_p(d_ct_ptr), ps,
                                                          int(nblocks), ctypes.c_void_p(d_out_ptr)),
               "cbs_aes128_ctr_transcipher_slots_dev")

    def transcipher_slots(self, ct, slots):
        """ECB ciphertext blocks, block b under slot slots[b] -> [nblocks][128][2049] (MSB first inside each byte)."""
        c, pc = _u8(ct)
        nblocks = c.size // 16
        s, ps = _slots(slots, nblocks)
        out, po = _out((nblocks, 128, LWE_BIG))
        _check(lib().cbs_aes128_transcipher_slots(self._h, pc, ps, nblocks, po), "cbs_aes128_transcipher_slots")
        return out

    def ctr_transcipher_slots(self, ctr, ct, slots):
        """CTR: ctr = the nblocks 16-byte counter blocks (each sender its own IV), ct = the AES-CTR ciphertext, block b under
        slot slots[b] -> [nblocks][128][2049] plaintext bits."""
        c, pc = _u8(ct)
        nblocks = c.size // 16
        k, pk = _u8(ctr)
        if k.size != c.size:
            raise ValueError(f"{k.size // 16} counter blocks for {nblocks} ciphertext blocks")
        s, ps = _slots(slots, nblocks)
        out, po = _out((nblocks, 128, LWE_BIG))
        _check(lib().cbs_aes128_ctr_transcipher_slots(self._h, pk, pc, ps, nblocks, po), "cbs_aes128_ctr_transcipher_slots")
        return out

    def ctr_transcipher_dev(self, d_ctr_ptr, d_ct_ptr, nblocks, d_out_ptr):
        """device-resident CTR transciphering: d_ctr = the public 16-byte counter blocks, d_ct = the AES-CTR ciphertext."""
        _check(lib().cbs_aes128_ctr_transcipher_dev(self._h, ctypes.c_void_p(d_ctr_ptr), ctypes.c_void_p(d_ct_ptr), nblocks,
                                                    ctypes.c_void_p(d_out_ptr)), "cbs_aes128_ctr_transcipher_dev")

    def transcipher_dev(self, d_ct_ptr, nblocks, d_out_ptr):
        _check(lib().cbs_aes128_transcipher_dev(self._h, ctypes.c_void_p(d_ct_ptr), int(nblocks), ctypes.c_void_p(d_out_ptr)),
               "cbs_aes128_transcipher_dev")

    # stage 8 on device buffers: raw device pointers, same results as the host-buffer calls, queued on the context stream
    def max_u16_dev(self, d_in_ptr, nvals, d_out_ptr):
        """d_in [nvals][16][2049] -> d_out [16][2049]; ladder or LUT circuit by the rule of max_u16."""
        _check(lib().cbs_max_u16_dev(self._h, ctypes.c_void_p(d_in_ptr), int(nvals), ctypes.c_void_p(d_out_ptr)), "cbs_max_u16_dev")

    def max_u16_lut_dev(self, d_in_ptr, nvals, d_out_ptr):
        _check(lib().cbs_max_u16_lut_dev(self._h, ctypes.c_void_p(d_in_ptr), int(nvals), ctypes.c_void_p(d_out_ptr)),
               "cbs_max_u16_lut_dev")

    def sum_u16_dev(self, d_in_ptr, nvals, d_out_ptr):
        _check(lib().cbs_sum_u16_dev(self._h, ctypes.c_void_p(d_in_ptr), int(nvals), ctypes.c_void_p(d_out_ptr)), "cbs_sum_u16_dev")

    def inner_product_u16_dev(self, d_x_ptr, d_y_ptr, npairs, d_out_ptr):
        """d_x, d_y [npairs][16][2049] -> d_out [16][2049] encrypting sum_i (x_i * y_i mod 2^16) mod 2^16."""
        _check(lib().cbs_inner_product_u16_dev(self._h, ctypes.c_void_p(d_x_ptr), ctypes.c_void_p(d_y_ptr), int(npairs),
                                               ctypes.c_void_p(d_out_ptr)), "cbs_inner_product_u16_dev")

    def pack_lwes_dev(self, d_in_ptr, count, d_out_ptr):
        """d_in [count][2049] big LWE (a transcipher_dev output as it is) -> d_out [ceil(count/1024)][3072] GLWE, queued on
        the context stream."""
        _check(lib().cbs_pack_lwes_dev(self._h, ctypes.c_void_p(d_in_ptr), int(count), ctypes.c_void_p(d_out_ptr)),
               "cbs_pack_lwes_dev")

    def circuit_bootstrap_dev(self, d_in_ptr, count):
        _check(lib().cbs_circuit_bootstrap_dev(self._h, ctypes.c_void_p(d_in_ptr), int(count)), "cbs_circuit_bootstrap_dev")

    def blind_rotate_dev(self, d_in_ptr, d_acc_ptr, count):
        _check(lib().cbs_blind_rotate_dev(self._h, ctypes.c_void_p(d_in_ptr), ctypes.c_void_p(d_acc_ptr), int(count)),
               "cbs_blind_rotate_dev")
