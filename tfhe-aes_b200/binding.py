"""ctypes binding of libtfhe_aes_b200.so (include/tfhe_aes_b200.h).

No CPU fallback: constructing an Engine without the built library or without a CUDA device raises.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))


def lib_path():
    return os.path.join(_HERE, "libtfhe_aes_b200.so")


class TfaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"tfhe_aes_b200 error {code}: {msg}")
        self.code = code


class Params(C.Structure):
    """WopbsParameters (client.rs:31-57)."""
    _fields_ = [(n, C.c_uint32) for n in (
        "lwe_dim", "glwe_dim", "poly_size", "pbs_base_log", "pbs_level", "ks_base_log", "ks_level",
        "pfks_base_log", "pfks_level", "cbs_base_log", "cbs_level", "message_modulus", "carry_modulus",
        "_pad")] + [("lwe_std", C.c_double), ("glwe_std", C.c_double), ("pfks_std", C.c_double)]


def param_opt():
    """PARAM_OPT (client.rs:31-57)."""
    return Params(669, 4, 512, 8, 5, 2, 6, 12, 3, 15, 1, 2, 1, 0,
                  3.0517578125e-05, 3.162026630747649e-16, 3.162026630747649e-16)


def param_test():
    """Small, insecure functional set for fast tests (main.rs:75 suggests one; none is given)."""
    return Params(24, 1, 512, 8, 5, 2, 6, 12, 3, 15, 1, 2, 1, 0, 2.0 ** -24, 2.0 ** -50, 2.0 ** -50)


def param_test2():
    """param_test with 2-bit blocks: general extract_bits (PBS loop) and CMux tree."""
    return Params(24, 1, 512, 8, 5, 2, 6, 12, 3, 15, 1, 4, 1, 0, 2.0 ** -24, 2.0 ** -50, 2.0 ** -50)


class TfaCtrStream(C.Structure):
    """tfa_ctr_stream: one public-IV AES-CTR stream (include/tfhe_aes_b200.h)."""
    _fields_ = [("round_keys", C.c_void_p), ("data", C.c_void_p), ("first_lo", C.c_uint64), ("first_hi", C.c_uint64),
                ("iv", C.c_uint8 * 16), ("nblk", C.c_int32), ("_pad", C.c_int32)]


assert C.sizeof(TfaCtrStream) == 56


def _ctr_stream(rk_ptr, iv, first, nblk, data_ptr):
    iv = iv.to_bytes(16, "big") if isinstance(iv, int) else bytes(iv)
    if len(iv) != 16:
        raise ValueError("iv must be an int or 16 bytes")
    first %= 2 ** 128
    return TfaCtrStream(rk_ptr, data_ptr, first & (2 ** 64 - 1), first >> 64, (C.c_uint8 * 16)(*iv), nblk, 0)


class TfaCtrEncStream(C.Structure):
    """tfa_ctr_enc_stream: one AES-CTR stream with an encrypted IV (include/tfhe_aes_b200.h)."""
    _fields_ = [("round_keys", C.c_void_p), ("iv_ct", C.c_void_p), ("data", C.c_void_p), ("first_lo", C.c_uint64),
                ("first_hi", C.c_uint64), ("nblk", C.c_int32), ("_pad", C.c_int32)]


assert C.sizeof(TfaCtrEncStream) == 48


def _ctr_enc_stream(rk_ptr, iv_ptr, first, nblk, data_ptr):
    first %= 2 ** 128
    return TfaCtrEncStream(rk_ptr, iv_ptr, data_ptr, first & (2 ** 64 - 1), first >> 64, nblk, 0)


_lib = None

_SIGS = {
    "tfa_ctx_create": [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_void_p)],
    "tfa_ctx_load_keys": [C.c_void_p] * 4,
    "tfa_ctx_key_buffers": [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_int)],
    "tfa_many_wopbs": [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p],
    "tfa_many_wopbs_dev": [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p],
    "tfa_sbox": [C.c_void_p, C.c_void_p, C.c_int, C.c_int],
    "tfa_many_sbox": [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p],
    "tfa_aes_key_expansion": [C.c_void_p] * 4,
    "tfa_aes_key_expansion_ex": [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p],
    "tfa_aes_encrypt_ex": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int],
    "tfa_aes_decrypt_ex": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int],
    "tfa_aes_key_expansion_dev": [C.c_void_p] * 4,
    "tfa_aes_encrypt": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_aes_decrypt": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_aes_encryption": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_aes_decryption": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_aes_encrypt_dev": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_aes_decrypt_dev": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_aes_round": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_aes_round_dev": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_add_scalar": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_add_scalar_dev": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_aes_ctr": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, C.c_void_p],
    "tfa_xor_clear": [C.c_void_p, C.c_void_p, C.c_char_p, C.c_int],
    "tfa_xor_clear_dev": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_aes_ctr_dev": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, C.c_void_p],
    "tfa_aes_ctr_public_iv": [C.c_void_p, C.POINTER(TfaCtrStream), C.c_int, C.c_int, C.c_void_p],
    "tfa_aes_ctr_public_iv_dev": [C.c_void_p, C.POINTER(TfaCtrStream), C.c_int, C.c_int, C.c_void_p],
    "tfa_aes_ctr_streams": [C.c_void_p, C.POINTER(TfaCtrEncStream), C.c_int, C.c_int, C.c_void_p],
    "tfa_aes_ctr_streams_dev": [C.c_void_p, C.POINTER(TfaCtrEncStream), C.c_int, C.c_int, C.c_void_p],
    "tfa_pack_lwe": [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p],
    "tfa_pack_lwe_dev": [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p],
    "tfa_unpack_lwe": [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p],
    "tfa_unpack_lwe_dev": [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p],
    "tfa_add_round_key": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_mix_columns": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_inv_mix_columns": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int],
    "tfa_shift_rows": [C.c_void_p, C.c_void_p, C.c_int, C.c_int],
    "tfa_keyswitch": [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p],
    "tfa_bootstrap": [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p],
    "tfa_extract_bits": [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p],
    "tfa_pfks": [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p],
    "tfa_circuit_bootstrap": [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p],
    "tfa_vertical_packing": [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p],
    "tfa_fourier_forward": [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p],
    "tfa_client_keygen": [C.c_void_p, C.c_uint64],
    "tfa_client_encrypt_bytes": [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_void_p],
    "tfa_client_decrypt_bytes": [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p],
    "tfa_client_encrypt_bytes_dev": [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_void_p],
    "tfa_client_decrypt_bytes_dev": [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p],
    "tfa_client_secret_keys": [C.c_void_p, C.c_void_p, C.c_void_p],
    "tfa_gen_lut": [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p],
    "tfa_bootstrap_dev": [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p],
    "tfa_client_set_secret_keys": [C.c_void_p, C.c_void_p, C.c_void_p],
    "tfa_ctx_profile": [C.c_void_p, C.c_int],
    "tfa_ctx_set_pbs_schedule": [C.c_void_p, C.c_int],
    "tfa_ctx_profile_report": [C.c_void_p, C.c_void_p, C.c_void_p],
    "tfa_measure_fp64_peak": [C.c_void_p, C.POINTER(C.c_double)],
    "tfa_measure_fp64_peaks": [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)],
    "tfa_lut_size": [C.c_void_p, C.c_int],
}


def load_library():
    """Load the C-ABI library.  Raises if it has not been built (there is no fallback)."""
    global _lib
    if _lib is None:
        path = lib_path()
        if not os.path.exists(path):
            raise RuntimeError(f"{path} is missing: run __graft_entry__.build() (nvcc, sm_100a). No CPU fallback exists.")
        lib = C.CDLL(path)
        lib.tfa_last_error.restype = C.c_char_p
        lib.tfa_last_error.argtypes = [C.c_void_p]
        lib.tfa_ctx_launch_count.restype = C.c_uint64
        lib.tfa_ctx_launch_count.argtypes = [C.c_void_p]
        lib.tfa_ctx_pbs_count.restype = C.c_uint64
        lib.tfa_ctx_pbs_count.argtypes = [C.c_void_p]
        lib.tfa_ctx_destroy.argtypes = [C.c_void_p]
        lib.tfa_ctx_destroy.restype = None
        for name in ("tfa_ctx_alloc_keys", "tfa_ctx_keys_ready", "tfa_ctx_synchronize"):
            getattr(lib, name).argtypes = [C.c_void_p]
        for name, sig in _SIGS.items():
            fn = getattr(lib, name)
            fn.argtypes = sig
            fn.restype = C.c_int
        _lib = lib
    return _lib


def _p(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)


def lut_size(params, nb_block):
    return load_library().tfa_lut_size(C.byref(params), nb_block)


def gen_lut(params, nb_block, f):
    """sbox::gen_lut::gen_lut (gen_lut.rs:9-42).  `f` is a callable or a table of f(v)."""
    log_basis = int(np.log2(params.message_modulus)) + int(np.log2(params.carry_modulus))
    nvals = 1 << (nb_block * log_basis)
    table = np.array([f(v) for v in range(nvals)], dtype=np.uint64) if callable(f) else np.ascontiguousarray(f, dtype=np.uint64)
    assert len(table) == nvals
    size = lut_size(params, nb_block)
    out = np.zeros((nb_block, size), dtype=np.uint64)
    rc = load_library().tfa_gen_lut(C.byref(params), nb_block, _p(table), _p(out))
    if rc:
        raise TfaError(rc, "gen_lut: bad arguments")
    return out


# tables/table.rs:2-37 and sbox.rs:20-42 in the clear (generated from the field arithmetic)
def _xtime(x):
    return ((x << 1) ^ (0x1B if x & 0x80 else 0)) & 0xFF


def _gmul(a, b):
    r = 0
    while b:
        if b & 1:
            r ^= a
        a = _xtime(a)
        b >>= 1
    return r


def _make_sbox():
    sb = [0] * 256
    for x in range(256):
        inv = 0
        if x:
            inv = next(y for y in range(1, 256) if _gmul(x, y) == 1)
        s = r = inv
        for _ in range(4):
            r = ((r << 1) | (r >> 7)) & 0xFF
            s ^= r
        sb[x] = s ^ 0x63
    inv = [0] * 256
    for x, s in enumerate(sb):
        inv[s] = x
    return bytes(sb), bytes(inv)


SBOX, INV_SBOX = _make_sbox()


def mul2(x): return _gmul(x, 2)
def mul3(x): return _gmul(x, 3)
def mul9(x): return _gmul(x, 9)
def mul11(x): return _gmul(x, 11)
def mul13(x): return _gmul(x, 13)
def mul14(x): return _gmul(x, 14)


class Engine:
    """Owns one tfa_ctx (one GPU).  Host-buffer methods take / return numpy uint64 arrays."""

    def __init__(self, params, device=0, stream=None):
        self.lib = load_library()
        self.params = params
        self.n, self.k, self.N = params.lwe_dim, params.glwe_dim, params.poly_size
        self.big = self.k * self.N
        self.lw = self.big + 1
        self.gsz = (self.k + 1) * self.N
        self.bpb = int(np.log2(params.message_modulus * params.carry_modulus))
        h = C.c_void_p()
        rc = self.lib.tfa_ctx_create(C.byref(params), device, C.c_void_p(stream) if stream else None, C.byref(h))
        if rc:
            raise TfaError(rc, self.lib.tfa_last_error(None).decode())
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.tfa_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc:
            raise TfaError(rc, self.lib.tfa_last_error(self.h).decode())

    @property
    def launch_count(self):
        return int(self.lib.tfa_ctx_launch_count(self.h))

    @property
    def pbs_count(self):
        """LWE ciphertexts blind-rotated on this context since creation"""
        return int(self.lib.tfa_ctx_pbs_count(self.h))

    def synchronize(self):
        self._ck(self.lib.tfa_ctx_synchronize(self.h))

    STAGES = ("ks_decompose", "ks_gemv", "pbs", "pfks_decompose", "pfks_gemv", "fourier", "vp", "cmux_tree", "linear", "misc")

    def set_pbs_schedule(self, schedule):
        """0 = automatic, 2 = warp-specialised PBS kernel, 3 = one ciphertext per two-CTA cluster, 4 = two ciphertext sets per CTA
        (include/tfhe_aes_b200.h: tfa_ctx_set_pbs_schedule).  Any other value raises TfaError with code 1 (TFA_ERR_PARAM)."""
        self._ck(self.lib.tfa_ctx_set_pbs_schedule(self.h, int(schedule)))

    def profile(self, enable=True):
        self._ck(self.lib.tfa_ctx_profile(self.h, int(enable)))

    def profile_report(self):
        ms = np.zeros(10, dtype=np.float64)
        cnt = np.zeros(10, dtype=np.int32)
        self._ck(self.lib.tfa_ctx_profile_report(self.h, _p(ms), _p(cnt)))
        return {n: (float(ms[i]), int(cnt[i])) for i, n in enumerate(self.STAGES) if cnt[i]}

    def measure_fp64_peaks(self):
        """(DFMA, DMMA) microbenchmarks of the FP64 pipe, TFLOP/s"""
        a, b = C.c_double(), C.c_double()
        self._ck(self.lib.tfa_measure_fp64_peaks(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def measure_fp64_peak(self):
        v = C.c_double()
        self._ck(self.lib.tfa_measure_fp64_peak(self.h, C.byref(v)))
        return v.value

    # device-pointer calls (ints are raw device addresses, e.g. torch.Tensor.data_ptr())
    def bootstrap_dev(self, in_ptr, count, lut_ptr, pre_add, post_add, out_ptr):
        self._ck(self.lib.tfa_bootstrap_dev(self.h, C.c_void_p(in_ptr), count, C.c_void_p(lut_ptr), pre_add, post_add, C.c_void_p(out_ptr)))

    def aes_ctr_dev(self, rk_ptr, iv_ptr, first, nblk, out_ptr):
        self._ck(self.lib.tfa_aes_ctr_dev(self.h, C.c_void_p(rk_ptr), C.c_void_p(iv_ptr), first & (2 ** 64 - 1), first >> 64, nblk, C.c_void_p(out_ptr)))

    def aes_ctr_public_iv_dev(self, streams, out_ptr, rounds=10):
        """streams: list of (round_keys device pointer, iv (int or 16 bytes), first, nblk, data device pointer or None);
        out_ptr: device [total][16][8][lw].  Asynchronous on the context stream."""
        arr = (TfaCtrStream * len(streams))(*[_ctr_stream(rk, iv, first, nblk, data) for rk, iv, first, nblk, data in streams])
        self._ck(self.lib.tfa_aes_ctr_public_iv_dev(self.h, arr, len(streams), rounds, C.c_void_p(out_ptr) if out_ptr else None))

    def aes_ctr_streams_dev(self, streams, out_ptr, rounds=10):
        """streams: list of (round_keys device pointer, encrypted IV device pointer, first, nblk, data device pointer or None);
        out_ptr: device [total][16][8][lw].  Streams with the same IV pointer share one IV.  Asynchronous on the context stream."""
        arr = (TfaCtrEncStream * len(streams))(*[_ctr_enc_stream(rk, iv, first, nblk, data) for rk, iv, first, nblk, data in streams])
        self._ck(self.lib.tfa_aes_ctr_streams_dev(self.h, arr, len(streams), rounds, C.c_void_p(out_ptr) if out_ptr else None))

    def pack_lwe_dev(self, lwe_ptr, count, packed_ptr):
        """device [count][lw] LWEs -> device uint16 [ceil(count / N)][k+1][N] (tfa_pack_lwe_dev).  Asynchronous on the context stream."""
        self._ck(self.lib.tfa_pack_lwe_dev(self.h, C.c_void_p(lwe_ptr), count, C.c_void_p(packed_ptr)))

    def unpack_lwe_dev(self, packed_ptr, count, lwe_ptr):
        """device uint16 [ceil(count / N)][k+1][N] -> device [count][lw] LWEs (tfa_unpack_lwe_dev).  Asynchronous on the context stream."""
        self._ck(self.lib.tfa_unpack_lwe_dev(self.h, C.c_void_p(packed_ptr), count, C.c_void_p(lwe_ptr)))

    def aes_encrypt_dev(self, rk_ptr, st_ptr, nblk):
        self._ck(self.lib.tfa_aes_encrypt_dev(self.h, C.c_void_p(rk_ptr), C.c_void_p(st_ptr), nblk))

    def aes_decrypt_dev(self, rk_ptr, st_ptr, nblk):
        self._ck(self.lib.tfa_aes_decrypt_dev(self.h, C.c_void_p(rk_ptr), C.c_void_p(st_ptr), nblk))

    def aes_round_dev(self, rk_ptr, st_ptr, nblk):
        self._ck(self.lib.tfa_aes_round_dev(self.h, C.c_void_p(rk_ptr), C.c_void_p(st_ptr), nblk))

    def aes_key_expansion_dev(self, key_ptr, rk_ptr, rcon_ptr=None):
        self._ck(self.lib.tfa_aes_key_expansion_dev(self.h, C.c_void_p(key_ptr), C.c_void_p(rcon_ptr) if rcon_ptr else None, C.c_void_p(rk_ptr)))

    def client_set_secret_keys(self, lwe_sk, glwe_sk):
        a = np.ascontiguousarray(lwe_sk, dtype=np.uint64)
        b = np.ascontiguousarray(glwe_sk, dtype=np.uint64)
        self._ck(self.lib.tfa_client_set_secret_keys(self.h, _p(a), _p(b)))

    # -- keys ------------------------------------------------------------------------------------
    def load_keys(self, bsk, ksk, pfpksk):
        bsk, ksk, pfpksk = (np.ascontiguousarray(a, dtype=np.uint64) for a in (bsk, ksk, pfpksk))
        self._ck(self.lib.tfa_ctx_load_keys(self.h, _p(bsk), _p(ksk), _p(pfpksk)))

    def alloc_keys(self):
        self._ck(self.lib.tfa_ctx_alloc_keys(self.h))

    def key_buffers(self):
        ptrs = (C.c_void_p * 8)()
        sizes = (C.c_size_t * 8)()
        cnt = C.c_int()
        self._ck(self.lib.tfa_ctx_key_buffers(self.h, ptrs, sizes, C.byref(cnt)))
        return [(int(ptrs[i]), int(sizes[i])) for i in range(cnt.value)]

    def keys_ready(self):
        self._ck(self.lib.tfa_ctx_keys_ready(self.h))

    # -- client harness --------------------------------------------------------------------------
    def client_keygen(self, seed):
        self._ck(self.lib.tfa_client_keygen(self.h, seed))

    def client_encrypt_bytes(self, data, seed=0):
        data = np.frombuffer(bytes(data), dtype=np.uint8).copy()
        out = np.zeros((len(data), 8, self.lw), dtype=np.uint64)
        self._ck(self.lib.tfa_client_encrypt_bytes(self.h, _p(data), len(data), seed, _p(out)))
        return out

    def client_decrypt_bytes(self, ct):
        ct = np.ascontiguousarray(ct, dtype=np.uint64).reshape(-1, 8, self.lw)
        out = np.zeros(len(ct), dtype=np.uint8)
        self._ck(self.lib.tfa_client_decrypt_bytes(self.h, _p(ct), len(ct), _p(out)))
        return bytes(out)

    def client_encrypt_bytes_dev(self, data, dev_ptr, seed=0):
        data = np.frombuffer(bytes(data), dtype=np.uint8).copy()
        self._ck(self.lib.tfa_client_encrypt_bytes_dev(self.h, _p(data), len(data), seed, C.c_void_p(dev_ptr)))

    def client_decrypt_bytes_dev(self, dev_ptr, count):
        out = np.zeros(count, dtype=np.uint8)
        self._ck(self.lib.tfa_client_decrypt_bytes_dev(self.h, C.c_void_p(dev_ptr), count, _p(out)))
        return bytes(out)

    def client_secret_keys(self):
        a = np.zeros(self.n, dtype=np.uint64)
        b = np.zeros(self.big, dtype=np.uint64)
        self._ck(self.lib.tfa_client_secret_keys(self.h, _p(a), _p(b)))
        return a, b

    # -- sbox module -----------------------------------------------------------------------------
    def many_wopbs(self, ct_in, luts):
        """ct_in [nct][nblocks][lw]; luts [L][nblocks][lut_size] -> [nct][L][nblocks][lw]"""
        ct_in = np.ascontiguousarray(ct_in, dtype=np.uint64)
        luts = np.ascontiguousarray(luts, dtype=np.uint64)
        nct, nblocks = ct_in.shape[0], ct_in.shape[1]
        L = luts.shape[0]
        assert luts.shape[1] == nblocks and ct_in.shape[2] == self.lw
        out = np.zeros((nct, L, nblocks, self.lw), dtype=np.uint64)
        self._ck(self.lib.tfa_many_wopbs(self.h, _p(ct_in), nct, nblocks, _p(luts), L, _p(out)))
        return out

    def sbox(self, bytes_ct, inv=False):
        b = np.array(bytes_ct, dtype=np.uint64).reshape(-1, 8 // self.bpb, self.lw)
        self._ck(self.lib.tfa_sbox(self.h, _p(b), len(b), int(inv)))
        return b

    def many_sbox(self, bytes_ct, inv=False):
        b = np.ascontiguousarray(bytes_ct, dtype=np.uint64).reshape(-1, 8 // self.bpb, self.lw)
        out = np.zeros((len(b), 4 if inv else 3, 8 // self.bpb, self.lw), dtype=np.uint64)
        self._ck(self.lib.tfa_many_sbox(self.h, _p(b), len(b), int(inv), _p(out)))
        return out

    # -- Server ----------------------------------------------------------------------------------
    def aes_key_expansion(self, key_ct, rcon_ct=None):
        key_ct = np.ascontiguousarray(key_ct, dtype=np.uint64).reshape(16, 8, self.lw)
        out = np.zeros((11, 16, 8, self.lw), dtype=np.uint64)
        rc = np.ascontiguousarray(rcon_ct, dtype=np.uint64) if rcon_ct is not None else None
        self._ck(self.lib.tfa_aes_key_expansion(self.h, _p(key_ct), _p(rc), _p(out)))
        return out

    def aes_key_expansion_ex(self, key_ct, rcon_ct=None):
        """AES-128/192/256: key_ct [16 | 24 | 32][8][lw] -> [11 | 13 | 15][16][8][lw]"""
        key_ct = np.ascontiguousarray(key_ct, dtype=np.uint64).reshape(-1, 8, self.lw)
        nb = len(key_ct)
        out = np.zeros((nb // 4 + 7, 16, 8, self.lw), dtype=np.uint64)
        rc = np.ascontiguousarray(rcon_ct, dtype=np.uint64) if rcon_ct is not None else None
        self._ck(self.lib.tfa_aes_key_expansion_ex(self.h, _p(key_ct), nb, _p(rc), _p(out)))
        return out

    def aes_crypt_ex(self, rk, states, decrypt=False):
        """rounds follow from the number of round keys (11 / 13 / 15)"""
        rk = np.ascontiguousarray(rk, dtype=np.uint64).reshape(-1, 16, 8, self.lw)
        st = np.array(states, dtype=np.uint64).reshape(-1, 16, 8, self.lw)
        fn = self.lib.tfa_aes_decrypt_ex if decrypt else self.lib.tfa_aes_encrypt_ex
        self._ck(fn(self.h, _p(rk), _p(st), len(st), len(rk) - 1))
        return st

    def _state_call(self, fn, rk, states):
        rk = np.ascontiguousarray(rk, dtype=np.uint64)
        st = np.array(states, dtype=np.uint64).reshape(-1, 16, 8, self.lw)
        self._ck(fn(self.h, _p(rk), _p(st), len(st)))
        return st

    def aes_encrypt(self, rk, states):
        return self._state_call(self.lib.tfa_aes_encrypt, rk, states)

    def aes_decrypt(self, rk, states):
        return self._state_call(self.lib.tfa_aes_decrypt, rk, states)

    def aes_round(self, round_key, states):
        return self._state_call(self.lib.tfa_aes_round, round_key, states)

    def add_scalar(self, states, counters):
        st = np.array(states, dtype=np.uint64).reshape(-1, 16, 8, self.lw)
        ctr = np.array([[c & (2 ** 64 - 1), c >> 64] for c in counters], dtype=np.uint64)
        assert len(ctr) == len(st)
        self._ck(self.lib.tfa_add_scalar(self.h, _p(st), _p(ctr), len(st)))
        return st

    def aes_ctr(self, rk, iv_ct, first, nblk):
        rk = np.ascontiguousarray(rk, dtype=np.uint64)
        iv_ct = np.ascontiguousarray(iv_ct, dtype=np.uint64)
        out = np.zeros((nblk, 16, 8, self.lw), dtype=np.uint64)
        self._ck(self.lib.tfa_aes_ctr(self.h, _p(rk), _p(iv_ct), first & (2 ** 64 - 1), first >> 64, nblk, _p(out)))
        return out

    def aes_ctr_public_iv(self, streams, rounds=10):
        """AES-CTR with public IVs, many streams in one call.  streams: list of (round_keys [rounds+1][16][8][lw], iv (int or
        16 bytes, AES byte order), first, nblk, data (16 * nblk bytes) or None).  Returns [total][16][8][lw]: block b of a stream
        encrypts AES(iv + first + b) XOR data[b], streams in order."""
        keep, rks = [], {}
        for rk, _, _, _, _ in streams:   # one array per distinct round-key object: the library uploads each pointer once
            if rk is not None and id(rk) not in rks:
                rks[id(rk)] = np.ascontiguousarray(rk, dtype=np.uint64)
        structs = []
        for rk, iv, first, nblk, data in streams:
            d = None
            if data is not None:
                d = np.frombuffer(bytes(data), dtype=np.uint8).copy()
                if len(d) != 16 * nblk:
                    raise ValueError("data must hold 16 bytes per block")
                keep.append(d)
            structs.append(_ctr_stream(_p(rks[id(rk)]) if rk is not None else None, iv, first, nblk, _p(d)))
        total = sum(max(int(s.nblk), 0) for s in structs)
        # an out-of-range total is left to the library to reject (TFA_ERR_PARAM) without allocating for it
        out = np.zeros((total, 16, 8, self.lw), dtype=np.uint64) if 0 < total < 2 ** 27 else None
        arr = (TfaCtrStream * len(structs))(*structs)
        self._ck(self.lib.tfa_aes_ctr_public_iv(self.h, arr, len(structs), rounds, _p(out)))
        return out

    def aes_ctr_streams(self, streams, rounds=10):
        """AES-CTR with encrypted IVs, many streams in one call.  streams: list of (round_keys [rounds+1][16][8][lw], encrypted IV
        [16][8][lw], first, nblk, data (16 * nblk bytes) or None).  Returns [total][16][8][lw]: block b of a stream encrypts
        AES(iv + first + b) XOR data[b], streams in order.  Each distinct round-key and IV object is uploaded once, and streams that
        pass the same IV object share its bit bootstraps."""
        arrays, keep = {}, []
        byte = (8 // self.bpb) * self.lw
        sizes = {0: (rounds + 1) * 16 * byte, 1: 16 * byte}
        for st in streams:                 # one array per distinct object: the library uploads each pointer once
            for i in (0, 1):
                a = st[i]
                if a is not None and id(a) not in arrays:
                    arr = np.ascontiguousarray(a, dtype=np.uint64)
                    if rounds in (10, 12, 14) and arr.size != sizes[i]:   # other rounds: TfaError from the library
                        raise ValueError(("round keys" if i == 0 else "encrypted IV") + f" must hold {sizes[i]} words, got {arr.size}")
                    arrays[id(a)] = arr
        structs = []
        for rk, iv, first, nblk, data in streams:
            d = None
            if data is not None:
                d = np.frombuffer(bytes(data), dtype=np.uint8).copy()
                if len(d) != 16 * nblk:
                    raise ValueError("data must hold 16 bytes per block")
                keep.append(d)
            ptr = [_p(arrays[id(a)]) if a is not None else None for a in (rk, iv)]
            structs.append(_ctr_enc_stream(ptr[0], ptr[1], first, nblk, _p(d)))
        total = sum(max(int(s.nblk), 0) for s in structs)
        # an out-of-range total is left to the library to reject (TFA_ERR_PARAM) without allocating for it
        out = np.zeros((total, 16, 8, self.lw), dtype=np.uint64) if 0 < total < 2 ** 27 else None
        arr = (TfaCtrEncStream * len(structs))(*structs)
        self._ck(self.lib.tfa_aes_ctr_streams(self.h, arr, len(structs), rounds, _p(out)))
        return out

    def xor_clear(self, states, data: bytes):
        """Transciphering step: states (keystream ciphertexts) ^= clear data blocks (16 bytes each)."""
        st = np.array(states, dtype=np.uint64).reshape(-1, 16, 8, self.lw)
        assert len(data) == 16 * len(st)
        self._ck(self.lib.tfa_xor_clear(self.h, _p(st), bytes(data), len(st)))
        return st

    def packed_glwes(self, count):
        """GLWEs that hold `count` packed LWEs: ceil(count / N)"""
        return -(-count // self.N)

    def pack_lwe(self, ct):
        """LWEs (any shape ending in lw, e.g. [nblk][16][8][lw]) -> np.uint16 [ceil(count / N)][k+1][N]: LWE j is coefficient j % N
        of GLWE j // N, words round(x / 2^48) mod 2^16 (include/tfhe_aes_b200.h: tfa_pack_lwe)"""
        ct = np.ascontiguousarray(ct, dtype=np.uint64).reshape(-1, self.lw)
        out = np.zeros((self.packed_glwes(len(ct)), self.k + 1, self.N), dtype=np.uint16)
        self._ck(self.lib.tfa_pack_lwe(self.h, _p(ct), len(ct), _p(out)))
        return out

    def unpack_lwe(self, packed, count):
        """np.uint16 [G][k+1][N] from pack_lwe -> the first `count` LWEs [count][lw] (sample extraction, no key needed)"""
        packed = np.ascontiguousarray(packed, dtype=np.uint16).reshape(-1, self.k + 1, self.N)
        if count > len(packed) * self.N:
            raise ValueError(f"{len(packed)} GLWEs hold at most {len(packed) * self.N} LWEs, not {count}")
        out = np.zeros((max(count, 0), self.lw), dtype=np.uint64)
        self._ck(self.lib.tfa_unpack_lwe(self.h, _p(packed), count, _p(out)))
        return out

    def add_round_key(self, states, rk):
        st = np.array(states, dtype=np.uint64).reshape(-1, 16, 8, self.lw)
        rk = np.ascontiguousarray(rk, dtype=np.uint64)
        self._ck(self.lib.tfa_add_round_key(self.h, _p(st), _p(rk), len(st)))
        return st

    def mix_columns(self, mul):
        mul = np.ascontiguousarray(mul, dtype=np.uint64).reshape(-1, 16, 3, 8, self.lw)
        out = np.zeros((len(mul), 16, 8, self.lw), dtype=np.uint64)
        self._ck(self.lib.tfa_mix_columns(self.h, _p(mul), _p(out), len(mul)))
        return out

    def inv_mix_columns(self, mul):
        mul = np.ascontiguousarray(mul, dtype=np.uint64).reshape(-1, 16, 4, 8, self.lw)
        out = np.zeros((len(mul), 16, 8, self.lw), dtype=np.uint64)
        self._ck(self.lib.tfa_inv_mix_columns(self.h, _p(mul), _p(out), len(mul)))
        return out

    def shift_rows(self, states, inverse=False):
        st = np.array(states, dtype=np.uint64).reshape(-1, 16, 8, self.lw)
        self._ck(self.lib.tfa_shift_rows(self.h, _p(st), len(st), int(inverse)))
        return st

    # -- primitives ------------------------------------------------------------------------------
    def keyswitch(self, ct):
        ct = np.ascontiguousarray(ct, dtype=np.uint64).reshape(-1, self.lw)
        out = np.zeros((len(ct), self.n + 1), dtype=np.uint64)
        self._ck(self.lib.tfa_keyswitch(self.h, _p(ct), len(ct), _p(out)))
        return out

    def bootstrap(self, ct, lut):
        ct = np.ascontiguousarray(ct, dtype=np.uint64).reshape(-1, self.n + 1)
        lut = np.ascontiguousarray(lut, dtype=np.uint64)
        out = np.zeros((len(ct), self.lw), dtype=np.uint64)
        self._ck(self.lib.tfa_bootstrap(self.h, _p(ct), len(ct), _p(lut), _p(out)))
        return out

    def extract_bits(self, ct, delta_log, nbits):
        ct = np.ascontiguousarray(ct, dtype=np.uint64).reshape(-1, self.lw)
        out = np.zeros((len(ct), nbits, self.n + 1), dtype=np.uint64)
        self._ck(self.lib.tfa_extract_bits(self.h, _p(ct), len(ct), delta_log, nbits, _p(out)))
        return out

    def pfks(self, key_index, ct):
        ct = np.ascontiguousarray(ct, dtype=np.uint64).reshape(-1, self.lw)
        out = np.zeros((len(ct), self.gsz), dtype=np.uint64)
        self._ck(self.lib.tfa_pfks(self.h, key_index, _p(ct), len(ct), _p(out)))
        return out

    def circuit_bootstrap(self, ct):
        ct = np.ascontiguousarray(ct, dtype=np.uint64).reshape(-1, self.n + 1)
        out = np.zeros((len(ct), self.params.cbs_level, self.k + 1, self.gsz), dtype=np.uint64)
        self._ck(self.lib.tfa_circuit_bootstrap(self.h, _p(ct), len(ct), _p(out)))
        return out

    def vertical_packing(self, lut, ggsw_std):
        """lut [nouts][npoly][N]; ggsw_std [nggsw][...] (index 0 = MSB) -> [nouts][lw]"""
        lut = np.ascontiguousarray(lut, dtype=np.uint64)
        ggsw_std = np.ascontiguousarray(ggsw_std, dtype=np.uint64)
        nouts, npoly = lut.shape[0], lut.shape[1]
        out = np.zeros((nouts, self.lw), dtype=np.uint64)
        self._ck(self.lib.tfa_vertical_packing(self.h, _p(lut), nouts, npoly, _p(ggsw_std), ggsw_std.shape[0], _p(out)))
        return out

    def fourier_forward(self, polys):
        polys = np.ascontiguousarray(polys, dtype=np.uint64).reshape(-1, self.N)
        out = np.zeros((len(polys), self.N // 2, 2), dtype=np.float64)
        self._ck(self.lib.tfa_fourier_forward(self.h, _p(polys), len(polys), _p(out)))
        return out[..., 0] + 1j * out[..., 1]
