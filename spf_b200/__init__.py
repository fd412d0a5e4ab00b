"""spf_b200 -- B200-native TFHE bootstrapping engine behind parasol_runtime's Evaluation boundary.

This package is a thin ctypes mirror of the reference's `Evaluation` / `KeylessEvaluation`
(parasol_runtime/src/crypto/evaluation.rs) over the C ABI of ``libspf_b200.so``
(``include/spf_b200.h``).  All arithmetic runs in hand-written sm_100a CUDA kernels
(``spf_b200/csrc``); there is NO CPU fallback -- if the library or a GPU is missing every
entry point raises.  Nothing here imports the test oracle.
"""
from __future__ import annotations

import ctypes as C
import operator
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# SPF_B200_LIB selects an alternative build of the same library (kernel-tuning experiments only)
LIB_PATH = os.environ.get("SPF_B200_LIB") or os.path.join(_HERE, "libspf_b200.so")


class SpfError(RuntimeError):
    """Mirrors parasol_runtime's RuntimeError(String) (runtime_error.rs:8) plus the panics of
    assert_is_valid (dst.rs:520-523), surfaced as exceptions with the C ABI's status code."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"spf_b200 error {code}: {msg}")
        self.code = code


class Radix(C.Structure):
    _fields_ = [("radix_log", C.c_uint32), ("count", C.c_uint32)]


class Params(C.Structure):
    """parasol_runtime/src/params.rs:59-91 (spf_params)."""

    _fields_ = [
        ("lwe_n", C.c_uint32),
        ("lwe_std", C.c_double),
        ("glwe_k", C.c_uint32),
        ("glwe_n", C.c_uint32),
        ("glwe_std", C.c_double),
        ("cbs", Radix),
        ("pbs", Radix),
        ("ks", Radix),
        ("pfks", Radix),
        ("ss", Radix),
        ("tr", Radix),
    ]


_lib = None
_vp = C.c_void_p
_sz = C.c_size_t

# name -> argtypes (restype int unless listed in _RESTYPES); this is the full export list of
# include/spf_b200.h and is what tests/test_abi.py checks the .so against.
ABI = {
    "spf_b200_default_128": [C.POINTER(Params)],
    "spf_b200_len_lwe_l0": [C.POINTER(Params)],
    "spf_b200_len_lwe_l1": [C.POINTER(Params)],
    "spf_b200_len_glwe_l1": [C.POINTER(Params)],
    "spf_b200_len_glev_l1": [C.POINTER(Params)],
    "spf_b200_len_ggsw_l1": [C.POINTER(Params)],
    "spf_b200_len_bsk": [C.POINTER(Params)],
    "spf_b200_len_ksk": [C.POINTER(Params)],
    "spf_b200_len_ssk": [C.POINTER(Params)],
    "spf_b200_len_ak": [C.POINTER(Params)],
    "spf_b200_create": [C.POINTER(Params), _vp, _sz, _vp, _sz, _vp, _sz, _vp, _sz, C.c_int, C.POINTER(_vp)],
    "spf_b200_create_from_device": [C.POINTER(Params), _vp, _sz, _vp, _sz, _vp, _sz, _vp, _sz, C.c_int, C.POINTER(_vp)],
    "spf_b200_destroy": [_vp],
    "spf_b200_last_error": [_vp],
    "spf_b200_kernel_launches": [_vp],
    "spf_b200_device": [_vp],
    "spf_b200_synchronize": [_vp],
    "spf_b200_circuit_bootstrap": [_vp, _vp, _vp, _sz],
    "spf_b200_programmable_bootstrap": [_vp, _vp, _vp, _vp, C.c_uint32, C.c_uint32, _sz],
    "spf_b200_cmux": [_vp, _vp, _vp, _vp, _vp, _sz],
    "spf_b200_glev_cmux": [_vp, _vp, _vp, _vp, _vp, _sz],
    "spf_b200_multiply_glwe_ggsw": [_vp, _vp, _vp, _vp, _sz],
    "spf_b200_keyswitch_lwe_l1_lwe_l0": [_vp, _vp, _vp, _sz],
    "spf_b200_sample_extract_l1": [_vp, _vp, _vp, _vp, C.c_uint32, _sz],
    "spf_b200_scheme_switch": [_vp, _vp, _vp, _sz],
    "spf_b200_trace": [_vp, _vp, _vp, _sz],
    "spf_b200_not": [_vp, _vp, _vp, _sz],
    "spf_b200_xor": [_vp, _vp, _vp, _vp, _sz],
    "spf_b200_mul_xn": [_vp, _vp, _vp, C.c_uint32, _sz],
    "spf_b200_rlwe_encrypt_public": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz],
    "spf_b200_dev_rlwe_encrypt_public": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp],
    "spf_b200_dev_circuit_bootstrap": [_vp, _vp, _vp, _sz, C.c_int, _vp],
    "spf_b200_dev_programmable_bootstrap": [_vp, _vp, _vp, _vp, C.c_uint32, C.c_uint32, _sz, _vp],
    "spf_b200_dev_cmux": [_vp, _vp, _vp, _sz, _vp, _vp, _sz, _vp],
    "spf_b200_dev_keyswitch_lwe_l1_lwe_l0": [_vp, _vp, _vp, _sz, _vp],
    "spf_b200_dev_sample_extract_l1": [_vp, _vp, _vp, _vp, C.c_uint32, _sz, _vp],
    "spf_b200_dev_fft_rescale": [_vp, _vp, _vp, _sz, C.c_int, _vp],
    "spf_b200_fp64_peak": [_vp, C.POINTER(C.c_double)],
    "spf_b200_serialized_size_compute_key": [C.POINTER(Params)],
    "spf_b200_serialized_limit_compute_key": [C.POINTER(Params)],
    "spf_b200_parse_compute_key": [C.POINTER(Params), _vp, _sz, C.POINTER(_sz * 4)],
    "spf_b200_write_compute_key": [C.POINTER(Params), _vp, _sz, _vp, _vp, _vp, _vp, C.POINTER(_sz)],
    "spf_b200_create_from_serialized": [C.POINTER(Params), _vp, _sz, C.c_int, C.POINTER(_vp)],
    "spf_b200_serialized_size_ciphertext": [C.POINTER(Params), C.c_int],
    "spf_b200_parse_ciphertext": [C.POINTER(Params), C.c_int, _vp, _sz, C.POINTER(_sz)],
    "spf_b200_write_ciphertext": [C.POINTER(Params), C.c_int, _vp, _vp, _sz, C.POINTER(_sz)],
}
_RESTYPES = {
    "spf_b200_default_128": None,
    "spf_b200_destroy": None,
    "spf_b200_last_error": C.c_char_p,
    "spf_b200_kernel_launches": C.c_uint64,
    **{n: _sz for n in ("spf_b200_len_lwe_l0", "spf_b200_len_lwe_l1", "spf_b200_len_glwe_l1", "spf_b200_len_glev_l1",
                        "spf_b200_len_ggsw_l1", "spf_b200_len_bsk", "spf_b200_len_ksk", "spf_b200_len_ssk",
                        "spf_b200_len_ak", "spf_b200_serialized_size_compute_key",
                        "spf_b200_serialized_limit_compute_key", "spf_b200_serialized_size_ciphertext")},
}


def lib() -> C.CDLL:
    """Load libspf_b200.so.  Fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `make` (or __graft_entry__.build()); "
                "spf_b200 has no CPU fallback")
        l = C.CDLL(LIB_PATH)
        for name, argtypes in ABI.items():
            fn = getattr(l, name)
            fn.argtypes = argtypes
            fn.restype = _RESTYPES.get(name, C.c_int)
        _lib = l
    return _lib


def default_128() -> Params:
    """DEFAULT_128 (parasol_runtime/src/params.rs:107-134)."""
    p = Params()
    lib().spf_b200_default_128(C.byref(p))
    return p


def _ptr(a) -> int:
    """Host pointer of a C-contiguous numpy array, or a raw integer device pointer."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        if not a.flags["C_CONTIGUOUS"]:
            raise SpfError(-1, "buffers must be C-contiguous")
        return a.ctypes.data
    return int(a)


class Evaluation:
    """`Evaluation` (+ the `KeylessEvaluation` it derefs to) of
    parasol_runtime/src/crypto/evaluation.rs, batched.  Every method takes arrays whose leading
    dimension is the batch; outputs are freshly allocated numpy arrays (the reference's
    `enc.allocate_*` + `&mut` out-parameter pattern, circuit_processor/mod.rs:333-340)."""

    def __init__(self, bsk_fft, ksk, ssk_fft, ak_fft, params: Params | None = None, device: int = 0,
                 on_device: bool = False):
        """Evaluation::new(Arc<ComputeKey>, &Params, &Encryption) (evaluation.rs:161-197).
        Key arrays are ComputeKey's four fields in the reference layout; with on_device=True
        they are raw device pointers (ints) to the same layout already on `device`."""
        l = lib()
        self.params = params if params is not None else default_128()
        p = self.params
        self._h = _vp()
        lens = (l.spf_b200_len_bsk(C.byref(p)), l.spf_b200_len_ksk(C.byref(p)), l.spf_b200_len_ssk(C.byref(p)),
                l.spf_b200_len_ak(C.byref(p)))
        if on_device:
            rc = l.spf_b200_create_from_device(C.byref(p), bsk_fft, lens[0], ksk, lens[1], ssk_fft, lens[2], ak_fft,
                                               lens[3], device, C.byref(self._h))
        else:
            arrs = []
            for a, dt, n, name in ((bsk_fft, np.complex128, lens[0], "bs_key"), (ksk, np.uint64, lens[1], "ks_key"),
                                   (ssk_fft, np.complex128, lens[2], "ss_key"), (ak_fft, np.complex128, lens[3], "auto_key")):
                a = np.ascontiguousarray(a, dtype=dt).reshape(-1)
                if a.size != n:
                    raise SpfError(-1, f"{name} has {a.size} elements, params require {n}")
                arrs.append(a)
            rc = l.spf_b200_create(C.byref(p), arrs[0].ctypes.data, lens[0], arrs[1].ctypes.data, lens[1],
                                   arrs[2].ctypes.data, lens[2], arrs[3].ctypes.data, lens[3], device,
                                   C.byref(self._h))
        if rc != 0:
            raise SpfError(rc, (l.spf_b200_last_error(None) or b"").decode())
        self.len_lwe_l0 = l.spf_b200_len_lwe_l0(C.byref(p))
        self.len_lwe_l1 = l.spf_b200_len_lwe_l1(C.byref(p))
        self.len_glwe = l.spf_b200_len_glwe_l1(C.byref(p))
        self.len_glev = l.spf_b200_len_glev_l1(C.byref(p))
        self.len_ggsw = l.spf_b200_len_ggsw_l1(C.byref(p))

    @classmethod
    def from_serialized(cls, data: bytes, params: Params | None = None, device: int = 0) -> "Evaluation":
        """safe_bincode::deserialize::<ComputeKey>(data, params) (safe_bincode.rs:16-27) followed by
        Evaluation::new: loads a compute-key file written by the reference, unmodified."""
        from . import serialize

        bsk, ksk, ssk, ak = serialize.load_compute_key(data, params)
        return cls(bsk, ksk, ssk, ak, params=params, device=device)

    # -- plumbing --------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().spf_b200_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise SpfError(rc, (lib().spf_b200_last_error(self._h) or b"").decode())

    @property
    def handle(self):
        return self._h

    @property
    def kernel_launches(self) -> int:
        return int(lib().spf_b200_kernel_launches(self._h))

    def synchronize(self):
        self._check(lib().spf_b200_synchronize(self._h))

    def set_max_in_flight(self, n: int) -> None:
        """Flow control of the asynchronous executor: at most n spawned graphs between dispatch and completion."""
        self._check(lib().spf_b200_set_max_in_flight(self._h, int(n)))

    def fp64_peak_tflops(self) -> float:
        out = C.c_double()
        self._check(lib().spf_b200_fp64_peak(self._h, C.byref(out)))
        return out.value

    @staticmethod
    def _in(a, dtype, width, name):
        a = np.ascontiguousarray(a, dtype=dtype)
        if a.ndim == 1:
            a = a.reshape(1, -1)
        if a.ndim != 2 or a.shape[1] != width:
            raise SpfError(-1, f"{name}: expected [batch][{width}] {np.dtype(dtype).name}, got {a.shape}")
        return a

    # -- Evaluation ------------------------------------------------------------------------
    def circuit_bootstrap(self, lwe0) -> np.ndarray:
        """Evaluation::circuit_bootstrap (evaluation.rs:211-225): L0 LWE -> L1 GGSW (FFT)."""
        x = self._in(lwe0, np.uint64, self.len_lwe_l0, "lwe0")
        out = np.empty((x.shape[0], self.len_ggsw), dtype=np.complex128)
        self._check(lib().spf_b200_circuit_bootstrap(self._h, out.ctypes.data, x.ctypes.data, x.shape[0]))
        return out

    def programmable_bootstrap(self, lwe0, lut_glwe, log_chi: int = 0, log_v: int = 0) -> np.ndarray:
        """generalized_programmable_bootstrap (programmable_bootstrapping.rs:342-410)."""
        x = self._in(lwe0, np.uint64, self.len_lwe_l0, "lwe0")
        lut = self._in(lut_glwe, np.uint64, self.len_glwe, "lut")
        out = np.empty((x.shape[0], self.len_glwe), dtype=np.uint64)
        self._check(lib().spf_b200_programmable_bootstrap(self._h, out.ctypes.data, x.ctypes.data, lut.ctypes.data,
                                                          log_chi, log_v, x.shape[0]))
        return out

    def keyswitch_lwe_l1_lwe_l0(self, lwe1) -> np.ndarray:
        """Evaluation::keyswitch_lwe_l1_lwe_l0 (evaluation.rs:243-252)."""
        x = self._in(lwe1, np.uint64, self.len_lwe_l1, "lwe1")
        out = np.empty((x.shape[0], self.len_lwe_l0), dtype=np.uint64)
        self._check(lib().spf_b200_keyswitch_lwe_l1_lwe_l0(self._h, out.ctypes.data, x.ctypes.data, x.shape[0]))
        return out

    def scheme_switch(self, glev) -> np.ndarray:
        """Evaluation::scheme_switch (evaluation.rs:231-240)."""
        x = self._in(glev, np.uint64, self.len_glev, "glev")
        out = np.empty((x.shape[0], self.len_ggsw), dtype=np.complex128)
        self._check(lib().spf_b200_scheme_switch(self._h, out.ctypes.data, x.ctypes.data, x.shape[0]))
        return out

    def trace(self, glwe) -> np.ndarray:
        """ops::automorphisms::trace (automorphisms/mod.rs:53-85)."""
        x = self._in(glwe, np.uint64, self.len_glwe, "glwe")
        out = np.empty_like(x)
        self._check(lib().spf_b200_trace(self._h, out.ctypes.data, x.ctypes.data, x.shape[0]))
        return out

    # -- KeylessEvaluation -----------------------------------------------------------------
    def cmux(self, sel, a, b) -> np.ndarray:
        """KeylessEvaluation::cmux(output, sel, a, b) (evaluation.rs:68-83): sel ? b : a."""
        s = self._in(sel, np.complex128, self.len_ggsw, "sel")
        a = self._in(a, np.uint64, self.len_glwe, "a")
        b = self._in(b, np.uint64, self.len_glwe, "b")
        if not (s.shape[0] == a.shape[0] == b.shape[0]):
            raise SpfError(-1, "cmux: batch sizes differ")
        out = np.empty_like(a)
        self._check(lib().spf_b200_cmux(self._h, out.ctypes.data, s.ctypes.data, a.ctypes.data, b.ctypes.data, a.shape[0]))
        return out

    def glev_cmux(self, sel, a, b) -> np.ndarray:
        """KeylessEvaluation::glev_cmux (evaluation.rs:86-101)."""
        s = self._in(sel, np.complex128, self.len_ggsw, "sel")
        a = self._in(a, np.uint64, self.len_glev, "a")
        b = self._in(b, np.uint64, self.len_glev, "b")
        if not (s.shape[0] == a.shape[0] == b.shape[0]):
            raise SpfError(-1, "glev_cmux: batch sizes differ")
        out = np.empty_like(a)
        self._check(lib().spf_b200_glev_cmux(self._h, out.ctypes.data, s.ctypes.data, a.ctypes.data, b.ctypes.data, a.shape[0]))
        return out

    def multiply_glwe_ggsw(self, glwe, ggsw) -> np.ndarray:
        """KeylessEvaluation::multiply_glwe_ggsw (evaluation.rs:104-123)."""
        g = self._in(glwe, np.uint64, self.len_glwe, "glwe")
        s = self._in(ggsw, np.complex128, self.len_ggsw, "ggsw")
        if g.shape[0] != s.shape[0]:
            raise SpfError(-1, "multiply_glwe_ggsw: batch sizes differ")
        out = np.empty_like(g)
        self._check(lib().spf_b200_multiply_glwe_ggsw(self._h, out.ctypes.data, g.ctypes.data, s.ctypes.data, g.shape[0]))
        return out

    def sample_extract_l1(self, glwe, idx) -> np.ndarray:
        """KeylessEvaluation::sample_extract_l1 (evaluation.rs:126-133); idx scalar or [batch]."""
        g = self._in(glwe, np.uint64, self.len_glwe, "glwe")
        out = np.empty((g.shape[0], self.len_lwe_l1), dtype=np.uint64)
        if np.isscalar(idx):
            rc = lib().spf_b200_sample_extract_l1(self._h, out.ctypes.data, g.ctypes.data, None, int(idx), g.shape[0])
        else:
            ix = np.ascontiguousarray(idx, dtype=np.uint32)
            if ix.shape != (g.shape[0],):
                raise SpfError(-1, "sample_extract_l1: idx must have one entry per ciphertext")
            rc = lib().spf_b200_sample_extract_l1(self._h, out.ctypes.data, g.ctypes.data, ix.ctypes.data, 0, g.shape[0])
        self._check(rc)
        return out

    def not_(self, glwe) -> np.ndarray:
        """KeylessEvaluation::not (evaluation.rs:48-50)."""
        g = self._in(glwe, np.uint64, self.len_glwe, "glwe")
        out = np.empty_like(g)
        self._check(lib().spf_b200_not(self._h, out.ctypes.data, g.ctypes.data, g.shape[0]))
        return out

    def xor(self, a, b) -> np.ndarray:
        """KeylessEvaluation::xor (evaluation.rs:53-55)."""
        a = self._in(a, np.uint64, self.len_glwe, "a")
        b = self._in(b, np.uint64, self.len_glwe, "b")
        if a.shape != b.shape:
            raise SpfError(-1, "xor: batch sizes differ")
        out = np.empty_like(a)
        self._check(lib().spf_b200_xor(self._h, out.ctypes.data, a.ctypes.data, b.ctypes.data, a.shape[0]))
        return out

    def mul_xn(self, glwe, n: int) -> np.ndarray:
        """KeylessEvaluation::mul_xn (evaluation.rs:58-65)."""
        g = self._in(glwe, np.uint64, self.len_glwe, "glwe")
        out = np.empty_like(g)
        self._check(lib().spf_b200_mul_xn(self._h, out.ctypes.data, g.ctypes.data, int(n), g.shape[0]))
        return out

    def rlwe_encrypt_public(self, public_key, encoded_msg, u, e0, e1) -> np.ndarray:
        """Encryption::encrypt_rlwe_l1 / rlwe_encrypt_public (encryption.rs:205-215, rlwe_encryption.rs:108-160) with the
        randomness (binary u, Gaussian e0 / e1) supplied by the caller: (p0 u + e0, p1 u + e1 + m), exact u64 arithmetic."""
        n = self.params.glwe_n
        pk = np.ascontiguousarray(public_key, dtype=np.uint64).reshape(-1)
        if pk.shape[0] != self.len_glwe:
            raise SpfError(-1, f"public_key: expected {self.len_glwe} u64, got {pk.shape[0]}")
        m = self._in(encoded_msg, np.uint64, n, "encoded_msg")
        uu, a0, a1 = (self._in(x, np.uint64, n, nm) for x, nm in ((u, "u"), (e0, "e0"), (e1, "e1")))
        if not (m.shape == uu.shape == a0.shape == a1.shape):
            raise SpfError(-1, "rlwe_encrypt_public: batch sizes differ")
        out = np.empty((m.shape[0], self.len_glwe), dtype=np.uint64)
        self._check(lib().spf_b200_rlwe_encrypt_public(self._h, out.ctypes.data, pk.ctypes.data, m.ctypes.data,
                                                       uu.ctypes.data, a0.ctypes.data, a1.ctypes.data, m.shape[0]))
        return out

    # -- device-pointer entry points (ints = CUdeviceptr), asynchronous on `stream` ----------
    def dev_circuit_bootstrap(self, d_ggsw_out: int, d_lwe0_in: int, batch: int, reference_scale: bool = False,
                              stream: int = 0):
        self._check(lib().spf_b200_dev_circuit_bootstrap(self._h, d_ggsw_out, d_lwe0_in, batch,
                                                         1 if reference_scale else 0, stream or None))

    def dev_programmable_bootstrap(self, d_glwe_out: int, d_lwe0_in: int, d_lut: int, log_chi: int, log_v: int,
                                   batch: int, stream: int = 0):
        self._check(lib().spf_b200_dev_programmable_bootstrap(self._h, d_glwe_out, d_lwe0_in, d_lut, log_chi, log_v,
                                                              batch, stream or None))

    def dev_cmux(self, d_out: int, d_sel: int, ggsw_stride: int, d_a: int, d_b: int, batch: int, stream: int = 0):
        self._check(lib().spf_b200_dev_cmux(self._h, d_out, d_sel, ggsw_stride, d_a, d_b, batch, stream or None))

    def dev_keyswitch_lwe_l1_lwe_l0(self, d_out: int, d_in: int, batch: int, stream: int = 0):
        self._check(lib().spf_b200_dev_keyswitch_lwe_l1_lwe_l0(self._h, d_out, d_in, batch, stream or None))

    def dev_sample_extract_l1(self, d_out: int, d_glwe: int, d_idx: int, idx_all: int, batch: int, stream: int = 0):
        self._check(lib().spf_b200_dev_sample_extract_l1(self._h, d_out, d_glwe, d_idx or None, idx_all, batch,
                                                         stream or None))

    def dev_rlwe_encrypt_public(self, d_out: int, d_pk: int, d_msg: int, d_u: int, d_e0: int, d_e1: int, batch: int,
                                stream: int = 0):
        self._check(lib().spf_b200_dev_rlwe_encrypt_public(self._h, d_out, d_pk, d_msg, d_u, d_e0, d_e1, batch,
                                                           stream or None))

    def dev_fft_rescale(self, d_dst: int, d_src: int, n: int, to_device: bool, stream: int = 0):
        self._check(lib().spf_b200_dev_fft_rescale(self._h, d_dst, d_src, n, 1 if to_device else 0, stream or None))


# ---------------------------------------------------------------------------------------------
# Graph execution: FheCircuit + CircuitProcessor::run_graph_blocking
# ---------------------------------------------------------------------------------------------
class _Node(C.Structure):
    _fields_ = [("op", C.c_uint32), ("arg", C.c_uint32), ("inp", C.c_int32 * 3), ("io", C.c_void_p)]


# FheOp (parasol_runtime/src/fhe_circuit.rs:34-127), same order as spf_op in include/spf_b200.h
OPS = ["InputLwe0", "InputLwe1", "InputGlwe1", "InputGgsw1", "InputGlev1", "OutputLwe0", "OutputLwe1", "OutputGlwe1",
       "OutputGgsw1", "OutputGlev1", "SampleExtract", "KeyswitchL1toL0", "Not", "GlweAdd", "CMux", "GlevCMux",
       "MultiplyGgswGlwe", "CircuitBootstrap", "SchemeSwitch", "ZeroLwe0", "OneLwe0", "ZeroGlwe1", "OneGlwe1",
       "ZeroGgsw1", "OneGgsw1", "ZeroGlev1", "OneGlev1", "Retire", "Nop", "MulXN"]
OP = {name: i for i, name in enumerate(OPS)}

ABI.update({
    "spf_b200_graph_build": [_vp, C.POINTER(_Node), _sz, C.POINTER(_vp)],
    "spf_b200_graph_run": [_vp],
    "spf_b200_graph_destroy": [_vp],
    "spf_b200_graph_levels": [_vp],
    "spf_b200_graph_launches": [_vp],
    "spf_b200_run_graph": [_vp, C.POINTER(_Node), _sz],
    "spf_b200_graph_set_io": [_vp, _sz, _vp],
    "spf_b200_graph_build_sharded": [_vp, C.POINTER(_Node), _sz, C.c_int, C.POINTER(_vp)],
    "spf_b200_graph_run_sharded": [_vp, C.c_int, C.c_int, _vp, _vp],
    "spf_b200_graph_output_rank": [_vp, _sz],
    "spf_b200_host_alloc": [C.POINTER(_vp), _sz],
    "spf_b200_host_free": [_vp],
    "spf_b200_graph_arena": [_vp],
    "spf_b200_graph_ipc_handle": [_vp, _vp],
    "spf_b200_graph_open_peers": [_vp, C.c_int, C.c_int, _vp],
    "spf_b200_graph_set_peers": [_vp, C.c_int, C.c_int, C.POINTER(_vp)],
    "spf_b200_graph_plan": [C.POINTER(Params), C.POINTER(_Node), _sz, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32)],
    "spf_b200_graph_spawn": [_vp, C.POINTER(_vp), _sz, _vp, _vp],
    "spf_b200_graph_wait": [_vp],
    "spf_b200_graph_status_message": [_vp],
    "spf_b200_set_max_in_flight": [_vp, C.c_int],
    "spf_b200_device_alloc": [_vp, C.POINTER(_vp), _sz],
    "spf_b200_device_free": [_vp, _vp],
})
# spf_completion_fn(user, status, message)
COMPLETION_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_char_p)


class _MuxNode(C.Structure):
    """spf_mux_node (include/spf_b200.h): one node of a generated MUX circuit."""
    _fields_ = [("op", C.c_uint32), ("arg", C.c_uint32), ("sel", C.c_int32), ("low", C.c_int32), ("high", C.c_int32)]


ABI.update({
    "spf_b200_mux_circuit": [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.POINTER(_MuxNode)), C.POINTER(_sz)],
    "spf_b200_mux_free": [C.POINTER(_MuxNode)],
})
_RESTYPES["spf_b200_mux_free"] = None
# spf_exchange_fn(user, d_buf, chunk_bytes, world, stream) -> int
EXCHANGE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p)
_RESTYPES.update({"spf_b200_graph_destroy": None, "spf_b200_graph_launches": C.c_uint64, "spf_b200_graph_arena": _vp,
                  "spf_b200_graph_status_message": C.c_char_p})

# one process, every GPU of a box (spf_b200_box_*)
ABI.update({
    "spf_b200_box_create": [C.POINTER(Params), _vp, _sz, _vp, _sz, _vp, _sz, _vp, _sz, C.POINTER(C.c_int), C.c_int,
                            C.POINTER(_vp)],
    "spf_b200_box_create_from_serialized": [C.POINTER(Params), _vp, _sz, C.POINTER(C.c_int), C.c_int, C.POINTER(_vp)],
    "spf_b200_box_destroy": [_vp],
    "spf_b200_box_last_error": [_vp],
    "spf_b200_box_size": [_vp],
    "spf_b200_box_device": [_vp, C.c_int],
    "spf_b200_box_context": [_vp, C.c_int],
    "spf_b200_box_key_replication_ms": [_vp],
    "spf_b200_box_key_slice": [_vp, C.c_int, C.c_int, _sz, _sz, _vp],
    "spf_b200_box_shard": [_sz, C.c_int, C.c_int, C.POINTER(_sz), C.POINTER(_sz)],
    "spf_b200_box_circuit_bootstrap": [_vp, _vp, _vp, _sz],
    "spf_b200_box_programmable_bootstrap": [_vp, _vp, _vp, _vp, C.c_uint32, C.c_uint32, _sz],
    "spf_b200_box_keyswitch_lwe_l1_lwe_l0": [_vp, _vp, _vp, _sz],
    "spf_b200_box_cmux": [_vp, _vp, _vp, _vp, _vp, _sz],
    "spf_b200_box_graph_build": [_vp, C.POINTER(_Node), _sz, C.POINTER(_vp)],
    "spf_b200_box_graph_build_on": [_vp, C.POINTER(_Node), _sz, C.POINTER(C.c_int), C.c_int, C.POINTER(_vp)],
    "spf_b200_box_graph_ranks": [_vp, C.POINTER(C.c_int)],
    "spf_b200_box_graph_run": [_vp],
    "spf_b200_box_graph_spawn": [_vp, C.POINTER(_vp), _sz, _vp, _vp],
    "spf_b200_box_graph_wait": [_vp],
    "spf_b200_box_graph_status_message": [_vp],
    "spf_b200_box_graph_set_io": [_vp, _sz, _vp],
    "spf_b200_box_graph_destroy": [_vp],
    "spf_b200_box_graph_levels": [_vp],
    "spf_b200_box_graph_launches": [_vp],
    "spf_b200_box_set_max_in_flight": [_vp, C.c_int],
    "spf_b200_box_ciphertext_alloc": [_vp, C.c_uint32, C.POINTER(_vp)],
    "spf_b200_box_ciphertext_free": [_vp],
    "spf_b200_box_ciphertext_write": [_vp, _vp],
    "spf_b200_box_ciphertext_read": [_vp, C.c_int, _vp],
})
_RESTYPES.update({"spf_b200_box_destroy": None, "spf_b200_box_last_error": C.c_char_p, "spf_b200_box_context": _vp,
                  "spf_b200_box_key_replication_ms": C.c_double, "spf_b200_box_shard": None,
                  "spf_b200_box_graph_status_message": C.c_char_p, "spf_b200_box_graph_destroy": None,
                  "spf_b200_box_graph_launches": C.c_uint64, "spf_b200_box_ciphertext_free": None})


class DeviceCiphertext:
    """A ciphertext HANDLE: `nbytes` of device memory holding one ciphertext that never leaves HBM (the role of the
    reference's Arc<AtomicRefCell<Option<Ciphertext>>> task outputs shared between graphs, circuit_processor/task.rs:10-16).
    Pass it as the `io` of an Output* node of one graph and of an Input* node of the next.  GGSWs behind a handle are in
    the device scale.  Wraps a raw pointer (`ptr`), a torch CUDA tensor, or allocates (`DeviceCiphertext.alloc`)."""

    def __init__(self, ptr, nbytes: int | None = None, owner=None):
        if hasattr(ptr, "data_ptr"):  # torch tensor
            owner, nbytes, ptr = ptr, ptr.numel() * ptr.element_size(), ptr.data_ptr()
        self.ptr, self.nbytes, self._owner = int(ptr), int(nbytes), owner

    @classmethod
    def alloc(cls, ev: "Evaluation", nbytes: int) -> "DeviceCiphertext":
        import weakref

        p = _vp()
        ev._check(lib().spf_b200_device_alloc(ev.handle, C.byref(p), nbytes))
        h = cls(p.value, nbytes, owner=ev)
        weakref.finalize(h, lib().spf_b200_device_free, ev.handle, p.value)
        return h


class BoxCiphertext:
    """A box ciphertext HANDLE (spf_b200_box_ciphertext_*): one ciphertext kept in HBM with one replica per rank of a
    BoxEvaluation -- the box's DeviceCiphertext.  Pass it as the `io` of an Output* node of one box graph and of an
    Input* node of the next; `ptr` is the handle address, `nbytes` the ciphertext size.  GGSWs stay in the device scale
    in the replicas; write() takes and read() returns the reference scale.  close() (or garbage collection) drops this
    reference: box graphs that still bind the handle keep its memory until they are closed or rebound."""

    def __init__(self, box: "BoxEvaluation", kind: str, ptr: int):
        import weakref

        self.box, self.kind, self.ptr = box, kind, int(ptr)
        self._box_ptr = box.handle.value  # the handle keeps the box's error slot alive, also after box.close()
        self.nbytes = io_bytes(kind, box.params)
        self._free = weakref.finalize(self, lib().spf_b200_box_ciphertext_free, self.ptr)

    @classmethod
    def alloc(cls, box: "BoxEvaluation", kind: str) -> "BoxCiphertext":
        """A zero-filled handle for a ciphertext of `kind` ("Lwe0", "Lwe1", "Glwe1", "Ggsw1" or "Glev1")."""
        if kind not in _IO_KIND:
            raise SpfError(-1, f"BoxCiphertext: unknown kind {kind!r}, expected one of {sorted(_IO_KIND)}")
        h = _vp()
        box._check(lib().spf_b200_box_ciphertext_alloc(box.handle, OP["Input" + kind], C.byref(h)))
        return cls(box, kind, h.value)

    def _array(self):
        return np.empty(self.nbytes // 16, np.complex128) if self.kind == "Ggsw1" else np.empty(self.nbytes // 8, np.uint64)

    def _check(self, rc: int):
        if rc != 0:
            raise SpfError(rc, (lib().spf_b200_box_last_error(self._box_ptr) or b"").decode())

    def _live(self):
        if not self._free.alive:
            raise SpfError(-1, "BoxCiphertext is closed")
        return self.ptr

    def write(self, arr) -> None:
        """Host ciphertext (reference layout and scale) -> every rank's replica."""
        a = np.ascontiguousarray(arr)
        dtypes = (np.dtype(np.complex128), np.dtype(np.float64)) if self.kind == "Ggsw1" else (np.dtype(np.uint64),)
        if a.dtype not in dtypes or a.nbytes != self.nbytes:
            raise SpfError(-1, f"BoxCiphertext.write: a {self.kind} ciphertext is {self.nbytes} bytes of {dtypes[0]}, "
                               f"got {a.nbytes} bytes of {a.dtype}")
        self._check(lib().spf_b200_box_ciphertext_write(self._live(), a.ctypes.data))

    def read(self, rank: int = 0) -> np.ndarray:
        """Rank `rank`'s replica, in the reference layout and scale."""
        out = self._array()
        self._check(lib().spf_b200_box_ciphertext_read(self._live(), int(rank), out.ctypes.data))
        return out

    def close(self) -> None:
        self._free()


def _io_ptr(io) -> int:
    return io.ptr if isinstance(io, (DeviceCiphertext, BoxCiphertext)) else io.ctypes.data


def _io_nbytes(io) -> int:
    return io.nbytes


# bytes of the ciphertext behind an Input* / Output* node at DEFAULT_128-style params: op name -> length function, element size
_IO_KIND = {"Lwe0": ("spf_b200_len_lwe_l0", 8), "Lwe1": ("spf_b200_len_lwe_l1", 8), "Glwe1": ("spf_b200_len_glwe_l1", 8),
            "Ggsw1": ("spf_b200_len_ggsw_l1", 16), "Glev1": ("spf_b200_len_glev_l1", 8)}


def io_bytes(op: str, params: "Params | None" = None) -> int:
    """Size in bytes of the buffer an Input* / Output* node reads or writes (spf_node carries no length: the executor
    DMAs exactly this many bytes through the raw pointer, so the host mirror checks it)."""
    kind = op.replace("Input", "").replace("Output", "")
    fn, elem = _IO_KIND[kind]
    p = params or default_128()
    return int(getattr(lib(), fn)(C.byref(p))) * elem


class FheCircuit:
    """A DAG of FheOp nodes (parasol_runtime/src/fhe_circuit.rs:205-208).  Edges are given when the
    consumer is added, by the reference's FheEdge names: unary ops take `x`; GlweAdd takes
    (left, right); CMux / GlevCMux take (sel, low, high); MultiplyGgswGlwe takes (glwe, ggsw).
    Input / Output nodes carry the numpy buffer they read from / write into."""

    _DT = np.dtype([("op", "<u4"), ("arg", "<u4"), ("inp", "<i4", (3,)), ("pad", "<u4"), ("io", "<u8")])  # spf_node

    def __init__(self, params: "Params | None" = None):
        self.params = params      # io buffer sizes are checked against these (default: DEFAULT_128)
        self._n = 0
        self._buf = np.zeros(64, dtype=self._DT)   # node table in the C ABI's layout, grown geometrically
        self._buf["inp"] = -1
        self._io: dict[int, np.ndarray] = {}      # node -> host buffer (kept alive here)

    def __len__(self) -> int:
        return self._n

    def _reserve(self, extra: int) -> None:
        if self._n + extra > len(self._buf):
            grown = np.zeros(max(2 * len(self._buf), self._n + extra), dtype=self._DT)
            grown["inp"] = -1
            grown[:self._n] = self._buf[:self._n]
            self._buf = grown

    def add(self, op: str, *inputs: int, arg: int = 0, io: np.ndarray | None = None) -> int:
        return self._append(OP[op], int(arg), tuple(inputs) + (-1,) * (3 - len(inputs)), io)

    def _check_io(self, opc: int, io) -> None:
        """An io buffer must hold exactly one ciphertext of the node's kind: the executor copies that many bytes
        through the raw pointer whatever the array's size (the reference is type-safe at this seam)."""
        if not isinstance(io, (DeviceCiphertext, BoxCiphertext)):
            if not isinstance(io, np.ndarray) or not io.flags["C_CONTIGUOUS"]:
                raise SpfError(-1, "io buffers must be C-contiguous numpy arrays, DeviceCiphertext or BoxCiphertext handles")
        name = OPS[opc]
        if not (name.startswith("Input") or name.startswith("Output")):
            raise SpfError(-1, f"{name} takes no io buffer")
        if isinstance(io, BoxCiphertext) and name.replace("Input", "").replace("Output", "") != io.kind:
            raise SpfError(-1, f"{name}: the BoxCiphertext holds a {io.kind} ciphertext")
        want = io_bytes(name, self.params)
        if _io_nbytes(io) != want:
            raise SpfError(-1, f"{name}: io buffer has {_io_nbytes(io)} bytes, the ciphertext has {want}")
        if isinstance(io, np.ndarray):
            ok = io.dtype in (np.dtype(np.complex128), np.dtype(np.float64)) if name.endswith("Ggsw1") else io.dtype == np.dtype(np.uint64)
            if not ok:
                raise SpfError(-1, f"{name}: io buffer has dtype {io.dtype}")

    def _append(self, opc: int, arg: int, ins, io) -> int:
        if io is not None:
            self._check_io(opc, io)
        self._reserve(1)
        i = self._n
        row = self._buf[i]
        row["op"], row["arg"], row["inp"] = opc, arg, ins
        if io is not None:
            self._io[i] = io
        self._n += 1
        return i

    def add_block(self, opcodes: np.ndarray, ins: np.ndarray) -> np.ndarray:
        """Append len(opcodes) nodes at once (opcodes: op codes, ins: [m, 3] producer indices, -1 = none) and
        return their indices -- the bulk path MUX-circuit expansion uses (tens of thousands of CMux nodes)."""
        m = len(opcodes)
        self._reserve(m)
        blk = self._buf[self._n:self._n + m]
        blk["op"], blk["arg"], blk["inp"] = opcodes, 0, ins
        self._n += m
        return np.arange(self._n - m, self._n, dtype=np.int64)

    @property
    def nodes(self) -> "_NodesView":
        """Sequence view of the nodes as (op code, arg, (in0, in1, in2), io buffer) tuples."""
        return _NodesView(self)

    @property
    def ops(self) -> np.ndarray:
        return self._buf["op"][:self._n]

    @property
    def inputs_of(self) -> np.ndarray:
        return self._buf["inp"][:self._n]

    def _pack(self):
        """The node table as the C ABI wants it (spf_node[]); io pointers are filled in here."""
        arr = self._buf[:max(self._n, 1)].copy()
        arr["io"] = 0
        for i, io in self._io.items():
            arr["io"][i] = _io_ptr(io)
        self._packed = arr  # keeps the memory alive for the duration of the call
        return arr.ctypes.data_as(C.POINTER(_Node))


class _NodesView:
    """list-like read view (plus append) over a FheCircuit's node table."""

    def __init__(self, c: FheCircuit):
        self._c = c

    def __len__(self):
        return self._c._n

    def __getitem__(self, i: int):
        c = self._c
        if i < 0:
            i += c._n
        if not 0 <= i < c._n:
            raise IndexError(i)
        row = c._buf[i]
        return int(row["op"]), int(row["arg"]), tuple(int(x) for x in row["inp"]), c._io.get(i)

    def __iter__(self):
        c = self._c
        ops, args, ins = c._buf["op"][:c._n].tolist(), c._buf["arg"][:c._n].tolist(), c._buf["inp"][:c._n].tolist()
        for i in range(c._n):
            yield ops[i], args[i], tuple(ins[i]), c._io.get(i)

    def append(self, node) -> None:
        opc, arg, ins, io = node
        self._c._append(int(opc), int(arg), tuple(ins), io)


def pinned_zeros(shape, dtype=np.uint64) -> np.ndarray:
    """A zeroed numpy array in page-locked host memory (ONE slab: slice it into ciphertext buffers).  Graph IO
    from such buffers is a DMA without per-buffer registration; the memory is released with the array."""
    import weakref

    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    ptr = _vp()
    rc = lib().spf_b200_host_alloc(C.byref(ptr), max(nbytes, 1))
    if rc:
        raise SpfError(rc, (lib().spf_b200_last_error(None) or b"").decode())
    buf = (C.c_uint8 * max(nbytes, 1)).from_address(ptr.value)
    weakref.finalize(buf, lib().spf_b200_host_free, ptr.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    arr[...] = 0
    return arr


def plan_graph(circuit: "FheCircuit", world: int = 1, params: Params | None = None) -> tuple[np.ndarray, np.ndarray]:
    """Host-only schedule of a graph (no GPU): (level, owner) per node -- the dependency level after
    bootstrap-stage alignment and, for a run sharded over `world` ranks, the rank that computes the node
    (-1: every rank).  Raises SpfError(-4, ...) for malformed graphs like CircuitProcessor.run_graph_blocking."""
    p = params or default_128()
    n = len(circuit.nodes)
    level, owner = np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1), np.int32)
    rc = lib().spf_b200_graph_plan(C.byref(p), circuit._pack(), n, world, level.ctypes.data_as(C.POINTER(C.c_int32)),
                                   owner.ctypes.data_as(C.POINTER(C.c_int32)))
    if rc:
        raise SpfError(rc, (lib().spf_b200_last_error(None) or b"").decode())
    return level[:n], owner[:n]


class CircuitProcessor:
    """CircuitProcessor (parasol_runtime/src/circuit_processor/mod.rs:62-655) on the GPU: a graph is
    compiled once into per-level batched launches and can be run repeatedly.  On a BoxEvaluation every graph runs
    over all GPUs of the box (BoxGraph) from the calling thread, or over the box ranks named in `ranks`."""

    def __init__(self, evaluation: "Evaluation | BoxEvaluation"):
        self.ev = evaluation

    def compile(self, circuit: FheCircuit, world: int = 1, rank: int = 0, exchange=None,
                ranks=None) -> "CompiledGraph | BoxGraph":
        if isinstance(self.ev, BoxEvaluation):
            if world != 1 or rank != 0 or exchange is not None:
                raise SpfError(-1, "a box graph is sharded over the box's ranks: world / rank / exchange do not apply")
            return BoxGraph(self.ev, circuit, ranks=ranks)
        if ranks is not None:
            raise SpfError(-1, "ranks place a graph on ranks of a BoxEvaluation; this evaluation is a single context")
        return CompiledGraph(self.ev, circuit, world=world, rank=rank, exchange=exchange)

    def run_graph_blocking(self, circuit: FheCircuit) -> None:
        """run_graph_blocking (mod.rs:641-655); raises SpfError(-4, ...) for malformed graphs as the
        reference returns Err(RuntimeError)."""
        g = self.compile(circuit)
        try:
            g.run()
        finally:
            g.close()

    def spawn_graph(self, circuit: FheCircuit, on_completion=None, after=(), ranks=None) -> "CompiledGraph":
        """spawn_graph (mod.rs:573-623): dispatches the graph and returns; `on_completion(error)` is called once when all
        of its ops have retired, with None or the first SpfError (CompletionHandler, completion_handler.rs:14-56) --
        validation errors included, as in the reference.  Outputs must not be read before.  Returns the compiled graph:
        pass it in `after` of a later spawn that consumes this one's DeviceCiphertext outputs, and close() it after
        wait().  `ranks` (BoxEvaluation only): the box ranks the graph runs on, as in BoxGraph."""
        try:
            g = self.compile(circuit, ranks=ranks)
        except SpfError as e:
            if on_completion is None:
                raise
            on_completion(e)
            return None
        g.spawn(after=after, on_complete=on_completion)
        return g


def _spawn(graph, spawn_fn, after, on_complete) -> None:
    """One asynchronous run of a CompiledGraph or BoxGraph through its spawn entry point: `after` and `on_complete` as
    in CompiledGraph.spawn."""
    deps = [d for d in after if d is not None]
    arr = (_vp * max(len(deps), 1))(*[d._h for d in deps])

    def _done(user, status, message):
        try:
            if on_complete is not None:
                on_complete(None if status == 0 else SpfError(int(status), (message or b"").decode()))
        except Exception:  # never let an exception cross the C ABI
            pass

    graph._spawn_cb = COMPLETION_FN(_done)  # kept alive until the next spawn / close
    graph.ev._check(spawn_fn(graph._h, arr, len(deps), C.cast(graph._spawn_cb, _vp), None))


def _wait(graph, wait_fn, message_fn) -> None:
    """Blocks until the graph's last run is over; raises its error, if any."""
    rc = wait_fn(graph._h)
    if rc:
        raise SpfError(int(rc), (message_fn(graph._h) or b"").decode() or "the graph's last run failed")


class CompiledGraph:
    """A levelised graph resident on one GPU.  With world > 1 the graph is laid out for a sharded
    run (spf_b200_graph_build_sharded): every CircuitBootstrap level is split into `world` chunks,
    this rank computes chunk `rank` and `exchange(d_buf, chunk_bytes, world, stream)` (see
    spf_b200.multi.NcclExchange) all-gathers the rest."""

    def __init__(self, ev: Evaluation, circuit: FheCircuit, world: int = 1, rank: int = 0, exchange=None):
        self.ev = ev
        self._keep = circuit  # keeps the io buffers alive
        self._h = _vp()
        self.world, self.rank = int(world), int(rank)
        arr = circuit._pack()
        ev._check(lib().spf_b200_graph_build_sharded(ev.handle, arr, len(circuit.nodes), self.world, C.byref(self._h)))
        self._exchange = exchange
        self._cb_error = None
        self._peers = False

        def _cb(user, d_buf, chunk_bytes, world_, stream):
            try:
                self._exchange(int(d_buf), int(chunk_bytes), int(world_), int(stream or 0))
                return 0
            except Exception as e:  # never let an exception cross the C ABI
                self._cb_error = e
                return 1

        self._cb = EXCHANGE_FN(_cb) if exchange is not None else None

    def run(self):
        if self.world == 1:
            self.ev._check(lib().spf_b200_graph_run(self._h))
            return
        if self._cb is None:
            if not self._peers:
                raise SpfError(-1, "a sharded graph needs an exchange callable or opened peer arenas")
            self.ev._check(lib().spf_b200_graph_run_sharded(self._h, self.rank, self.world, None, None))
            return
        self._cb_error = None
        rc = lib().spf_b200_graph_run_sharded(self._h, self.rank, self.world, C.cast(self._cb, _vp), None)
        if self._cb_error is not None:
            raise self._cb_error
        self.ev._check(rc)

    def set_io(self, node: int, buf) -> None:
        """Re-point an Input*/Output* node at another buffer of the same ciphertext kind (a numpy array -- page-locked
        or pageable -- or a DeviceCiphertext handle): a compiled graph is reusable across invocations of the same
        instruction shape."""
        if not 0 <= node < len(self._keep):
            raise SpfError(-1, f"set_io: node {node} out of range")
        if isinstance(buf, BoxCiphertext):
            raise SpfError(-1, "set_io: a BoxCiphertext is the io of box graphs only (BoxGraph)")
        self._keep._check_io(int(self._keep.ops[node]), buf)
        self.ev._check(lib().spf_b200_graph_set_io(self._h, node, _io_ptr(buf)))
        self._bound = getattr(self, "_bound", {})
        self._bound[node] = buf  # keep alive

    def spawn(self, after=(), on_complete=None) -> None:
        """One asynchronous run (spf_b200_graph_spawn): returns as soon as the work is enqueued (or blocks while the
        context's flow-control limit of in-flight graphs is reached).  `after`: CompiledGraphs whose last spawned run must
        finish first (ordered on the device).  on_complete(error) is called from a CUDA callback thread with None or
        the first SpfError of the run; it must not call into spf_b200 or CUDA."""
        if self.world != 1:
            raise SpfError(-1, "sharded graphs are not spawned")
        _spawn(self, lib().spf_b200_graph_spawn, after, on_complete)

    def wait(self) -> None:
        """Block until the last run (spawned or blocking) is over; raises its error, if any."""
        _wait(self, lib().spf_b200_graph_wait, lib().spf_b200_graph_status_message)

    # ---- peer-memory exchange (no exchange callable): every rank maps every other rank's arena ----
    @property
    def arena(self) -> int:
        return int(lib().spf_b200_graph_arena(self._h) or 0)

    def ipc_handle(self) -> bytes:
        """64-byte cudaIpcMemHandle_t of this graph's arena, to be gathered over all ranks."""
        buf = (C.c_uint8 * 64)()
        self.ev._check(lib().spf_b200_graph_ipc_handle(self._h, buf))
        return bytes(buf)

    def open_peers(self, handles: list[bytes]) -> None:
        """handles[r] = rank r's ipc_handle(); afterwards run() exchanges over peer memory (NVLink P2P)."""
        if len(handles) != self.world or any(len(h) != 64 for h in handles):
            raise SpfError(-1, "open_peers: one 64-byte handle per rank")
        blob = (C.c_uint8 * (64 * self.world)).from_buffer_copy(b"".join(handles))
        self.ev._check(lib().spf_b200_graph_open_peers(self._h, self.rank, self.world, blob))
        self._peers = True

    def set_peers(self, arenas: list[int]) -> None:
        """Same-process variant (tests): arenas[r] = CompiledGraph.arena of rank r's graph."""
        arr = (_vp * self.world)(*arenas)
        self.ev._check(lib().spf_b200_graph_set_peers(self._h, self.rank, self.world, arr))
        self._peers = True

    def output_rank(self, node: int) -> int:
        """Rank whose run() writes Output* node `node` (-1: every rank).  In a sharded run the outputs of
        a MUX tree are delivered on the rank that owns the tree."""
        r = int(lib().spf_b200_graph_output_rank(self._h, node))
        if r == -2:
            raise SpfError(-1, f"node {node} is not an Output* node")
        return r

    @property
    def levels(self) -> int:
        return int(lib().spf_b200_graph_levels(self._h))

    @property
    def launches(self) -> int:
        return int(lib().spf_b200_graph_launches(self._h))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().spf_b200_graph_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---------------------------------------------------------------------------------------------
# One process, every GPU of a box: BoxEvaluation + BoxGraph (spf_b200_box_*)
# ---------------------------------------------------------------------------------------------
def box_shard(batch: int, n: int, rank: int) -> tuple[int, int]:
    """(start, count) of rank `rank`'s slice of a batch in the box ops (spf_b200_box_shard; multi.shard's rule)."""
    start, count = _sz(), _sz()
    lib().spf_b200_box_shard(int(batch), int(n), int(rank), C.byref(start), C.byref(count))
    return int(start.value), int(count.value)


class BoxEvaluation:
    """`Evaluation` over several GPUs of one box, from one thread: rank r is a context on devices[r] (a device may
    repeat).  The compute key is uploaded once and replicated device to device.  The batched ops split the batch
    contiguously over the ranks (box_shard) and run every rank at once; CircuitProcessor(box) runs graphs over all
    ranks.  Single-device work goes through the rank contexts (`contexts`)."""

    _in = staticmethod(Evaluation._in)

    def __init__(self, bsk_fft, ksk, ssk_fft, ak_fft, devices=(0,), params: Params | None = None):
        l = lib()
        self.params = params if params is not None else default_128()
        p = self.params
        self._h = _vp()
        lens = (l.spf_b200_len_bsk(C.byref(p)), l.spf_b200_len_ksk(C.byref(p)), l.spf_b200_len_ssk(C.byref(p)),
                l.spf_b200_len_ak(C.byref(p)))
        arrs = []
        for a, dt, n, name in ((bsk_fft, np.complex128, lens[0], "bs_key"), (ksk, np.uint64, lens[1], "ks_key"),
                               (ssk_fft, np.complex128, lens[2], "ss_key"), (ak_fft, np.complex128, lens[3], "auto_key")):
            a = np.ascontiguousarray(a, dtype=dt).reshape(-1)
            if a.size != n:
                raise SpfError(-1, f"{name} has {a.size} elements, params require {n}")
            arrs.append(a)
        devs = self._devices(devices)
        self._check_create(l.spf_b200_box_create(C.byref(p), arrs[0].ctypes.data, lens[0], arrs[1].ctypes.data, lens[1],
                                                 arrs[2].ctypes.data, lens[2], arrs[3].ctypes.data, lens[3], devs,
                                                 len(devs), C.byref(self._h)))
        self._init_lengths()

    @staticmethod
    def _devices(devices):
        devices = [int(d) for d in devices]
        return (C.c_int * max(len(devices), 1))(*devices)

    def _check_create(self, rc):
        if rc != 0:
            raise SpfError(rc, (lib().spf_b200_box_last_error(None) or b"").decode())

    def _init_lengths(self):
        l, p = lib(), self.params
        self.len_lwe_l0 = l.spf_b200_len_lwe_l0(C.byref(p))
        self.len_lwe_l1 = l.spf_b200_len_lwe_l1(C.byref(p))
        self.len_glwe = l.spf_b200_len_glwe_l1(C.byref(p))
        self.len_glev = l.spf_b200_len_glev_l1(C.byref(p))
        self.len_ggsw = l.spf_b200_len_ggsw_l1(C.byref(p))

    @classmethod
    def from_serialized(cls, data: bytes, params: Params | None = None, devices=(0,)) -> "BoxEvaluation":
        """safe_bincode::deserialize::<ComputeKey> + a box over `devices` (spf_b200_box_create_from_serialized)."""
        self = cls.__new__(cls)
        self.params = params if params is not None else default_128()
        self._h = _vp()
        buf = np.frombuffer(bytes(data), dtype=np.uint8)
        devs = cls._devices(devices)
        self._check_create(lib().spf_b200_box_create_from_serialized(C.byref(self.params), buf.ctypes.data, buf.size, devs,
                                                                     len(devs), C.byref(self._h)))
        self._init_lengths()
        return self

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().spf_b200_box_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise SpfError(rc, (lib().spf_b200_box_last_error(self._h) or b"").decode())

    @property
    def handle(self):
        return self._h

    @property
    def size(self) -> int:
        return int(lib().spf_b200_box_size(self._h))

    @property
    def devices(self) -> list[int]:
        return [int(lib().spf_b200_box_device(self._h, r)) for r in range(self.size)]

    @property
    def contexts(self) -> list[int]:
        """spf_b200_ctx* of every rank (owned by the box), for the dev_* entry points of that rank's device."""
        return [int(lib().spf_b200_box_context(self._h, r) or 0) for r in range(self.size)]

    @property
    def key_replication_ms(self) -> float:
        return float(lib().spf_b200_box_key_replication_ms(self._h))

    @property
    def kernel_launches(self) -> int:
        return sum(int(lib().spf_b200_kernel_launches(c)) for c in self.contexts)

    def key_slice(self, rank: int, which: int, offset: int, count: int) -> np.ndarray:
        """Elements [offset, offset + count) of key array `which` (0 bs_key, 1 ks_key, 2 ss_key, 3 auto_key) as resident
        on rank `rank`'s device, in the reference layout and scale."""
        out = np.empty(int(count), dtype=np.uint64 if which == 1 else np.complex128)
        self._check(lib().spf_b200_box_key_slice(self._h, int(rank), int(which), int(offset), int(count), out.ctypes.data))
        return out

    def synchronize(self):
        for c in self.contexts:
            rc = lib().spf_b200_synchronize(c)
            if rc:
                raise SpfError(rc, (lib().spf_b200_last_error(c) or b"").decode())

    def set_max_in_flight(self, n: int) -> None:
        """Flow control of spawned box graphs: at most n runs per box between dispatch and completion."""
        self._check(lib().spf_b200_box_set_max_in_flight(self._h, int(n)))

    def circuit_bootstrap(self, lwe0) -> np.ndarray:
        x = self._in(lwe0, np.uint64, self.len_lwe_l0, "lwe0")
        out = np.empty((x.shape[0], self.len_ggsw), dtype=np.complex128)
        self._check(lib().spf_b200_box_circuit_bootstrap(self._h, out.ctypes.data, x.ctypes.data, x.shape[0]))
        return out

    def programmable_bootstrap(self, lwe0, lut_glwe, log_chi: int = 0, log_v: int = 0) -> np.ndarray:
        x = self._in(lwe0, np.uint64, self.len_lwe_l0, "lwe0")
        lut = self._in(lut_glwe, np.uint64, self.len_glwe, "lut")
        out = np.empty((x.shape[0], self.len_glwe), dtype=np.uint64)
        self._check(lib().spf_b200_box_programmable_bootstrap(self._h, out.ctypes.data, x.ctypes.data, lut.ctypes.data,
                                                              log_chi, log_v, x.shape[0]))
        return out

    def keyswitch_lwe_l1_lwe_l0(self, lwe1) -> np.ndarray:
        x = self._in(lwe1, np.uint64, self.len_lwe_l1, "lwe1")
        out = np.empty((x.shape[0], self.len_lwe_l0), dtype=np.uint64)
        self._check(lib().spf_b200_box_keyswitch_lwe_l1_lwe_l0(self._h, out.ctypes.data, x.ctypes.data, x.shape[0]))
        return out

    def cmux(self, sel, a, b) -> np.ndarray:
        s = self._in(sel, np.complex128, self.len_ggsw, "sel")
        a = self._in(a, np.uint64, self.len_glwe, "a")
        b = self._in(b, np.uint64, self.len_glwe, "b")
        if not (s.shape[0] == a.shape[0] == b.shape[0]):
            raise SpfError(-1, "cmux: batch sizes differ")
        out = np.empty_like(a)
        self._check(lib().spf_b200_box_cmux(self._h, out.ctypes.data, s.ctypes.data, a.ctypes.data, b.ctypes.data, a.shape[0]))
        return out



class BoxGraph:
    """A graph over the ranks of a BoxEvaluation (spf_b200_box_graph_*), with the CompiledGraph surface: run, spawn,
    wait, set_io, levels, launches, close.  io buffers are host numpy arrays or BoxCiphertext handles of the same box
    (DeviceCiphertext handles are refused).  `ranks`: the box ranks the graph runs on, in member order (None: every
    rank in order); the graph is sharded over them as over a box of len(ranks) ranks.  Handle outputs still reach the
    replica of every rank of the box.  A graph that writes a handle another graph reads, on any rank, must be in that
    reader's `after` (and the reader in the writer's, when the writer runs later)."""

    def __init__(self, box: BoxEvaluation, circuit: FheCircuit, ranks=None):
        self.ev = box
        self._keep = circuit
        self._h = _vp()
        if ranks is None:
            box._check(lib().spf_b200_box_graph_build(box.handle, circuit._pack(), len(circuit.nodes), C.byref(self._h)))
            return
        try:
            rs = [operator.index(r) for r in ranks]
        except TypeError:
            raise SpfError(-1, f"BoxGraph: ranks must be a sequence of box rank numbers, got {ranks!r}") from None
        if any(not -2**31 <= r < 2**31 for r in rs):  # a C int each: no silent wrap-around into a valid rank
            raise SpfError(-1, f"BoxGraph: ranks {rs} are not ranks of a box")
        arr = (C.c_int * max(len(rs), 1))(*rs)
        box._check(lib().spf_b200_box_graph_build_on(box.handle, circuit._pack(), len(circuit.nodes), arr, len(rs),
                                                     C.byref(self._h)))

    def run(self) -> None:
        self.ev._check(lib().spf_b200_box_graph_run(self._h))

    def set_io(self, node: int, buf) -> None:
        if not 0 <= node < len(self._keep):
            raise SpfError(-1, f"set_io: node {node} out of range")
        self._keep._check_io(int(self._keep.ops[node]), buf)
        self.ev._check(lib().spf_b200_box_graph_set_io(self._h, node, _io_ptr(buf)))
        self._bound = getattr(self, "_bound", {})
        self._bound[node] = buf

    def spawn(self, after=(), on_complete=None) -> None:
        """One asynchronous run over all ranks; on_complete(error) fires once, after every rank has retired, from a CUDA
        callback thread (it must not call into spf_b200 or CUDA).  `after`: BoxGraphs of the same box."""
        _spawn(self, lib().spf_b200_box_graph_spawn, after, on_complete)

    def wait(self) -> None:
        _wait(self, lib().spf_b200_box_graph_wait, lib().spf_b200_box_graph_status_message)

    @property
    def levels(self) -> int:
        return int(lib().spf_b200_box_graph_levels(self._h))

    @property
    def launches(self) -> int:
        return int(lib().spf_b200_box_graph_launches(self._h))

    @property
    def ranks(self) -> list[int]:
        """The box ranks the graph runs on, in member order."""
        n = int(lib().spf_b200_box_graph_ranks(self._h, None))
        out = (C.c_int * max(n, 1))()
        lib().spf_b200_box_graph_ranks(self._h, out)
        return list(out[:n])

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().spf_b200_box_graph_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
