"""The exact regime (tests/exact_keys.py) on the CPU: with integer-polynomial keys, the oracle's C code, the kernel
bodies run by the host emulator and a plain numpy restatement agree BIT FOR BIT on blind rotations, traces and CMUXes of
arbitrary u64 inputs.  This is the premise of tests/test_gpu_exact.py, which compares the device kernels with the oracle
at that sharpness; here it is guarded where it can run anywhere.

The numpy restatement is the third witness: signed digits as in math/radix.rs, negacyclic products through np.fft, and
an assertion that every value before rounding lies within 2^-8 of an integer -- so the oracle is not the only evidence
that the regime is exact.
"""
import ctypes as C

import numpy as np
import pytest

import emu_util as E
from exact_keys import exact_ggsw, exact_keys, interleaved_masks, lwe_with_mask, random_u64

N = 2048
M64 = (1 << 64) - 1


@pytest.fixture(scope="module")
def xk(oracle):
    return exact_keys(0xE0AC7)


@pytest.fixture(scope="module")
def dev_bsk(xk):
    return E.to_device_scale(xk.bsk_fft)


# ---- numpy restatement ----------------------------------------------------------------------------------------------

def np_modulus_switch(x: int, log_chi: int, log_v: int, log_modulus: int = 12) -> int:
    """ops/ciphertext/lwe_ciphertext_ops.rs:129-142 on Python integers."""
    x = (x << log_chi) & M64
    shift = 64 - (log_modulus - log_v)
    rnd = (x >> (shift - 1)) & 1
    return (((x >> shift) + rnd) & ((1 << log_modulus) - 1)) << log_v


def np_monomial(p: np.ndarray, d: int) -> np.ndarray:
    """p * X^d in Z_{2^64}[X] / (X^N + 1), any integer d."""
    j = (np.arange(N) - d) % (2 * N)
    out = p[j % N].copy()
    out[j >= N] = np.uint64(0) - out[j >= N]
    return out


def np_signed_digits(x: np.ndarray, radix_log: int, count: int) -> list[np.ndarray]:
    """math/radix.rs:81-113: round x to its top radix_log * count bits, then signed digits in [-B/2, B/2), LSB first."""
    shift = 64 - radix_log * count
    s = [(int(v) >> shift) + ((int(v) >> (shift - 1)) & 1) for v in x]
    digits = []
    for _ in range(count):
        d = [v & ((1 << radix_log) - 1) for v in s]
        carry = [v >> (radix_log - 1) for v in d]
        digits.append(np.array([v - (c << radix_log) for v, c in zip(d, carry)], dtype=np.int64))
        s = [(v >> radix_log) + c for v, c in zip(s, carry)]
    return digits


_TWIST = np.exp(1j * np.pi * np.arange(N) / N)


def np_negacyclic_fft(p: np.ndarray) -> np.ndarray:
    return np.fft.fft(p.astype(np.float64) * _TWIST)


def np_negacyclic_ifft_exact(f: np.ndarray) -> np.ndarray:
    """Inverse of np_negacyclic_fft, rounded to integers mod 2^64 -- after asserting that every real part is within
    2^-8 of an integer (the exact regime) and every imaginary part within 2^-8 of 0."""
    z = np.fft.ifft(f) * np.conj(_TWIST)
    r = np.rint(z.real)
    assert np.abs(z.real - r).max() <= 2.0 ** -8 and np.abs(z.imag).max() <= 2.0 ** -8, "outside the exact regime"
    assert np.abs(r).max() < 2.0 ** 53
    return r.astype(np.int64).view(np.uint64)


def np_external_product(glwe: np.ndarray, ggsw_int: np.ndarray, radix_log: int, count: int) -> np.ndarray:
    """fft_ops.rs:23-56 with exact integer GGSW polynomials ggsw_int[row][level][poly][N]: sum over rows (GLWE
    polynomials) and levels (the LSB digit pairs with the last level) of digit * GGSW polynomial."""
    acc = [np.zeros(N, dtype=np.complex128) for _ in range(2)]
    for row in range(2):
        for t, d in enumerate(np_signed_digits(glwe[row * N:(row + 1) * N], radix_log, count)):
            level = count - 1 - t
            fd = np_negacyclic_fft(d)
            for q in range(2):
                acc[q] += fd * np_negacyclic_fft(ggsw_int[row, level, q])
    return np.concatenate([np_negacyclic_ifft_exact(a) for a in acc])


def np_cmux(d0, d1, ggsw_int, radix_log, count):
    return np_external_product(d1 - d0, ggsw_int, radix_log, count) + d0


def np_blind_rotation(lwe: np.ndarray, lut: np.ndarray, bsk_int: np.ndarray, log_chi: int, log_v: int) -> np.ndarray:
    """programmable_bootstrapping.rs:342-410: acc = LUT X^-b~, then acc <- CMUX(BSK_i, acc, acc X^a~_i) per step."""
    n = len(lwe) - 1
    ms = [np_modulus_switch(int(x), log_chi, log_v) for x in lwe]
    acc = np.concatenate([np_monomial(lut[q * N:(q + 1) * N], -ms[n]) for q in range(2)])
    for i in range(n):
        rot = np.concatenate([np_monomial(acc[q * N:(q + 1) * N], ms[i]) for q in range(2)])
        acc = np_cmux(acc, rot, bsk_int[i], 16, 2)
    return acc


# ---- tests ---------------------------------------------------------------------------------------------------------

def _emu_pbs(fn, lwe, lut, dev_bsk, log_chi, log_v):
    out = np.zeros(2 * N, dtype=np.uint64)
    fn(out, np.ascontiguousarray(lwe), lut.ctypes.data, dev_bsk, len(lwe) - 1, log_chi, log_v, 4, 4)
    return out


@pytest.mark.parametrize("mask,log_chi,log_v", [("random", 0, 0), ("random", 3, 2), ("every3", 0, 1)])
def test_full_pbs_oracle_equals_both_kernel_bodies(oracle, xk, dev_bsk, mask, log_chi, log_v):
    """A whole 637-step PBS of a u64 LWE and a u64 LUT: oracle == pair body (pbs_kernel) == quad body
    (pbs_quad_kernel), every coefficient."""
    rng = np.random.default_rng(log_chi * 16 + log_v)
    lwe = lwe_with_mask(mask, rng)
    lut = random_u64(rng, 2 * N)
    ref = oracle.pbs_generalized(xk, lwe, lut, log_chi, log_v)
    for fn in (E.lib().emu_pbs, E.lib().emu_pbs_quad):
        out = _emu_pbs(fn, lwe, lut, dev_bsk, log_chi, log_v)
        assert np.array_equal(out, ref), f"{fn.__name__}: {np.count_nonzero(out != ref)} coefficients differ"


def test_trace_and_cmux_bodies_equal_oracle(oracle, xk):
    """trace_ss_team (mode 1: plain trace), cmux_team and cmux_wide (with and without d0) on u64 inputs."""
    rng = np.random.default_rng(5)
    ak, ssk = E.to_device_scale(xk.ak_fft), E.to_device_scale(xk.ssk_fft)
    for _ in range(2):
        g = random_u64(rng, 2 * N)
        out = np.zeros(2 * N, dtype=np.uint64)
        E.lib().emu_trace_ss(g, out.ctypes.data, None, ak, ssk, 0, 1, 4, 4, 7, 6, 3, 15)
        assert np.array_equal(out, oracle.trace(xk, g))
        ggsw = exact_ggsw(rng, xk)
        gd = E.to_device_scale(ggsw)
        a, b = random_u64(rng, 2 * N), random_u64(rng, 2 * N)
        want = oracle.cmux(xk, a, b, ggsw)
        for fn in (E.lib().emu_cmux, E.lib().emu_cmux_wide):
            out = np.zeros(2 * N, dtype=np.uint64)
            fn(out, a.ctypes.data, b, gd, 4, 4)
            assert np.array_equal(out, want), fn.__name__
        out = np.zeros(2 * N, dtype=np.uint64)
        E.lib().emu_cmux_wide(out, None, b, gd, 4, 4)
        assert np.array_equal(out, oracle.multiply_glwe_ggsw(xk, b, ggsw))


@pytest.mark.parametrize("log_chi,log_v", [(0, 0), (2, 3)])
def test_short_blind_rotation_numpy_restatement(oracle, xk, dev_bsk, log_chi, log_v):
    """Three blind-rotation steps of u64 inputs (random mask, then one coefficient that switches to 0): numpy == oracle
    == both kernel bodies.  The numpy side asserts that every inverse transform is within 2^-8 of an integer."""
    rng = np.random.default_rng(70 + log_v)
    lwe = random_u64(rng, 4)
    lwe[1] = np.uint64(12345)  # switches to 0: the identity step
    lut = random_u64(rng, 2 * N)
    bsk_int = xk.bsk_int[:3 * 8].reshape(3, 2, 2, 2, N)  # [step][row][level][poly][N]
    want = np_blind_rotation(lwe, lut, bsk_int, log_chi, log_v)
    p = oracle.Params.from_buffer_copy(xk.params)
    p.lwe_n = 3
    ref = np.zeros(2 * N, dtype=np.uint64)
    oracle.lib().orc_pbs_generalized(ref, lwe, lut, xk.bsk_fft, log_chi, log_v, C.byref(p))
    assert np.array_equal(ref, want), "oracle vs numpy"
    for fn in (E.lib().emu_pbs, E.lib().emu_pbs_quad):
        assert np.array_equal(_emu_pbs(fn, lwe, lut, dev_bsk, log_chi, log_v), want), fn.__name__


def test_cmux_numpy_restatement(oracle, xk):
    rng = np.random.default_rng(8)
    ggsw, ints = exact_ggsw(rng, xk, with_ints=True)
    a, b = random_u64(rng, 2 * N), random_u64(rng, 2 * N)
    want = np_cmux(a, b, ints.reshape(2, 4, 2, N), 4, 4)
    assert np.array_equal(oracle.cmux(xk, a, b, ggsw), want)
    out = np.zeros(2 * N, dtype=np.uint64)
    E.lib().emu_cmux(out, a.ctypes.data, b, E.to_device_scale(ggsw), 4, 4)
    assert np.array_equal(out, want)


def test_interleaved_masks_skip_what_they_claim(oracle):
    """The mask patterns tests/test_gpu_exact.py feeds the PBS kernels: check the modulus-switch outcomes they are
    meant to produce, so the GPU tests cover the skipped-step paths they name."""
    lwe, kinds = interleaved_masks(20, 1)
    for x, kind in zip(lwe, kinds):
        ms = np.array([np_modulus_switch(int(v), 0, 0) for v in x[:-1]])
        zeros = np.flatnonzero(ms == 0)
        if kind in ("zero", "ones"):
            assert len(zeros) == 637, kind
        elif kind.startswith("every"):
            assert set(range(0, 637, int(kind[5:]))) <= set(zeros.tolist()), kind
        elif kind in ("first", "last"):
            assert (0 if kind == "first" else 636) in zeros
        elif kind == "runs":
            assert {1, 199, 400, 459, 537, 636} <= set(zeros.tolist())
        elif kind == "halfway":
            assert all(int(v) % (1 << 52) == 1 << 51 for v in x[:-1])
    # 2^64 - 1 switches to 2N at log_v > 0: a rotation by 2N (identity) that the kernels do not skip
    assert np_modulus_switch(M64, 0, 2) == 2 * N
    assert oracle.lib().orc_modulus_switch(M64, 0, 2, 12) == 2 * N
