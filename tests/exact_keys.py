"""Exact-regime keys: NOT SECURE, test infrastructure only.

Every FFT-domain key polynomial (bootstrapping key, automorphism key, scheme-switch key, test GGSWs) is the forward
transform of a seeded polynomial with integer coefficients in [-K, K].  With K = 2^16, every inverse transform a blind
rotation, a trace or a CMUX computes is then an integer well below 2^53 (|digit| <= 2^15, so a PBS product is at most
2 x 2 x 2048 x 2^15 x 2^16 = 2^44), and the floating-point value lies within a tiny fraction of a unit of it.  Any two
FFT implementations round it to the same integer, so the GPU kernels and the oracle's independent C code agree BIT FOR
BIT on whole blind rotations, traces and CMUXes of arbitrary u64 inputs, not only on honest encryptions.  (With real
keys the transforms carry torus-sized values, the two implementations pick different digits after the first blind-
rotation step and only decryptions and phase distances are comparable.)  The bound leaves a margin: the emulator and
the oracle stay bit-identical up to K = 2^24 and part at 2^28.

The keys encrypt nothing: they are small public polynomials, which is exactly what makes the arithmetic exact.  The
keyswitching key is the oracle's real one (keyswitching is integer arithmetic, exact for any key).
"""
from __future__ import annotations

from concurrent.futures import ThreadPoolExecutor

import numpy as np

import oracle as O

K_DEFAULT = 2 ** 16
N = 2048


def int_polys(rng: np.random.Generator, npoly: int, K: int = K_DEFAULT) -> np.ndarray:
    """[npoly, N] int64 polynomials with coefficients uniform in [-K, K]."""
    return rng.integers(-K, K + 1, (npoly, N)).astype(np.int64)


def polys_fft(ints: np.ndarray) -> np.ndarray:
    """oracle.poly_fft of every row, concatenated: the reference's FFT-domain layout, N / 2 bins per polynomial."""
    return np.concatenate([O.poly_fft(p) for p in ints.view(np.uint64)])


def exact_keys(seed: int, K: int = K_DEFAULT) -> O.Keys:
    """oracle.Keys(seed=seed) with bsk_fft, ak_fft and ssk_fft replaced by integer-polynomial transforms of the same
    shapes.  The integer polynomials are kept as bsk_int / ak_int / ssk_int ([npoly, N] int64, same order)."""
    keys = O.Keys(seed=seed)
    rng = np.random.default_rng(seed)
    for name in ("bsk", "ak", "ssk"):
        ints = int_polys(rng, getattr(keys, name + "_fft").size // (N // 2), K)
        setattr(keys, name + "_int", ints)
        setattr(keys, name + "_fft", polys_fft(ints))
    return keys


def exact_ggsw(rng: np.random.Generator, keys: O.Keys, K: int = K_DEFAULT, with_ints: bool = False):
    """A GGSW-FFT (reference scale, cbs radix shape) of integer polynomials in [-K, K]; optionally also the integers."""
    ints = int_polys(rng, keys.ggsw_fft_len // (N // 2), K)
    return (polys_fft(ints), ints) if with_ints else polys_fft(ints)


def random_u64(rng: np.random.Generator, *shape) -> np.ndarray:
    return rng.integers(0, 1 << 64, shape, dtype=np.uint64)


def par_map(fn, items, threads: int | None = None) -> list:
    """fn over items on a thread pool.  The oracle's ctypes calls release the GIL, so references for hundreds of items
    run on every core."""
    with ThreadPoolExecutor(threads or O.hw_threads()) as ex:
        return list(ex.map(fn, items))


# ---- LWE masks with chosen modulus-switch outcomes ----------------------------------------------------------------
# A mask coefficient whose modulus switch is 0 makes the blind-rotation step an identity, which the kernels skip
# (at == 0).  "Zero" entries are small nonzero values (< 2^40) that switch to 0 for every log_chi <= 11.

MASK_KINDS = ("random", "zero", "every2", "every3", "every7", "first", "last", "runs", "ones", "halfway")


def lwe_with_mask(kind: str, rng: np.random.Generator, n: int = 637) -> np.ndarray:
    """An L0 LWE (n mask coefficients + random body) whose mask follows `kind`."""
    a = random_u64(rng, n + 1)
    zero = rng.integers(0, 1 << 40, n, dtype=np.uint64)
    i = np.arange(n)
    if kind == "zero":
        a[:n] = zero
    elif kind.startswith("every"):
        k = int(kind[5:])
        a[:n] = np.where(i % k == 0, zero, a[:n])
    elif kind == "first":
        a[0] = zero[0]
    elif kind == "last":
        a[n - 1] = zero[n - 1]
    elif kind == "runs":  # long runs of skipped steps, including the last step
        run = ((i >= 1) & (i < 200)) | ((i >= 400) & (i < 460)) | (i >= n - 100)
        a[:n] = np.where(run, zero, a[:n])
    elif kind == "ones":  # 2^64 - 1 switches to 2N: wraps to 0 at log_v = 0, an identity rotation by 2N otherwise
        a[:n] = np.uint64((1 << 64) - 1)
    elif kind == "halfway":  # m 2^52 + 2^51: exactly half-way between two rotations at log_chi = log_v = 0
        a[:n] = (rng.integers(0, 1 << 12, n, dtype=np.uint64) << np.uint64(52)) + np.uint64(1 << 51)
    else:
        assert kind == "random", kind
    return a


def interleaved_masks(batch: int, seed: int, n: int = 637) -> tuple[np.ndarray, list[str]]:
    """batch LWEs cycling through MASK_KINDS: consecutive items -- which the PBS kernels place on different pairs and
    CTAs, and items c, c + grid, c + 2 grid sharing a CTA -- skip different steps."""
    rng = np.random.default_rng(seed)
    kinds = [MASK_KINDS[c % len(MASK_KINDS)] for c in range(batch)]
    return np.stack([lwe_with_mask(k, rng, n) for k in kinds]), kinds
