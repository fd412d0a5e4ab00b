// tables.h -- host-side constant tables and layout conversions shared by the C-ABI library
// and the host emulator.
#pragma once
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#include "fft16.cuh"

namespace spf {

// T1[k1*64 + a] = e^{i pi a / 2048} * e^{-2 pi i a k1 / 1024}  (twist share of thread a, times
// the pass-1 -> pass-2 twiddle); T2[q*17 + k2] = e^{-2 pi i q k2 / 64}.
inline void fill_twiddle_tables(C2* T1, C2* T2) {
  const long double pi = 3.14159265358979323846264338327950288L;
  for (int k1 = 0; k1 < 16; k1++)
    for (int a = 0; a < 64; a++) {
      long double ang = pi * (long double)(a * (1 - 4 * k1)) / 2048.0L;
      T1[k1 * 64 + a] = C2{(double)cosl(ang), (double)sinl(ang)};
    }
  for (int q = 0; q < 4; q++)
    for (int k2 = 0; k2 < kT2Pad; k2++) {
      long double ang = -2.0L * pi * (long double)(q * k2) / 64.0L;
      T2[q * kT2Pad + k2] = C2{(double)cosl(ang), (double)sinl(ang)};
    }
}

// inverse of k_r = N / 2^r + 1 modulo 2N, r = 0..10 (ops/automorphisms/mod.rs:72-73)
inline void fill_kinv(uint32_t* kinv) {
  for (int r = 0; r < 11; r++) {
    uint32_t k = kN / (1u << r) + 1, x = 1;
    for (int it = 0; it < 12; it++) x = (x * (2 - k * x)) & (2 * kN - 1);  // Newton, mod 2^12
    kinv[r] = x & (2 * kN - 1);
  }
}

// reference scale (unnormalised DFT) <-> device scale (2^-10 folded in); same bin order
inline void import_fft_poly(const C2* nat, C2* dev) {
  for (int k = 0; k < kM; k++) dev[k] = C2{nat[k].x * (1.0 / 1024.0), nat[k].y * (1.0 / 1024.0)};
}
inline void export_fft_poly(const C2* dev, C2* nat) {
  for (int k = 0; k < kM; k++) nat[k] = C2{dev[k].x * 1024.0, dev[k].y * 1024.0};
}

}  // namespace spf
