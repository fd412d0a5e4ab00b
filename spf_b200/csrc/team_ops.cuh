// team_ops.cuh -- bodies of the hot-path kernels, written once for a TEAM of 64 threads and
// compiled for BOTH the device (kernels.cu, barrier = named bar.sync) and the host emulator
// (emu.cpp, barrier = pthread barrier over 64 host threads).  One team owns one GLWE
// accumulator / one ciphertext at a time.
//
// Device conventions (see DESIGN.md):
//  * time domain: thread u owns coefficients j = u + 64*i, i = 0..31 of every polynomial
//    (i < 16 -> real part of FFT point m = i, i >= 16 -> imaginary part of point m = i - 16);
//  * frequency domain: thread u owns the 16 bins bin_of(u, s) = u + 64*slot_row(s); arrays are
//    stored in the reference's natural bin order, so each slot is a coalesced 1 KiB row;
//  * every FFT-domain key / GGSW resident on the device carries a factor 2^-10 (= 1/(N/2), the
//    normalisation of complex_untwist, simd/scalar.rs:27); scaling by a power of two is exact
//    so results are bit-identical to normalising after the inverse transform.
#pragma once
#include <type_traits>

#include "fft16.cuh"

namespace spf {

constexpr double kInvM = 1.0 / 1024.0;

SPF_HD C2 ldg_c2(const C2* p) {
#if defined(__CUDA_ARCH__)
  const double2 t = __ldg(reinterpret_cast<const double2*>(p));
  return C2{t.x, t.y};
#else
  return *p;
#endif
}
SPF_HD C2 cscale(C2 a, double f) { return C2{a.x * f, a.y * f}; }
SPF_HD uint64_t ldg_u64(const uint64_t* p) {
#if defined(__CUDA_ARCH__)
  return __ldg(reinterpret_cast<const unsigned long long*>(p));
#else
  return *p;
#endif
}

// ---- whole-polynomial transforms for a team ------------------------------------------------
// xbuf must not be in use by any thread of the team on entry (the leading sync guarantees the
// previous transform's reads are complete).
// Cx::kTmemTwiddles: the thread's 16 pass-1 and 15 pass-2 twiddles come from its tensor-memory columns (cx.t1_mul / t2_mul,
// same products in the same order) instead of the shared-memory tables: 31 LDS.128 per transform less on the pipe that
// bounds these kernels.
template <class Cx>
SPF_HD void team_fft_fwd(Cx& cx, C2 (&v)[16], C2* xbuf, const C2* T1, const C2* T2) {
  if constexpr (Cx::kTmemTwiddles) {
    fwd_pass1_core(v);
    cx.template t1_mul<false>(v);
  } else {
    fwd_pass1(v, cx.u, T1);
  }
  cx.sync();
  fwd_x1_write(v, xbuf, cx.u);
  cx.sync();
  fwd_x1_read(v, xbuf, cx.u);
  if constexpr (Cx::kTmemTwiddles) {
    dft16<false>(v);
    cx.template t2_mul<false>(v);
  } else {
    fwd_pass2(v, cx.u, T2);
  }
  fwd_x2_write(v, xbuf, cx.u);  // in place: overwrites only what this thread has just read
  cx.sync();
  fwd_x2_read(v, xbuf, cx.u);
  fwd_pass3(v);
}
template <class Cx>
SPF_HD void team_fft_inv(Cx& cx, C2 (&v)[16], C2* xbuf, const C2* T1, const C2* T2) {
  inv_pass3(v);
  cx.sync();
  inv_x2_write(v, xbuf, cx.u);
  cx.sync();
  inv_x2_read(v, xbuf, cx.u);
  if constexpr (Cx::kTmemTwiddles) {
    cx.template t2_mul<true>(v);
    dft16<true>(v);
  } else {
    inv_pass2(v, cx.u, T2);
  }
  inv_x1_write(v, xbuf, cx.u);  // in place
  cx.sync();
  inv_x1_read(v, xbuf, cx.u);
  if constexpr (Cx::kTmemTwiddles) {
    cx.template t1_mul<true>(v);
    inv_pass1_core(v);
  } else {
    inv_pass1(v, cx.u, T1);
  }
}

// acc[p][s] += v[s] * G[p][s][u]   (glwe_polynomial_mad, ops/fft_ops.rs:107-124)
SPF_HD void mad_glwe(C2 (&acc)[2][16], const C2 (&v)[16], const C2* g, int u) {
#pragma unroll
  for (int h = 0; h < 4; h++) {  // 4 slots x 2 polys in flight per batch
    C2 b0[4], b1[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      b0[i] = ldg_c2(g + bin_of(u, 4 * h + i));
      b1[i] = ldg_c2(g + kM + bin_of(u, 4 * h + i));
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
      cmad(acc[0][4 * h + i], v[4 * h + i], b0[i]);
      cmad(acc[1][4 * h + i], v[4 * h + i], b1[i]);
    }
  }
}

SPF_HD void zero_acc(C2 (&acc)[2][16]) {
#pragma unroll
  for (int p = 0; p < 2; p++)
#pragma unroll
    for (int s = 0; s < 16; s++) acc[p][s] = C2{0.0, 0.0};
}

// Plain FFT of a torus polynomial (PolynomialRef::fft, entities/polynomial.rs:257-274):
// u64 -> i64 -> f64, transform; result scaled by 2^-10 (device convention).
template <class Cx, class F>
SPF_HD void team_poly_fft(Cx& cx, C2 (&v)[16], F coef, C2* xbuf, const C2* T1, const C2* T2) {
#pragma unroll
  for (int m = 0; m < 16; m++) {
    v[m].x = i64_to_f64((int64_t)coef(cx.u + 64 * m));
    v[m].y = i64_to_f64((int64_t)coef(cx.u + 64 * m + kM));
  }
  team_fft_fwd(cx, v, xbuf, T1, T2);
#pragma unroll
  for (int s = 0; s < 16; s++) { v[s].x *= kInvM; v[s].y *= kInvM; }
}

// ---- generic gadget product -----------------------------------------------------------------
// PolynomialRadixIterator::new (math/radix.rs:81-99): per-coefficient rounded state, kept in a
// team-private smem array st[i*64 + u].
template <class Cx, class F>
SPF_HD void state_init(Cx& cx, uint64_t* st, int radix_log, int count, F coef) {
#pragma unroll 4
  for (int i = 0; i < 32; i++) st[i * 64 + cx.u] = radix_round(coef(cx.u + 64 * i), radix_log, count);
}

// decomposed_polynomial_glev_mad (ops/fft_ops.rs:67-98): for each digit (LSB first) FFT it and
// multiply-accumulate against the GLEV's GLWE in REVERSE level order.  glev: [level][p][bin].
template <class Cx>
SPF_HD void gadget_mad(Cx& cx, C2 (&acc)[2][16], uint64_t* st, C2* xbuf, const C2* T1, const C2* T2,
                       const C2* glev, int radix_log, int count) {
  for (int t = 0; t < count; t++) {
    C2 v[16];
#pragma unroll
    for (int m = 0; m < 16; m++) {
      uint64_t s0 = st[m * 64 + cx.u], s1 = st[(m + 16) * 64 + cx.u];
      v[m].x = i32_to_f64(next_digit(s0, radix_log));
      v[m].y = i32_to_f64(next_digit(s1, radix_log));
      st[m * 64 + cx.u] = s0;
      st[(m + 16) * 64 + cx.u] = s1;
    }
    team_fft_fwd(cx, v, xbuf, T1, T2);
    mad_glwe(acc, v, glev + (size_t)(count - 1 - t) * 2 * kM, cx.u);
  }
}

// Stateless variant: the digits of level t are read straight out of the bit fields of
// r' = round(coef(j)) + radix_offset (no carry chain, so nothing to update between levels).  r' is
// evaluated ONCE per product (the automorphism gather and the 64-bit rounding are the expensive part)
// and parked with cx.rp_store: tensor-memory columns of the thread on the device, so neither the
// 16 KiB shared-memory state array of gadget_mad nor 64 registers are needed.
template <class Cx, class F>
SPF_HD void gadget_mad_stateless(Cx& cx, C2 (&acc)[2][16], F coef, C2* xbuf, const C2* T1, const C2* T2, const C2* glev,
                                 int radix_log, int count) {
  const uint64_t off = radix_offset(radix_log, count);
  const uint64_t dmask = (1ull << radix_log) - 1;
  const int32_t half = 1 << (radix_log - 1);
  {
    uint64_t rp[32];
#pragma unroll
    for (int i2 = 0; i2 < 32; i2++) rp[i2] = radix_round(coef(cx.u + 64 * i2), radix_log, count) + off;
    cx.rp_store(rp);
  }
  for (int t = 0; t < count; t++) {
    C2 v[16];
    {
      uint64_t rp[32];
      cx.rp_load(rp);
#pragma unroll
      for (int m = 0; m < 16; m++) {
        v[m].x = i32_to_f64((int32_t)((rp[m] >> (t * radix_log)) & dmask) - half);
        v[m].y = i32_to_f64((int32_t)((rp[m + 16] >> (t * radix_log)) & dmask) - half);
      }
    }
    team_fft_fwd(cx, v, xbuf, T1, T2);
    mad_glwe(acc, v, glev + (size_t)(count - 1 - t) * 2 * kM, cx.u);
  }
}

// ---- CMUX / external product (ops/fft_ops.rs:23-56,149-181) ---------------------------------
// out = d0 + IFFT(GGSW [*] (d1 - d0)).  d0 == nullptr: plain external product of d1
// (KeylessEvaluation::multiply_glwe_ggsw, parasol_runtime/src/crypto/evaluation.rs:104-123).
// ggsw: [row][level][p][bin], 2^-10 scaled.  All GLWE pointers are global.
template <class Cx>
SPF_HD void cmux_team(Cx& cx, uint64_t* out, const uint64_t* d0, const uint64_t* d1, const C2* ggsw,
                      uint64_t* st, C2* xbuf, const C2* T1, const C2* T2, int radix_log, int count) {
  C2 acc[2][16];
  zero_acc(acc);
  for (int r = 0; r < 2; r++) {
    const uint64_t* a1 = d1 + r * kN;
    const uint64_t* a0 = d0 ? d0 + r * kN : nullptr;
    state_init(cx, st, radix_log, count,
               [&](int j) { return a0 ? ldg_u64(a1 + j) - ldg_u64(a0 + j) : ldg_u64(a1 + j); });
    gadget_mad(cx, acc, st, xbuf, T1, T2, ggsw + (size_t)r * count * 2 * kM, radix_log, count);
  }
#pragma unroll
  for (int p = 0; p < 2; p++) {
    team_fft_inv(cx, acc[p], xbuf, T1, T2);
#pragma unroll
    for (int m = 0; m < 16; m++) {
      const int j = cx.u + 64 * m;
      uint64_t re = f64_to_torus(acc[p][m].x), im = f64_to_torus(acc[p][m].y);
      if (d0) { re += ldg_u64(d0 + p * kN + j); im += ldg_u64(d0 + p * kN + j + kM); }
      out[p * kN + j] = re;
      out[p * kN + j + kM] = im;
    }
  }
}

// ---- programmable bootstrap (blind rotation) -------------------------------------------------
// generalized_programmable_bootstrap (ops/bootstrapping/programmable_bootstrapping.rs:342-410)
// for pbs_radix = (logB 16, l 2).  acc: pair smem u64[2][2048].
// bsk: [i][row][level][p][bin] (the reference's BootstrapKeyFft order), 2^-10 scaled.
// lut == nullptr selects circuit-bootstrap mode: hi_noise_lwe_to_lo_noise_glwe
// (circuit_bootstrapping.rs:387-428): b += q/4, LUT = fill_multifunctional_cbs_decomposition_lut
// (:430-482) generated on the fly, log_v = ceil(log2(cbs_count)).
struct PbsArgs {
  const uint64_t* lwe_in;  // n + 1
  const uint64_t* lut;     // GLWE [2][2048] or nullptr (CBS mode)
  uint64_t* glwe_out;      // [2][2048]
  const C2* bsk;
  int lwe_n;
  int log_chi, log_v;
  int cbs_radix_log, cbs_count;  // CBS mode only
};

SPF_HD uint32_t modulus_switch(uint64_t x, int log_chi, int log_v, int log_modulus) {
  // ops/ciphertext/lwe_ciphertext_ops.rs:129-142
  const uint64_t mask = (1ull << log_modulus) - 1;
  x <<= log_chi;
  const int shift = 64 - (log_modulus - log_v);
  const uint64_t rnd = (x >> (shift - 1)) & 1;
  x >>= shift;
  return (uint32_t)(((x + rnd) & mask) << log_v);
}

SPF_HD uint64_t cbs_lut_coeff(int idx, int cbs_radix_log, int cbs_count, int v) {
  const int f = idx & (v - 1);
  if (f >= cbs_count) return 0;
  const int pb = cbs_radix_log * (f + 1) + 1;
  return pb < 64 ? 0 - (1ull << (64 - pb)) : 0;  // Torus::encode(2^pb - 1, pb)
}

// acc[s] (+)= v[s] * G[s]  (one output polynomial); INIT assigns instead of accumulating so the
// accumulator is not live (and not spilled) before the first product of a step.
template <bool INIT>
SPF_HD void mad_poly(C2 (&acc)[16], const C2 (&v)[16], const C2* g, int u) {
#pragma unroll
  for (int h = 0; h < 4; h++) {
    C2 b[4];
#pragma unroll
    for (int i = 0; i < 4; i++) b[i] = ldg_c2(g + bin_of(u, 4 * h + i));
#pragma unroll
    for (int i = 0; i < 4; i++) {
      if (INIT) acc[4 * h + i] = cmul(v[4 * h + i], b[i]);
      else cmad(acc[4 * h + i], v[4 * h + i], b[i]);
    }
  }
}
// acc[s] += D[s][u] * G[s], D read from a partner team's shared buffer (layout [s][u])
SPF_HD void mad_poly_shared(C2 (&acc)[16], const C2* dbuf, const C2* g, int u) {
#pragma unroll
  for (int h = 0; h < 4; h++) {
    C2 b[4], d[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      b[i] = ldg_c2(g + bin_of(u, 4 * h + i));
      d[i] = dbuf[(4 * h + i) * 64 + u];
    }
#pragma unroll
    for (int i = 0; i < 4; i++) cmad(acc[4 * h + i], d[i], b[i]);
  }
}

// signed 16-bit digit (given as its low 16 bits) -> f64 with one integer op and one DADD:
// 2^52 + ((d & 0xFFFF) ^ 0x8000) = 2^52 + 2^15 + sext16(d).
SPF_HD double digit16_to_f64(uint32_t d) {
  const uint64_t bits = 0x4330000000000000ull | (uint64_t)((d & 0xFFFFu) ^ 0x8000u);
  double x;
#if defined(__CUDA_ARCH__)
  x = __longlong_as_double((long long)bits);
#else
  __builtin_memcpy(&x, &bits, 8);
#endif
  return x - 4503599627403264.0;  // 2^52 + 2^15
}

// Signed 16-bit digit sitting in the LOW half of d (upper half ignored) -> f64.  Host: one IMAD and one DADD: the low
// word (d << 16) + 2^31 of a double with exponent 2^36 (ulp 2^-16) reads as 2^36 + 2^15 + sext16(d).  Device: one
// conversion instruction (I2F.F64.S16 on the conversion pipe, which selects the half word itself) instead of an integer
// op, a move for the exponent word and a DADD on the FP64 pipe; the values are identical (measured: 6.96 -> 6.73 ms per
// 444-ciphertext wave of pbs_kernel, profiles/r2_zz_i2f_ab.txt).
SPF_HD double digit_lo16_to_f64(uint32_t d) {
#if defined(__CUDA_ARCH__)
  double r;
  asm("{\n\t.reg .b16 lo, hi;\n\tmov.b32 {lo, hi}, %1;\n\tcvt.rn.f64.s16 %0, lo;\n\t}" : "=d"(r) : "r"(d));
  return r;
#else
  return bits_f64(0x4230000000000000ull | (uint64_t)(uint32_t)(d * 65536u + 0x80000000u)) - 68719509504.0;  // 2^36 + 2^15
#endif
}
// the same for a digit sitting in the HIGH half of d (lower half ignored); host: one LOP3 and one DADD
SPF_HD double digit_hi16_to_f64(uint32_t d) {
#if defined(__CUDA_ARCH__)
  double r;
  asm("{\n\t.reg .b16 lo, hi;\n\tmov.b32 {lo, hi}, %1;\n\tcvt.rn.f64.s16 %0, hi;\n\t}" : "=d"(r) : "r"(d));
  return r;
#else
  return bits_f64(0x4230000000000000ull | (uint64_t)(uint32_t)((d & 0xFFFF0000u) ^ 0x80000000u)) - 68719509504.0;
#endif
}

// PAIR-TEAM blind rotation, BIN-SPLIT: one ciphertext = 128 threads = two teams of 64 (half h).
// Time domain: half h owns GLWE polynomial h (decomposition of acc[h]*X^a - acc[h], passes 1-2 of
// its two forward FFTs, passes 2-1 of its inverse FFT, accumulator update).  Frequency domain:
// half h owns the bins with bit 7 == h of ALL polynomials: after pass 2 each half leaves its
// spectrum-in-progress in its exchange buffer, and BOTH halves run the final radix-4 pass on
// their 8 bins per thread of BOTH digit polynomials, multiply-accumulate them against the BSK
// into both output polynomials (f[2][8], the same 64 registers as one full polynomial) and run
// the first inverse pass before handing the halves of each output polynomial back through the
// exchange buffers.  No spectrum is ever published a second time: compared with sharing whole
// FFT outputs this removes 128 KiB of shared-memory traffic per CMUX step.
// Both digit levels come out of ONE gather pass over the accumulator; the second level waits
// packed 2x16 bit in 16 registers while the first is transformed.
//   cx.u: thread in half (0..63)   cx.h: half   cx.sync(): 64-thread barrier of the half
//   cx.pair_sync(): 128-thread barrier of the pair
//   xb: the pair's two exchange buffers, xb + h*kXBuf belongs to half h.

// Register slot s' = 4 jj + k3 of thread u in half h holds bin u + 64 * (2h + jj + 4 k3).
SPF_HD constexpr int split_bin(int u, int h, int s) { return u + 64 * (2 * h + (s >> 2) + 4 * (s & 3)); }

// ---- reader-side pass-2 twiddles -----------------------------------------------------------------------------------
// The pass-2 -> pass-3 twiddle W64^(q' k2) of a forward transform does not have to be applied by the thread that produced
// z[k2] (15 complex multiplies per transform): the thread that CONSUMES the value in mad_split_rt knows q' (its loop index)
// and k2 = q + 4 (2 h + jj) (its own bins), needs only 3 twiddles per radix-4 group -- the same 6 for all four spectra of a
// step -- and can apply them in the tan form  w = c (1 + i t):  two FMAs per value, the factored-out c riding into the
// butterfly as scale ratios (bfly4_r; the same instruction count as the plain butterfly).  4 x 2 x 3 x 2 = 48 FP64
// instructions per thread and step instead of 2 x 15 x 4 = 120.  In the inverse direction the bin owner multiplies by the
// conjugates before it hands the values back (12 complex multiplies instead of 15 on the receiving side).
// Constants of thread (q = u >> 4, half h), group jj: o[6 jj + 0..2] = t_1..t_3, o[6 jj + 3..5] = c_1, c_2, c_3 / c_1.
// cos(pi/2) in the table is ~1e-20, not 0 (tables.h rounds a long double): the quarter turn q' = 2, k2 = 8 comes out as
// t ~ 1e19, c ~ 1e-20, exact to 2^-64; an exact zero is replaced so that no infinity can arise.
SPF_HD void rt2_fwd_consts(const C2* T2, int q, int h, double (&o)[12]) {
  for (int jj = 0; jj < 2; jj++) {
    const int k2 = q + 4 * (2 * h + jj);
    double c[4];
    for (int qp = 1; qp < 4; qp++) {
      const C2 w = T2[qp * kT2Pad + k2];
      c[qp] = w.x == 0.0 ? 8.470329472543003e-22 /* 2^-70 */ : w.x;
      o[6 * jj + qp - 1] = w.y / c[qp];
    }
    o[6 * jj + 3] = c[1];
    o[6 * jj + 4] = c[2];
    o[6 * jj + 5] = c[3] / c[1];
  }
}
SPF_HD void rt2_inv_consts(const C2* T2, int q, int h, C2 (&o)[6]) {
  for (int jj = 0; jj < 2; jj++)
    for (int qp = 1; qp < 4; qp++) o[3 * jj + qp - 1] = T2[qp * kT2Pad + q + 4 * (2 * h + jj)];
}
// the same constants for ONE radix-4 group k2 = q + 4 grp (the quad kernel: team g owns group g): tw[0..2] = t_1..t_3,
// tw[3..5] = c_1, c_2, c_3 / c_1; wi[0..2] = W64^(q' k2), q' = 1..3 (conjugated by the consumer)
SPF_HD void rt2_group_consts(const C2* T2, int q, int grp, double (&tw)[6], C2 (&wi)[3]) {
  const int k2 = q + 4 * grp;
  double c[4];
  for (int qp = 1; qp < 4; qp++) {
    const C2 w = T2[qp * kT2Pad + k2];
    wi[qp - 1] = w;
    c[qp] = w.x == 0.0 ? 8.470329472543003e-22 /* 2^-70 */ : w.x;
    tw[qp - 1] = w.y / c[qp];
  }
  tw[3] = c[1];
  tw[4] = c[2];
  tw[5] = c[3] / c[1];
}
// final forward radix-4 pass on this half's bins of digit polynomial b (spectrum-in-progress in xbb, its pass-2 twiddles NOT
// applied yet: tw from rt2_fwd_consts), then f[p] (+)= D * G[b][level][p] for both output polynomials p.  Written as two
// independent 4-bin batches: the compiler hoists the second batch's BSK loads above the first batch's arithmetic
// (measured: explicit earlier prefetching only costs registers and spills).
template <bool INIT, class Cx>
SPF_HD void mad_split_rt(Cx& cx, C2 (&f)[2][8], const C2* xbb, const C2* g /* GGSW row b, level: [p][bin] */, int u, int h,
                         const double (&tw)[12]) {
  const int k1 = u & 15, q = u >> 4;
#pragma unroll
  for (int jj = 0; jj < 2; jj++) {
    C2 d[4], g0[4], g1[4];
#pragma unroll
    for (int qp = 0; qp < 4; qp++) d[qp] = xbb[k1 * kXPad + qp + 4 * q + 16 * (2 * h + jj)];
#pragma unroll
    for (int k3 = 0; k3 < 4; k3++) {
      g0[k3] = cx.bsk_load(g + split_bin(u, h, 4 * jj + k3));
      g1[k3] = cx.bsk_load(g + kM + split_bin(u, h, 4 * jj + k3));
    }
#pragma unroll
    for (int qp = 1; qp < 4; qp++) {
      const double t = tw[6 * jj + qp - 1];
      d[qp] = C2{spf_fma(-t, d[qp].y, d[qp].x), spf_fma(t, d[qp].x, d[qp].y)};  // d (1 + i t); the factor c rides in the ratios
    }
    bfly4_r<false>(d[0], d[1], d[2], d[3], tw[6 * jj + 3], tw[6 * jj + 4], tw[6 * jj + 5]);
#pragma unroll
    for (int k3 = 0; k3 < 4; k3++) {
      const int s = 4 * jj + k3;
      if (INIT) { f[0][s] = cmul(d[k3], g0[k3]); f[1][s] = cmul(d[k3], g1[k3]); }
      else { cmad(f[0][s], d[k3], g0[k3]); cmad(f[1][s], d[k3], g1[k3]); }
    }
  }
}

// BSK ring (device only): the key is consumed in CHUNKS of one (row, level) GLEV row [p][bin] = 32 KiB, four
// per CMUX step in the order (row 0, level 1), (row 1, level 1), (row 0, level 0), (row 1, level 0).  All pairs of a
// CTA walk the same chunk sequence G = 4 i + k (continuing over the ciphertexts they process: the key repeats), so
// ONE bulk copy per chunk (cp.async.bulk -> mbarrier, kernels.cuh) serves all of them from a small shared-memory ring:
// bsk_acquire waits until chunk G has landed, bsk_release (one thread per pair, after a pair barrier that follows the
// last read) counts the pair off; the last pair to release a stage re-arms it with chunk G + stages.
template <class Cx>
SPF_HD void pbs_pair_team(Cx& cx, const PbsArgs& A, C2* xb, const C2* T1, const C2* T2, int& G) {
  const int u = cx.u, h = cx.h;
  const int k1 = u & 15, q = u >> 4;
  const int n = A.lwe_n;
  const bool cbs = A.lut == nullptr;
  const int log2n = 12;  // log2(2N)
  C2* xown = xb + h * kXBuf;
  // The accumulator polynomial of this half lives ONLY in the threads' own-coefficient copies (device: tensor memory);
  // the shared-memory image the rotated gather reads is written into the half's exchange buffer at the end of a step
  // and is dead once the digits have been taken, so a pair needs no persistent 32 KiB accumulator in shared memory
  // (two more half-barriers per step: gather -> first exchange write, last exchange read -> image write).
  uint64_t* pa = reinterpret_cast<uint64_t*>(xown);  // the polynomial this half owns
  // 1. acc = LUT * X^{-b~}   (programmable_bootstrapping.rs:378-390)
  {
    uint64_t b = ldg_u64(A.lwe_in + n);
    if (cbs) b += 1ull << 62;  // lwe_rotate by Torus::encode(1, 2 bits) (circuit_bootstrapping.rs:403-408)
    const int bt = (int)modulus_switch(b, A.log_chi, A.log_v, log2n);
    const int rot = (2 * kN - bt) & (2 * kN - 1);
    const int v = 1 << A.log_v;
    for (int i = 0; i < 32; i++) {
      const int j = u + 64 * i;
      int idx = j - rot;
      bool neg = false;
      if (idx < 0) { idx += kN; neg = true; }
      if (idx < 0) { idx += kN; neg = false; }
      uint64_t c;
      if (cbs) c = h ? cbs_lut_coeff(idx, A.cbs_radix_log, A.cbs_count, v) : 0;
      else c = ldg_u64(A.lut + h * kN + idx);
      pa[u + 64 * i] = neg ? 0 - c : c;
    }
  }
  cx.sync();
  // 2. 637 CMUXes (programmable_bootstrapping.rs:396-409)
  uint64_t a_next = n > 0 ? ldg_u64(A.lwe_in) : 0;
  // own[]: the thread's own coefficients pa[u + 64 i2], fetched from the thread's tensor-memory copy 8 (gather) or
  // 4 + 4 (update) at a time, so neither phase holds all 32 next to a 16-point transform.
  uint64_t own[8];
  {
    uint64_t o0[32];
#pragma unroll
    for (int i2 = 0; i2 < 32; i2++) o0[i2] = pa[u + 64 * i2];
    cx.own_store(o0);
  }
#pragma unroll 1
  for (int i = 0; i < n; i++) {
    const int at = (int)modulus_switch(a_next, A.log_chi, A.log_v, log2n);
    if (i + 1 < n) a_next = ldg_u64(A.lwe_in + i + 1);
    if (at == 0) {  // rot == acc: the CMUX adds IFFT(0) = 0 exactly (uniform over the pair)
      cx.bsk_skip(G);  // the pair still counts itself off the four chunks of this step
      G += 4;
      continue;
    }
    const C2* ggsw = A.bsk + (size_t)i * 8 * kM;
    C2 f[2][8];
    {
      C2 v[16];
      uint32_t pk[16];
      // diff = acc*X^{a~} - acc (rotation fused into the gather); round to 32 bits; split into two
      // signed 16-bit digits, LSB first (math/radix.rs:81-113 for logB=16, l=2).  The source index
      // of coefficient j = u + 64 i2 is (u - a~ + 64 i2) mod 2N: bit 11 = negacyclic sign.
      {
        const int base = (u - at) & (2 * kN - 1);
        // byte address of source row tt = (base >> 6) + i2 (mod 32) of this thread's column:
        // rows are 512 B apart, so the row index lives in bits 9..13 of the offset
        const char* col = reinterpret_cast<const char*>(pa) + 8 * (base & 63);
        const uint32_t bh9 = (uint32_t)(base >> 6) << 9;
#pragma unroll
        for (int i2 = 0; i2 < 32; i2++) {
          if ((i2 & 7) == 0) cx.own_ld8(own, i2 >> 3);  // own[0..7] = coefficients 8c .. 8c + 7
          const uint32_t t9 = bh9 + 512u * i2;  // bit 14 = negacyclic sign
          const uint64_t x = *reinterpret_cast<const uint64_t*>(col + (t9 & 0x3E00u));
          const uint64_t diff = ((t9 & 0x4000u) ? 0 - x : x) - own[i2 & 7];
          const uint32_t w = (uint32_t)(diff >> 32) + ((uint32_t)diff >> 31);
          const uint32_t w1 = w + 0x8000u;  // high half = second digit: (w >> 16) + carry of the first
          if (i2 < 16) { v[i2].x = digit_lo16_to_f64(w); pk[i2] = w1 >> 16; }
          else { v[i2 - 16].y = digit_lo16_to_f64(w); pk[i2 - 16] |= w1 & 0xFFFF0000u; }
        }
      }
#pragma unroll
      for (int t = 0; t < 2; t++) {
        const int level = 1 - t;  // LSB digit <-> last GLEV level (fft_ops.rs:92)
        if (t == 1) {
#pragma unroll
          for (int m = 0; m < 16; m++) { v[m].x = digit_lo16_to_f64(pk[m]); v[m].y = digit_hi16_to_f64(pk[m]); }
        }
        fwd_pass1_core(v);
        cx.template t1_mul<false>(v, T1);  // v[k1] *= T1[k1][u]
        if (t == 1) { cx.pair_sync(); cx.bsk_release(G); cx.bsk_release(G + 1); }  // both halves have consumed the level-0 spectra (and the key chunks)
        else cx.sync();  // every thread of the half has gathered from the accumulator image in xown
        fwd_x1_write(v, xown, u);
        cx.sync();
        fwd_x1_read(v, xown, u);
        dft16<false>(v);
        fwd_x2_write(v, xown, u);  // in place: no barrier after fwd_x1_read; the pass-2 twiddles are applied by the readers
        if (t == 1) cx.f_load(f);
        cx.pair_sync();
        const C2* g0 = cx.bsk_acquire(G + 2 * t, ggsw + (size_t)((0 * 2 + level) * 2) * kM);
        double tw[12];
        cx.rt2_fwd(tw, T2);
        if (t == 0) mad_split_rt<true>(cx, f, xb, g0, u, h, tw);
        else mad_split_rt<false>(cx, f, xb, g0, u, h, tw);
        const C2* g1 = cx.bsk_acquire(G + 2 * t + 1, ggsw + (size_t)((1 * 2 + level) * 2) * kM);
        mad_split_rt<false>(cx, f, xb + kXBuf, g1, u, h, tw);
        if (t == 0) cx.f_store(f);  // device: parked in tensor memory while the second transform runs
      }
    }
    // first inverse pass on this half's bins of both output polynomials, hand them to their owners
#pragma unroll
    for (int p = 0; p < 2; p++) {
      bfly4<true>(f[p][0], f[p][1], f[p][2], f[p][3]);
      bfly4<true>(f[p][4], f[p][5], f[p][6], f[p][7]);
    }
    {  // the conjugate pass-2 twiddles of the inverse transform, applied by the bin owner
      C2 wi[6];
      cx.rt2_inv(wi, T2);
#pragma unroll
      for (int p = 0; p < 2; p++)
#pragma unroll
        for (int jj = 0; jj < 2; jj++)
#pragma unroll
          for (int qp = 1; qp < 4; qp++) f[p][4 * jj + qp] = cmul_conj(f[p][4 * jj + qp], wi[3 * jj + qp - 1]);
    }
    // in place: every thread overwrites exactly the 8 locations per buffer it read in mad_split_rt
#pragma unroll
    for (int p = 0; p < 2; p++) {
#pragma unroll
      for (int jj = 0; jj < 2; jj++) {
#pragma unroll
        for (int qp = 0; qp < 4; qp++) xb[p * kXBuf + k1 * kXPad + qp + 4 * q + 16 * (2 * h + jj)] = f[p][4 * jj + qp];
      }
    }
    cx.pair_sync();
    cx.bsk_release(G + 2);
    cx.bsk_release(G + 3);
    G += 4;
    // acc[h] += IFFT(output polynomial h)
    {
      C2 w[16];
      inv_x2_read(w, xown, u);
      dft16<true>(w);
      inv_x1_write(w, xown, u);  // in place: no barrier after inv_x2_read
      cx.sync();
      inv_x1_read(w, xown, u);
      cx.sync();  // xown becomes the accumulator image again (every thread has read its inverse-pass inputs)
      cx.template t1_mul<true>(w, T1);  // w[k1] *= conj(T1[k1][u])
      double ws[16];
      inv_pass1_core_s(w, ws);  // true value ws[m] * w[m]: the untwist's real factor rides into the conversion
      // The saturating-cast corner of the conversion (probability ~2^-53 per value) is tested once
      // per 8 values: the fast conversion only tracks the largest exponent word it saw.
#pragma unroll
      for (int m4 = 0; m4 < 16; m4 += 4) {
        uint32_t mag_max = 0;
        uint64_t r[8];
#pragma unroll
        for (int i = 0; i < 4; i++) {
          r[2 * i] = f64_to_torus_s_fast(w[m4 + i].x, ws[m4 + i], mag_max);
          r[2 * i + 1] = f64_to_torus_s_fast(w[m4 + i].y, ws[m4 + i], mag_max);
        }
        if (__builtin_expect(mag_max == kTorusCornerMag, 0)) {
#pragma unroll
          for (int i = 0; i < 4; i++) {
            r[2 * i] = f64_to_torus_s(w[m4 + i].x, ws[m4 + i]);
            r[2 * i + 1] = f64_to_torus_s(w[m4 + i].y, ws[m4 + i]);
          }
        }
        cx.own_ld4x2(own, m4);  // own[0..3] = coefficients m4 .. m4 + 3, own[4..7] = m4 + 16 .. m4 + 19
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const int j = u + 64 * (m4 + i);
          own[i] += r[2 * i];
          own[4 + i] += r[2 * i + 1];
          pa[j] = own[i];
          pa[j + kM] = own[4 + i];
        }
        cx.own_st4x2(own, m4);
      }
      cx.own_st_wait();
    }
    cx.sync();  // next step gathers rotated coefficients written by other threads of this half
  }
  // 3. result
  for (int i = 0; i < 32; i++) A.glwe_out[h * kN + u + 64 * i] = pa[u + 64 * i];
  cx.sync();  // the next ciphertext of this pair overwrites the image
}

// QUAD-TEAM blind rotation (latency mode, batches of at most one ciphertext per SM): one ciphertext
// = 256 threads = 4 teams (h, t): team (h, t) transforms digit level t of polynomial h, all four
// forward transforms of a CMUX step run concurrently, the bins are split four ways for the
// multiply-accumulate (f[2][4] per thread) and teams (p, 0) finish the inverse transform of output
// polynomial p.  The critical path of a step is one forward transform + one MAD phase + one inverse
// instead of two + two + one; the arithmetic per coefficient is identical to pbs_pair_team.
//   cx.u, cx.h, cx.t;  cx.sync(): team barrier;  cx.quad_sync(): the ciphertext's 256 threads
//   xb: 4 exchange buffers, team (h, t) owns xb + (2 h + t) * kXBuf.
//   executed: running count of executed steps on this CTA (phase bookkeeping of the staged-row barrier)
template <class Cx>
SPF_HD void pbs_quad_team(Cx& cx, const PbsArgs& A, uint64_t* acc, C2* xb, const C2* T1, const C2* T2, int& executed) {
  const int u = cx.u, h = cx.h, t = cx.t, g = 2 * h + t;
  const int k1 = u & 15, q = u >> 4;
  const int n = A.lwe_n;
  const bool cbs = A.lut == nullptr;
  const int log2n = 12;  // log2(2N)
  uint64_t* pa = acc + h * kN;
  C2* xown = xb + g * kXBuf;
#if defined(SPF_QUAD_TRACE) && defined(__CUDA_ARCH__)
  long long qt[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, qc = 0, qn = 0;
#define SPF_QT(k) do { const long long now_ = clock64(); qt[k] += now_ - qc; qc = now_; } while (0)
#else
#define SPF_QT(k) do { } while (0)
#endif
  // 1. acc = LUT * X^{-b~}: team (h, t) fills half t of polynomial h
  {
    uint64_t b = ldg_u64(A.lwe_in + n);
    if (cbs) b += 1ull << 62;
    const int bt = (int)modulus_switch(b, A.log_chi, A.log_v, log2n);
    const int rot = (2 * kN - bt) & (2 * kN - 1);
    const int v = 1 << A.log_v;
    for (int i = 16 * t; i < 16 * t + 16; i++) {
      const int j = u + 64 * i;
      int idx = j - rot;
      bool neg = false;
      if (idx < 0) { idx += kN; neg = true; }
      if (idx < 0) { idx += kN; neg = false; }
      uint64_t c;
      if (cbs) c = h ? cbs_lut_coeff(idx, A.cbs_radix_log, A.cbs_count, v) : 0;
      else c = ldg_u64(A.lut + h * kN + idx);
      pa[j] = neg ? 0 - c : c;
    }
  }
  cx.quad_sync();
  uint64_t a_next = n > 0 ? ldg_u64(A.lwe_in) : 0;
  uint64_t own[32];
#pragma unroll
  for (int i2 = 0; i2 < 32; i2++) own[i2] = pa[u + 64 * i2];
  // The BSK row of the NEXT executed step is staged in shared memory by a bulk copy (device: TMA,
  // cp.async.bulk + mbarrier) while the current step's inverse transform and the next forward
  // transform run, so the multiply-accumulate phase never waits for L2.
  auto next_executed = [&](int from) {  // first step >= from whose rotation is not the identity
    int j = from;
    while (j < n && modulus_switch(ldg_u64(A.lwe_in + j), A.log_chi, A.log_v, log2n) == 0) j++;
    return j;
  };
  {
    const int j0 = next_executed(0);
    if (j0 < n) cx.row_prefetch(A.bsk + (size_t)j0 * 8 * kM);
  }
#pragma unroll 1
  for (int i = 0; i < n; i++) {
    const int at = (int)modulus_switch(a_next, A.log_chi, A.log_v, log2n);
    if (i + 1 < n) a_next = ldg_u64(A.lwe_in + i + 1);
    if (at == 0) continue;
    const C2* ggsw = A.bsk + (size_t)i * 8 * kM;
#if defined(SPF_QUAD_TRACE) && defined(__CUDA_ARCH__)
    qc = clock64(); qn++;
#endif
    {
      C2 v[16];
      const int base = (u - at) & (2 * kN - 1);
      const char* col = reinterpret_cast<const char*>(pa) + 8 * (base & 63);
      const uint32_t bh9 = (uint32_t)(base >> 6) << 9;
      // The two teams of a polynomial need the same 32 rounded differences, one digit level each.  Each gathers HALF of
      // them (team t the coefficients 16 t .. 16 t + 15 of its column), keeps its own digit and hands the other level's
      // 16 digits, packed two to a word, to the partner thread (same u, other t) -- on the device through eight
      // tensor-memory columns of the lane the two threads share.  The digits are those of a full gather: a 16-bit digit d
      // is converted by digit_lo16_to_f64(d), which equals digit_hi16_to_f64(d << 16).
      uint32_t pk[8];
      auto gather_half = [&](auto tt) {  // the half is a compile-time constant: own[] stays in registers
        constexpr int T = decltype(tt)::value;
#pragma unroll
        for (int k = 0; k < 16; k++) {
          const int i2 = 16 * T + k;
          const uint32_t t9 = bh9 + 512u * i2;
          const uint64_t x = *reinterpret_cast<const uint64_t*>(col + (t9 & 0x3E00u));
          const uint64_t diff = ((t9 & 0x4000u) ? 0 - x : x) - own[i2];
          const uint32_t w = (uint32_t)(diff >> 32) + ((uint32_t)diff >> 31);
          const uint32_t w1 = w + 0x8000u;
          const uint32_t other = T ? (w & 0xFFFFu) : (w1 >> 16);  // the digit of level 1 - T
          if (T) v[k].y = digit_hi16_to_f64(w1); else v[k].x = digit_lo16_to_f64(w);
          if (k & 1) pk[k >> 1] |= other << 16; else pk[k >> 1] = other;
        }
      };
      if (t) gather_half(std::integral_constant<int, 1>{}); else gather_half(std::integral_constant<int, 0>{});
      cx.digit_xchg(pk);
#pragma unroll
      for (int k = 0; k < 16; k++) {
        const double d = digit_lo16_to_f64(pk[k >> 1] >> (16 * (k & 1)));
        if (t) v[k].x = d; else v[k].y = d;  // team 1 lacked the first half (real parts), team 0 the second
      }
      SPF_QT(0);
      fwd_pass1_core(v);
      cx.template t1_mul<false>(v, T1);
      fwd_x1_write(v, xown, u);
      cx.sync();
      SPF_QT(1);
      fwd_x1_read(v, xown, u);
      dft16<false>(v);
      fwd_x2_write(v, xown, u);  // in place; the pass-2 twiddles are applied by the readers below (as in pbs_pair_team)
      SPF_QT(2);
    }
    cx.quad_sync();
    SPF_QT(3);
    // MAD: team g owns the bins u + 64 (g + 4 k3) of every polynomial
    const C2* staged = cx.row_wait(executed, ggsw);  // this step's BSK row (device: in shared memory)
    executed++;
    SPF_QT(4);
    C2 f[2][4];
    double rtw[6];
    C2 rwi[3];
    cx.rt2(rtw, rwi, T2);  // this thread's pass-2 twiddles in the tan form (rt2_group_consts)
#pragma unroll
    for (int b = 0; b < 4; b++) {  // spectrum of team b = (hb, tb): digit tb <-> GLEV level 1 - tb
      const C2* grow = staged + (size_t)(((b >> 1) * 2 + (1 - (b & 1))) * 2) * kM;
      C2 d[4], g0[4], g1[4];
#pragma unroll
      for (int qp = 0; qp < 4; qp++) d[qp] = xb[b * kXBuf + k1 * kXPad + qp + 4 * q + 16 * g];
#pragma unroll
      for (int k3 = 0; k3 < 4; k3++) {
        g0[k3] = cx.row_load(grow + u + 64 * (g + 4 * k3));
        g1[k3] = cx.row_load(grow + kM + u + 64 * (g + 4 * k3));
      }
#pragma unroll
      for (int qp = 1; qp < 4; qp++) d[qp] = C2{spf_fma(-rtw[qp - 1], d[qp].y, d[qp].x), spf_fma(rtw[qp - 1], d[qp].x, d[qp].y)};
      bfly4_r<false>(d[0], d[1], d[2], d[3], rtw[3], rtw[4], rtw[5]);
#pragma unroll
      for (int k3 = 0; k3 < 4; k3++) {
        if (b == 0) { f[0][k3] = cmul(d[k3], g0[k3]); f[1][k3] = cmul(d[k3], g1[k3]); }
        else { cmad(f[0][k3], d[k3], g0[k3]); cmad(f[1][k3], d[k3], g1[k3]); }
      }
    }
    // first inverse pass; output polynomial p goes (in place) into the buffer of team (p, 0)
#pragma unroll
    for (int p = 0; p < 2; p++) {
      bfly4<true>(f[p][0], f[p][1], f[p][2], f[p][3]);
#pragma unroll
      for (int qp = 1; qp < 4; qp++) f[p][qp] = cmul_conj(f[p][qp], rwi[qp - 1]);  // the inverse transform's conjugate pass-2 twiddles
#pragma unroll
      for (int qp = 0; qp < 4; qp++) xb[2 * p * kXBuf + k1 * kXPad + qp + 4 * q + 16 * g] = f[p][qp];
    }
    SPF_QT(5);
    cx.quad_sync();
    SPF_QT(6);
    {  // every thread is done with the staged row: fetch the one of the next executed step
      const int jn = next_executed(i + 1);
      if (jn < n) cx.row_prefetch(A.bsk + (size_t)jn * 8 * kM);
    }
    if (t == 0) {
      C2 w[16];
      double ws[16];
      inv_x2_read(w, xown, u);
      dft16<true>(w);
      inv_x1_write(w, xown, u);  // in place
      cx.sync();
      SPF_QT(7);
      inv_x1_read(w, xown, u);
      cx.template t1_mul<true>(w, T1);
      inv_pass1_core_s(w, ws);
      SPF_QT(8);
      // as in pbs_pair_team: the saturating-cast corner of the conversion (probability ~2^-53 per value) is tested once
      // per 8 values, the fast conversion only tracks the largest exponent word it saw
#pragma unroll
      for (int m4 = 0; m4 < 16; m4 += 4) {
        uint32_t mag_max = 0;
        uint64_t r[8];
#pragma unroll
        for (int i = 0; i < 4; i++) {
          r[2 * i] = f64_to_torus_s_fast(w[m4 + i].x, ws[m4 + i], mag_max);
          r[2 * i + 1] = f64_to_torus_s_fast(w[m4 + i].y, ws[m4 + i], mag_max);
        }
        if (__builtin_expect(mag_max == kTorusCornerMag, 0)) {
#pragma unroll
          for (int i = 0; i < 4; i++) {
            r[2 * i] = f64_to_torus_s(w[m4 + i].x, ws[m4 + i]);
            r[2 * i + 1] = f64_to_torus_s(w[m4 + i].y, ws[m4 + i]);
          }
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const int m = m4 + i, j = u + 64 * m;
          own[m] += r[2 * i];
          own[m + 16] += r[2 * i + 1];
          pa[j] = own[m];
          pa[j + kM] = own[m + 16];
        }
      }
    }
    SPF_QT(9);
    cx.quad_sync();
    if (t == 1) {
#pragma unroll
      for (int i2 = 16; i2 < 32; i2++) own[i2] = pa[u + 64 * i2];
    }
  }
#if defined(SPF_QUAD_TRACE) && defined(__CUDA_ARCH__)
  if (threadIdx.x == 0 && blockIdx.x == 0 && qn > 0)
    printf("QT digits %lld p1 %lld p2 %lld qsync1 %lld rowwait %lld mad %lld qsync2 %lld inv2 %lld inv1 %lld store %lld steps %lld\n", qt[0] / qn, qt[1] / qn,
           qt[2] / qn, qt[3] / qn, qt[4] / qn, qt[5] / qn, qt[6] / qn, qt[7] / qn, qt[8] / qn, qt[9] / qn, qn);
#endif
  // 3. result: team (h, t) stores half t of polynomial h
  for (int i = 16 * t; i < 16 * t + 16; i++) {
    const int j = u + 64 * i;
    A.glwe_out[h * kN + j] = pa[j];
  }
}

// The 32 coefficients a thread holds after an inverse transform -> torus.  The saturating-cast corner of the conversion
// (|x| = 2^63 modulo 2^64, probability ~2^-53 per value) is tested once per 8 values: the fast conversion only tracks the
// largest exponent word it saw, and a group that hit the corner is redone with the complete conversion (same results).
SPF_HD void poly_to_torus(uint64_t (&r)[32], const C2 (&w)[16]) {
#pragma unroll
  for (int m4 = 0; m4 < 16; m4 += 4) {
    uint32_t mag_max = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      r[m4 + i] = f64_to_torus_impl<false, false>(w[m4 + i].x, 1.0, &mag_max);
      r[m4 + i + 16] = f64_to_torus_impl<false, false>(w[m4 + i].y, 1.0, &mag_max);
    }
    if (__builtin_expect(mag_max == kTorusCornerMag, 0)) {
#pragma unroll
      for (int i = 0; i < 4; i++) {
        r[m4 + i] = f64_to_torus(w[m4 + i].x);
        r[m4 + i + 16] = f64_to_torus(w[m4 + i].y);
      }
    }
  }
}

// ---- trace + scheme switch ---------------------------------------------------------------------
// One team = one (ciphertext, cbs level) pair: mod_switch_trace_and_rotate for that level
// (circuit_bootstrapping.rs:260-298), trace (ops/automorphisms/mod.rs:53-85) and that level's
// share of scheme_switch_fft (ops/fft_ops.rs:225-279,403-442), fused.
struct TraceSsArgs {
  const uint64_t* glwe_in;  // PBS output [2][2048] (CBS) or the GLWE to trace
  uint64_t* glev_out;       // optional: this level's traced GLWE [2][2048] (nullptr to skip)
  C2* ggsw_out;             // optional: GGSW base [row][level][p][bin]
  const C2* ak;             // [round][level][p][bin], 2^-10 scaled
  const C2* ssk;            // [level][p][bin], 2^-10 scaled
  const uint32_t* kinv;     // [11] inverse of k_r = N/2^(r-1)+1 modulo 2N
  int level;                // cbs level i
  int mode;                 // 0: CBS pre-processing + trace (+SS); 1: plain trace; 2: SS only (glwe_in = x_i)
  int cbs_radix_log, cbs_count;
  int tr_radix_log, tr_count;
  int ss_radix_log, ss_count;
  double out_scale;         // 1.0: GGSW stays device-resident (2^-10 convention); 1024.0: reference scale
  // Sharded graphs, peer-memory exchange: every GGSW element is also stored at the same offset in the arenas of
  // the other ranks (P2P over NVLink), peer_off[r] = byte distance from the local arena to peer r's arena.
  int n_peers;
  const long long* peer_off;
};

// PEERS is a compile-time switch: the replica / single-GPU instantiation carries no peer loop at all (the loop was
// unrolled for up to 7 peers behind predicates at each of the 64 store sites: 2 112 STG in a 19 k-instruction kernel
// whose instruction fetch already showed up in the stall samples).
template <bool PEERS>
SPF_HD void ggsw_store(const TraceSsArgs& A, C2* p, C2 v) {
  *p = v;
  if (PEERS) {
#pragma unroll 1
    for (int r = 0; r < A.n_peers; r++) *reinterpret_cast<C2*>(reinterpret_cast<char*>(p) + A.peer_off[r]) = v;
  }
}

// y[j] of sigma_k(p): polynomial_pow_k (ops/polynomial/mod.rs:62-87) as a gather.
SPF_HD uint64_t automorph_coeff(const uint64_t* p, int j, uint32_t kinv) {
  const uint32_t i = ((uint32_t)j * kinv) & (2 * kN - 1);
  return i < (uint32_t)kN ? p[i] : 0 - p[i - kN];
}

template <bool PEERS = true, class Cx>
SPF_HD void trace_ss_team(Cx& cx, const TraceSsArgs& A, uint64_t* g /*smem [2][2048]*/, C2* xbuf, const C2* T1,
                          const C2* T2) {
  const int u = cx.u;
  // ---- load / pre-process ----
  if (A.mode == 0) {
    // rotated.b[i'] += encode(1, 4(i'+1)+1) for i' <= level (cumulative, :284-285), * X^{-level},
    // then glwe_mod_switch_and_expand_pow_2 by log2 N (glwe_ciphertext_ops.rs:268-281)
    const int rot = (2 * kN - A.level) & (2 * kN - 1);
    for (int i = 0; i < 32; i++) {
      const int j = u + 64 * i;
      int idx = j - rot;
      bool neg = false;
      if (idx < 0) { idx += kN; neg = true; }
      if (idx < 0) { idx += kN; neg = false; }
      uint64_t ca = ldg_u64(A.glwe_in + idx), cb = ldg_u64(A.glwe_in + kN + idx);
      if (idx <= A.level) cb += 1ull << (64 - (A.cbs_radix_log * (idx + 1) + 1));
      if (neg) { ca = 0 - ca; cb = 0 - cb; }
      g[j] = (ca >> 11) + ((ca >> 10) & 1);
      g[kN + j] = (cb >> 11) + ((cb >> 10) & 1);
    }
  } else {
    for (int i = 0; i < 32; i++) {
      const int j = u + 64 * i;
      g[j] = ldg_u64(A.glwe_in + j);
      g[kN + j] = ldg_u64(A.glwe_in + kN + j);
    }
  }
  cx.sync();
  // ---- trace ----
  if (A.mode != 2) {
    for (int r = 0; r < 11; r++) {
      const uint32_t kinv = A.kinv[r];
      C2 f[2][16];
      zero_acc(f);
      gadget_mad_stateless(cx, f, [&](int j) { return automorph_coeff(g, j, kinv); }, xbuf, T1, T2,
                           A.ak + (size_t)r * A.tr_count * 2 * kM, A.tr_radix_log, A.tr_count);
      // keyswitch_glwe_to_glwe (fft_ops.rs:457-495): ks = (0, y_b) - IFFT(sum); out += ks
      team_fft_inv(cx, f[1], xbuf, T1, T2);
      uint64_t db[32];
      poly_to_torus(db, f[1]);  // db[m] / db[m + 16]: coefficients u + 64 m and u + 64 m + 1024
#pragma unroll
      for (int m = 0; m < 16; m++) {
        const int j = u + 64 * m;
        db[m] = automorph_coeff(g + kN, j, kinv) - db[m];
        db[m + 16] = automorph_coeff(g + kN, j + kM, kinv) - db[m + 16];
      }
      team_fft_inv(cx, f[0], xbuf, T1, T2);
      cx.sync();  // every gather of this round is done
      {
        uint64_t da[32];
        poly_to_torus(da, f[0]);
#pragma unroll
        for (int m = 0; m < 16; m++) {
          const int j = u + 64 * m;
          g[j] -= da[m];
          g[j + kM] -= da[m + 16];
          g[kN + j] += db[m];
          g[kN + j + kM] += db[m + 16];
        }
      }
      cx.sync();
    }
    if (A.glev_out) {
      for (int i = 0; i < 32; i++) {
        const int j = u + 64 * i;
        A.glev_out[j] = g[j];
        A.glev_out[kN + j] = g[kN + j];
      }
    }
  }
  // ---- scheme switch share of this level (k = 1) ----
  if (A.ggsw_out) {
    const size_t glwe_f = 2 * kM;
    C2* row0 = A.ggsw_out + ((size_t)0 * A.cbs_count + A.level) * glwe_f;
    C2* row1 = A.ggsw_out + ((size_t)1 * A.cbs_count + A.level) * glwe_f;
    C2 f[2][16];
    // FFT(x.b): row 1 b-slot, and the a-slot of row 0 (update_encrypted_secret_key_component_fft)
    team_poly_fft(cx, f[0], [&](int j) { return g[kN + j]; }, xbuf, T1, T2);
#pragma unroll
    for (int s = 0; s < 16; s++) { ggsw_store<PEERS>(A, row1 + kM + bin_of(u, s), cscale(f[0][s], A.out_scale)); f[1][s] = C2{0.0, 0.0}; }
    gadget_mad_stateless(cx, f, [&](int j) { return g[j]; }, xbuf, T1, T2, A.ssk, A.ss_radix_log, A.ss_count);
#pragma unroll
    for (int s = 0; s < 16; s++) {
      ggsw_store<PEERS>(A, row0 + bin_of(u, s), cscale(f[0][s], A.out_scale));
      ggsw_store<PEERS>(A, row0 + kM + bin_of(u, s), cscale(f[1][s], A.out_scale));
    }
    // row 1 a-slot: FFT(x.a)
    team_poly_fft(cx, f[0], [&](int j) { return g[j]; }, xbuf, T1, T2);
#pragma unroll
    for (int s = 0; s < 16; s++) ggsw_store<PEERS>(A, row1 + bin_of(u, s), cscale(f[0][s], A.out_scale));
  }
}

// ---- WIDE CMUX: one CMUX / external product on 8 teams ------------------------------------------
// A CMUX inside a ripple MUX chain (one per dependency level) is pure latency: cmux_team runs its
// 8 forward transforms, 16 multiply-accumulates and 2 inverse transforms one after the other on 64
// threads.  Here team j = 4 r + t transforms digit t of polynomial r of d1 - d0 (digits straight
// from the bit fields of the rounded value, see radix_offset), all 8 concurrently; then every
// thread of the CTA finishes the radix-4 pass for ONE group of 4 bins of ONE output polynomial over
// all 8 spectra and multiply-accumulates it against the GGSW; teams 0 and 1 run the two inverse
// transforms.  Critical path: 1 forward + 1 MAD phase + 1 inverse instead of 8 + 16 + 2.
//   cx.u / cx.team: thread in team, team 0..7;  cx.sync(): team barrier;  cx.cta_sync(): all 512
//   xb: 8 exchange buffers.  count must be 4 (k = 1): 2 polynomials x 4 levels = 8 teams.
constexpr int kWideTeams = 8;
#if defined(SPF_WIDE_TRACE) && defined(__CUDA_ARCH__)
#define SPF_WT(k) do { if (threadIdx.x == 0 && blockIdx.x == 0) wt[k] = clock64(); } while (0)
#else
#define SPF_WT(k) do { } while (0)
#endif
template <class Cx>
SPF_HD void cmux_wide(Cx& cx, uint64_t* out, const uint64_t* d0, const uint64_t* d1, const C2* ggsw, C2* xb,
                      const C2* T1, const C2* T2, int radix_log, int count) {
  const int u = cx.u, team = cx.team;
  const int r = team / count, t = team % count;
  C2* xown = xb + team * kXBuf;
#if defined(SPF_WIDE_TRACE) && defined(__CUDA_ARCH__)
  long long wt[8];
#endif
  SPF_WT(0);
  {
    const uint64_t off = radix_offset(radix_log, count);
    const uint64_t dmask = (1ull << radix_log) - 1;
    const int32_t half = 1 << (radix_log - 1);
    C2 v[16];
    const int shift = 64 - radix_log * count;
    if (shift >= 33) {
      // All digits and the rounding bit lie in the high word (cbs_radix: 16 bits): digit_t is a bit field of
      // hi(x) + round + offset, 32-bit arithmetic only (the general form below costs ~2.5x the integer work).
      const uint32_t c1 = (1u << (shift - 33)) + ((uint32_t)off << (shift - 32));
      const int sh = shift - 32 + t * radix_log;
#pragma unroll
      for (int m = 0; m < 16; m++) {
        const int j = r * kN + u + 64 * m;
        const uint64_t x0 = d0 ? d1[j] - d0[j] : d1[j];  // d0 / d1 may be shared-memory copies (cmux_wide_kernel)
        const uint64_t x1 = d0 ? d1[j + kM] - d0[j + kM] : d1[j + kM];
        v[m].x = i32_to_f64((int32_t)((((uint32_t)(x0 >> 32) + c1) >> sh) & (uint32_t)dmask) - half);
        v[m].y = i32_to_f64((int32_t)((((uint32_t)(x1 >> 32) + c1) >> sh) & (uint32_t)dmask) - half);
      }
    } else {
#pragma unroll
      for (int m = 0; m < 16; m++) {
        const int j = r * kN + u + 64 * m;
        const uint64_t x0 = d0 ? d1[j] - d0[j] : d1[j];
        const uint64_t x1 = d0 ? d1[j + kM] - d0[j + kM] : d1[j + kM];
        const uint64_t r0 = radix_round(x0, radix_log, count) + off, r1 = radix_round(x1, radix_log, count) + off;
        v[m].x = i32_to_f64((int32_t)((r0 >> (t * radix_log)) & dmask) - half);
        v[m].y = i32_to_f64((int32_t)((r1 >> (t * radix_log)) & dmask) - half);
      }
    }
    SPF_WT(1);
    fwd_pass1_core(v);
#pragma unroll
    for (int k1i = 0; k1i < 16; k1i++) v[k1i] = cmul(v[k1i], T1[k1i * 64 + u]);
    fwd_x1_write(v, xown, u);
    cx.sync();
    SPF_WT(2);
    fwd_x1_read(v, xown, u);
    dft16<false>(v);
    {
      const int qq = u >> 4;
#pragma unroll
      for (int k2i = 1; k2i < 16; k2i++) v[k2i] = cmul(v[k2i], T2[qq * kT2Pad + k2i]);
    }
    fwd_x2_write(v, xown, u);  // in place
  }
  cx.cta_sync();
  SPF_WT(3);
  // ---- MAD: thread (p, k1, k2) owns bins k1 + 16 k2 + 256 k3, k3 = 0..3, of output polynomial p ----
  const int tid = team * kTeam + u;
  const int p = tid >> 8, k1 = tid & 15, k2 = (tid >> 4) & 15;
  C2 f[4];
#pragma unroll
  for (int jb = 0; jb < 2 * 4; jb += 4) {  // 4 spectra per batch: their GGSW values are requested together
    C2 g[4][4], d[4][4];
#pragma unroll
    for (int jj = 0; jj < 4; jj++) {
      const int j = jb + jj, rr = j / count, tt = j % count;  // digit tt <-> GGSW level count-1-tt (fft_ops.rs:92)
      const C2* grow = ggsw + ((size_t)(rr * count + (count - 1 - tt)) * 2 + p) * kM;
#pragma unroll
      for (int k3 = 0; k3 < 4; k3++) g[jj][k3] = ldg_c2(grow + k1 + 16 * k2 + 256 * k3);
#pragma unroll
      for (int qp = 0; qp < 4; qp++) d[jj][qp] = xb[j * kXBuf + k1 * kXPad + qp + 4 * k2];
    }
#pragma unroll
    for (int jj = 0; jj < 4; jj++) {
      bfly4<false>(d[jj][0], d[jj][1], d[jj][2], d[jj][3]);
#pragma unroll
      for (int k3 = 0; k3 < 4; k3++) {
        if (jb + jj == 0) f[k3] = cmul(d[jj][k3], g[jj][k3]);
        else cmad(f[k3], d[jj][k3], g[jj][k3]);
      }
    }
  }
  bfly4<true>(f[0], f[1], f[2], f[3]);
  SPF_WT(4);
  cx.cta_sync();  // every spectrum has been consumed: buffers 0 and 1 take the two outputs
#pragma unroll
  for (int qp = 0; qp < 4; qp++) xb[p * kXBuf + k1 * kXPad + qp + 4 * k2] = f[qp];
  cx.cta_sync();
  SPF_WT(5);
  if (team < 2) {  // team p finishes the inverse transform of output polynomial p
    C2 w[16];
    double ws[16];
    inv_x2_read(w, xown, u);
    inv_pass2(w, u, T2);
    inv_x1_write(w, xown, u);  // in place
    cx.sync();
    SPF_WT(6);
    inv_x1_read(w, xown, u);
#pragma unroll
    for (int k1i = 0; k1i < 16; k1i++) w[k1i] = cmul_conj(w[k1i], T1[k1i * 64 + u]);
    inv_pass1_core_s(w, ws);
    SPF_WT(7);
#pragma unroll
    for (int m = 0; m < 16; m++) {
      const int j = team * kN + u + 64 * m;
      uint64_t re = f64_to_torus_s(w[m].x, ws[m]), im = f64_to_torus_s(w[m].y, ws[m]);
      if (d0) { re += d0[j]; im += d0[j + kM]; }
      out[j] = re;
      out[j + kM] = im;
    }
#if defined(SPF_WIDE_TRACE) && defined(__CUDA_ARCH__)
    if (threadIdx.x == 0 && blockIdx.x == 0)
      printf("WT load %lld p1 %lld p2 %lld mad %lld sync %lld inv2 %lld inv1 %lld store %lld total %lld\n", wt[1] - wt[0], wt[2] - wt[1],
             wt[3] - wt[2], wt[4] - wt[3], wt[5] - wt[4], wt[6] - wt[5], wt[7] - wt[6], clock64() - wt[7], clock64() - wt[0]);
#endif
  }
}

}  // namespace spf
