// fft16.cuh -- the negacyclic f64 FFT of an N=2048 torus polynomial for one TEAM of 64 threads,
// 16 complex points per thread held in registers.  Replaces TwistedFft::{forward,reverse}
// (sunscreen_tfhe/src/math/fft/negacyclic/mod.rs:96-122) + complex_twist/untwist
// (math/simd/scalar.rs:19-35) + the rustfft butterflies behind them.
//
// Everything here is __host__ __device__: the SAME index arithmetic is executed on the CPU
// by csrc/emu.cpp (one loop iteration per virtual thread, phases split at the barriers) so the
// factorisation is validated against the oracle without a GPU.
//
// Factorisation of the length-1024 complex DFT: 1024 = 16 x 16 x 4.
//   n = a + 64 m           (a = thread, m = register)           time index
//   k = k1 + 16 (k2 + 16 k3)                                    frequency index
//   pass 1  thread a      : u[m] = x[m] * e^{i pi m/32}  (the m-part of the twist, constants)
//                           y[k1] = DFT16_m(u) * T1[a][k1],  T1 = e^{i pi a/2048} * W1024^{a k1}
//   xchg 1  (smem)        : thread (k1,q) gathers y[q + 4 m'][k1], m' = 0..15
//   pass 2  thread (k1,q) : z[k2] = DFT16_m'(y) * W64^{q k2}
//   xchg 2  (smem)        : thread (k1,q) gathers z[k1][q'][k2] for q'=0..3, k2 = q + 4 j
//   pass 3  thread (k1,q) : X[k1 + 16 k2 + 256 k3] = DFT4_q'(z)      -> slot s = 4 j + k3
// The inverse runs the adjoint passes in reverse order (no bit-reversal anywhere): the forward
// output ownership (thread u, slot s) is exactly the inverse input ownership, so FFT-domain
// accumulators never leave registers.  Frequency-domain arrays in device memory keep the
// reference's natural bin order: register slot s of thread u is bin spf::bin_of(u, s).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define SPF_HD __host__ __device__ __forceinline__
#else
#define SPF_HD inline __attribute__((always_inline))
#endif

#include "fft_consts.h"

namespace spf {

struct alignas(16) C2 {
  double x, y;
};

constexpr int kN = 2048;        // polynomial degree (DEFAULT_128 l1_params)
constexpr int kM = 1024;        // complex FFT length
constexpr int kTeam = 64;       // threads per polynomial transform
constexpr int kR = 16;          // complex points per thread
constexpr int kXPad = 65;       // exchange-buffer row stride in complex elements (odd: conflict-free)
constexpr int kXBuf = 16 * kXPad;  // complex elements per team exchange buffer (16640 B)
constexpr int kT2Pad = 17;
constexpr int kT1Elems = 16 * 64;
constexpr int kT2Elems = 4 * kT2Pad;

// Register slot s = 4 j + k3 of thread u = k1 + 16 q holds frequency bin
//   k = k1 + 16 (q + 4 j) + 256 k3 = u + 64 * slot_row(s),
// so FFT-domain arrays stay in the reference's natural bin order in memory and every slot is a
// fully coalesced row of 64 consecutive complex values.
SPF_HD constexpr int slot_row(int s) { return (s >> 2) + 4 * (s & 3); }
SPF_HD constexpr int bin_of(int u, int s) { return u + 64 * slot_row(s); }

SPF_HD C2 cadd(C2 a, C2 b) { return C2{a.x + b.x, a.y + b.y}; }
SPF_HD C2 csub(C2 a, C2 b) { return C2{a.x - b.x, a.y - b.y}; }
// Every multiply-add of the hot path is an EXPLICIT fma: the library is compiled with -fmad=false and
// the host emulator with -ffp-contract=off, so neither compiler chooses which product of
// `a*b - c*d` to fuse and the GPU and the emulator produce bit-identical doubles
// (tests/test_gpu_parity.py::test_pbs_bit_exact_vs_emulator).
SPF_HD double spf_fma(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
  return fma(a, b, c);
#else
  return __builtin_fma(a, b, c);
#endif
}
// a * (c + i s)
SPF_HD C2 cmul_cs(C2 a, double c, double s) {
  return C2{spf_fma(a.x, c, -(a.y * s)), spf_fma(a.x, s, a.y * c)}; }
SPF_HD C2 cmul(C2 a, C2 b) {
  return C2{spf_fma(a.x, b.x, -(a.y * b.y)), spf_fma(a.x, b.y, a.y * b.x)}; }
SPF_HD C2 cmul_conj(C2 a, C2 b) {
  return C2{spf_fma(a.x, b.x, a.y * b.y), spf_fma(a.y, b.x, -(a.x * b.y))}; }  // a * conj(b)
// acc += a * b as four chained FMAs
SPF_HD void cmad(C2& acc, C2 a, C2 b) {
  acc.x = spf_fma(-a.y, b.y, spf_fma(a.x, b.x, acc.x));
  acc.y = spf_fma(a.y, b.x, spf_fma(a.x, b.y, acc.y));
}

// 4-point DFT in place: (a,b,c,d) -> (X0,X1,X2,X3); INV uses e^{+...}
template <bool INV>
SPF_HD void bfly4(C2& a, C2& b, C2& c, C2& d) {
  C2 apc = cadd(a, c), amc = csub(a, c), bpd = cadd(b, d), bmd = csub(b, d);
  a = cadd(apc, bpd);
  c = csub(apc, bpd);
  if (!INV) {
    b = C2{amc.x + bmd.y, amc.y - bmd.x};
    d = C2{amc.x - bmd.y, amc.y + bmd.x};
  } else {
    b = C2{amc.x - bmd.y, amc.y + bmd.x};
    d = C2{amc.x + bmd.y, amc.y - bmd.x};
  }
}

// ---- constant providers -----------------------------------------------------------------------------------------------
// The deferred-scale transforms below take their ~40 distinct double constants per pass (tangents, scale ratios) from a
// PROVIDER kp(v); KLit returns the literal, which the device code materialises as FMA immediates.  (Reading them from a
// __constant__ pool instead was measured: no gain in pbs_kernel, 6.75 vs 6.73 ms per wave, and spills in the 255-register
// trace_ss_kernel, 7.4 -> 9.0 ms.)
struct KLit {
  SPF_HD double operator()(double v) { return v; }
};

// ---- deferred-scale arithmetic --------------------------------------------------------------
// Inside the in-register transforms a value is a pair (v, s): the true value is s * v, where s is a
// real constant that is known at compile time once the loops are unrolled (on the device every s
// below folds into FMA immediates; the host emulator simply computes them).  A rotation by a
// constant angle then costs 2 FMAs instead of the 4 operations of a complex multiply:
//   e^{i t} = cos t (1 + i tan t)  or  sin t (cot t + i)     (whichever factor is larger in magnitude)
// and the factored-out cos / sin goes into s; adding two values of different scale costs one FMA
// per component (a + (s_b / s_a) b, scale s_a), the same as the plain add.  A 16-point DFT with its
// inter-stage twiddles therefore needs 128 + 18 instead of 128 + 36 FP64 instructions, the twist of
// pass 1 30 instead of 60 (Linzer-Feig style FMA butterflies).
SPF_HD constexpr double spf_abs(double x) { return x < 0 ? -x : x; }
// (v, s) *= e^{i pi e / 32}
template <class KP>
SPF_HD void rot_s(C2& v, double& s, int e, KP& kp) {
  e &= 63;
  if (e == 0) return;
  // quarter turns are sign changes and swaps (they fold into the operand modifiers of the next FMA); the tan / cot form
  // below would spend two FMAs with a zero factor on them (the compiler may not drop fma(0, x, y): x could be NaN)
  if (e == 16) { v = C2{-v.y, v.x}; return; }
  if (e == 32) { v = C2{-v.x, -v.y}; return; }
  if (e == 48) { v = C2{v.y, -v.x}; return; }
  const double c = spf_cos32(e), sn = spf_sin32(e);
  if (spf_abs(c) >= spf_abs(sn)) {
    const double t = kp(sn / c);
    v = C2{spf_fma(-t, v.y, v.x), spf_fma(t, v.x, v.y)};
    s *= c;
  } else {
    const double t = kp(c / sn);
    v = C2{spf_fma(t, v.x, -v.y), spf_fma(t, v.y, v.x)};
    s *= sn;
  }
}
SPF_HD void rot_s(C2& v, double& s, int e) {
  KLit kp;
  rot_s(v, s, e, kp);
}
// 4-point DFT of (a, sa) .. (d, sd); all four results carry scale sa.
template <bool INV, class KP>
SPF_HD void bfly4_s(C2& a, C2& b, C2& c, C2& d, double sa, double sb, double sc, double sd, KP& kp) {
  const double rc = kp(sc / sa), rd = kp(sd / sb), rb = kp(sb / sa);
  const C2 apc{spf_fma(rc, c.x, a.x), spf_fma(rc, c.y, a.y)}, amc{spf_fma(-rc, c.x, a.x), spf_fma(-rc, c.y, a.y)};
  const C2 bpd{spf_fma(rd, d.x, b.x), spf_fma(rd, d.y, b.y)}, bmd{spf_fma(-rd, d.x, b.x), spf_fma(-rd, d.y, b.y)};
  a = C2{spf_fma(rb, bpd.x, apc.x), spf_fma(rb, bpd.y, apc.y)};
  c = C2{spf_fma(-rb, bpd.x, apc.x), spf_fma(-rb, bpd.y, apc.y)};
  if (!INV) {
    b = C2{spf_fma(rb, bmd.y, amc.x), spf_fma(-rb, bmd.x, amc.y)};
    d = C2{spf_fma(-rb, bmd.y, amc.x), spf_fma(rb, bmd.x, amc.y)};
  } else {
    b = C2{spf_fma(-rb, bmd.y, amc.x), spf_fma(rb, bmd.x, amc.y)};
    d = C2{spf_fma(rb, bmd.y, amc.x), spf_fma(-rb, bmd.x, amc.y)};
  }
}

template <bool INV>
SPF_HD void bfly4_s(C2& a, C2& b, C2& c, C2& d, double sa, double sb, double sc, double sd) {
  KLit kp;
  bfly4_s<INV>(a, b, c, d, sa, sb, sc, sd, kp);
}
// The same butterfly with the three scale ratios given at RUN time (rb = sb / sa, rc = sc / sa, rd = sd / sb; results carry
// scale sa): the reader-side pass-2 twiddles of the pair kernel (team_ops.cuh: rt2_fwd_consts) arrive as per-thread constants.
template <bool INV>
SPF_HD void bfly4_r(C2& a, C2& b, C2& c, C2& d, double rb, double rc, double rd) {
  const C2 apc{spf_fma(rc, c.x, a.x), spf_fma(rc, c.y, a.y)}, amc{spf_fma(-rc, c.x, a.x), spf_fma(-rc, c.y, a.y)};
  const C2 bpd{spf_fma(rd, d.x, b.x), spf_fma(rd, d.y, b.y)}, bmd{spf_fma(-rd, d.x, b.x), spf_fma(-rd, d.y, b.y)};
  a = C2{spf_fma(rb, bpd.x, apc.x), spf_fma(rb, bpd.y, apc.y)};
  c = C2{spf_fma(-rb, bpd.x, apc.x), spf_fma(-rb, bpd.y, apc.y)};
  if (!INV) {
    b = C2{spf_fma(rb, bmd.y, amc.x), spf_fma(-rb, bmd.x, amc.y)};
    d = C2{spf_fma(-rb, bmd.y, amc.x), spf_fma(rb, bmd.x, amc.y)};
  } else {
    b = C2{spf_fma(-rb, bmd.y, amc.x), spf_fma(rb, bmd.x, amc.y)};
    d = C2{spf_fma(rb, bmd.y, amc.x), spf_fma(-rb, bmd.x, amc.y)};
  }
}

// 16-point DFT, natural order in -> natural order out, all twiddles compile-time constants.
// Inputs (v[i], s[i]); every output carries the INPUT scale s[0] (each butterfly group takes the
// scale of its first element, and the first element of every second-layer group descends from
// v[0] without a twiddle), so the results are plain values whenever s[0] == 1.
template <bool INV, class KP>
SPF_HD void dft16_s(C2 (&v)[16], double (&s)[16], KP& kp) {
#pragma unroll
  for (int m0 = 0; m0 < 4; m0++) {
    bfly4_s<INV>(v[m0], v[m0 + 4], v[m0 + 8], v[m0 + 12], s[m0], s[m0 + 4], s[m0 + 8], s[m0 + 12], kp);
    s[m0 + 4] = s[m0 + 8] = s[m0 + 12] = s[m0];
  }
  // v[m0 + 4 kl] = Y[m0][kl];  twiddle W16^{m0 kl}
#pragma unroll
  for (int m0 = 1; m0 < 4; m0++) {
#pragma unroll
    for (int kl = 1; kl < 4; kl++) {
      const int e = 4 * m0 * kl;  // angle pi*e/32 = 2 pi m0 kl / 16
      rot_s(v[m0 + 4 * kl], s[m0 + 4 * kl], INV ? e : 64 - e, kp);
    }
  }
#pragma unroll
  for (int kl = 0; kl < 4; kl++) {
    bfly4_s<INV>(v[4 * kl], v[4 * kl + 1], v[4 * kl + 2], v[4 * kl + 3], s[4 * kl], s[4 * kl + 1], s[4 * kl + 2], s[4 * kl + 3], kp);
    s[4 * kl + 1] = s[4 * kl + 2] = s[4 * kl + 3] = s[4 * kl];
  }
  // v[4 kl + kh] = X[kl + 4 kh] -> natural order
  C2 t[16];
  double ts[16];
#pragma unroll
  for (int i = 0; i < 16; i++) { t[i] = v[i]; ts[i] = s[i]; }
#pragma unroll
  for (int kl = 0; kl < 4; kl++) {
#pragma unroll
    for (int kh = 0; kh < 4; kh++) { v[kl + 4 * kh] = t[4 * kl + kh]; s[kl + 4 * kh] = ts[4 * kl + kh]; }
  }
}
template <bool INV>
SPF_HD void dft16_s(C2 (&v)[16], double (&s)[16]) {
  KLit kp;
  dft16_s<INV>(v, s, kp);
}
template <bool INV, class KP>
SPF_HD void dft16_k(C2 (&v)[16], KP& kp) {
  double s[16];
#pragma unroll
  for (int i = 0; i < 16; i++) s[i] = 1.0;
  dft16_s<INV>(v, s, kp);  // unit input scales -> unit output scales
}
template <bool INV>
SPF_HD void dft16(C2 (&v)[16]) {
  KLit kp;
  dft16_k<INV>(v, kp);
}

// ------------------------------------------------------------------------------------------
// forward passes.  v[m] on entry to fwd_pass1 = (p[a + 64 m], p[a + 64 m + 1024]) as doubles.
// ------------------------------------------------------------------------------------------
// pass 1 without its thread-dependent twiddle (applied by the caller: table in shared memory
// below, or the thread's tensor-memory columns in the blind-rotation kernel)
template <class KP>
SPF_HD void fwd_pass1_core_k(C2 (&v)[16], KP& kp) {
  double s[16];
  s[0] = 1.0;
#pragma unroll
  for (int m = 1; m < 16; m++) { s[m] = 1.0; rot_s(v[m], s[m], m, kp); }
  dft16_s<false>(v, s, kp);  // the twist factors fold into the butterflies; outputs carry s[0] = 1
}
SPF_HD void fwd_pass1_core(C2 (&v)[16]) {
  KLit kp;
  fwd_pass1_core_k(v, kp);
}
SPF_HD void fwd_pass1(C2 (&v)[16], int a, const C2* T1) {
  fwd_pass1_core(v);
#pragma unroll
  for (int k1 = 0; k1 < 16; k1++) v[k1] = cmul(v[k1], T1[k1 * 64 + a]);
}
SPF_HD void fwd_x1_write(const C2 (&v)[16], C2* buf, int a) {
#pragma unroll
  for (int k1 = 0; k1 < 16; k1++) buf[k1 * kXPad + a] = v[k1];
}
SPF_HD void fwd_x1_read(C2 (&v)[16], const C2* buf, int u) {
  const int k1 = u & 15, q = u >> 4;
#pragma unroll
  for (int mp = 0; mp < 16; mp++) v[mp] = buf[k1 * kXPad + q + 4 * mp];
}
SPF_HD void fwd_pass2(C2 (&v)[16], int u, const C2* T2) {
  const int q = u >> 4;
  dft16<false>(v);
#pragma unroll
  for (int k2 = 1; k2 < 16; k2++) v[k2] = cmul(v[k2], T2[q * kT2Pad + k2]);
}
// Second exchange, IN PLACE: thread (k1, q) stores z[k2] at (row k1, column q + 4 k2), exactly the
// 16 locations it has just read in fwd_x1_read, so no barrier is needed between that read and this
// write (each thread only overwrites what it alone consumed).  The reader of pass 3, thread
// (k1, q), finds z of thread (k1, q') for k2 = q + 4 j at column q' + 4 q + 16 j of row k1.
SPF_HD void fwd_x2_write(const C2 (&v)[16], C2* buf, int u) {
  const int k1 = u & 15, q = u >> 4;
#pragma unroll
  for (int k2 = 0; k2 < 16; k2++) buf[k1 * kXPad + q + 4 * k2] = v[k2];
}
SPF_HD void fwd_x2_read(C2 (&v)[16], const C2* buf, int u) {
  const int k1 = u & 15, q = u >> 4;
#pragma unroll
  for (int j = 0; j < 4; j++) {
#pragma unroll
    for (int qp = 0; qp < 4; qp++) v[4 * j + qp] = buf[k1 * kXPad + qp + 4 * q + 16 * j];
  }
}
SPF_HD void fwd_pass3(C2 (&v)[16]) {
#pragma unroll
  for (int j = 0; j < 4; j++) bfly4<false>(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}

// ------------------------------------------------------------------------------------------
// inverse passes (adjoint of the forward ones).  On exit from inv_pass1,
// v[m] = (re, im) with re -> coefficient a + 64 m, im -> coefficient a + 64 m + 1024, both
// multiplied by 1024 (the 1/(N/2) of complex_untwist is folded into the key material).
// ------------------------------------------------------------------------------------------
SPF_HD void inv_pass3(C2 (&v)[16]) {
#pragma unroll
  for (int j = 0; j < 4; j++) bfly4<true>(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}
// Inverse direction, same in-place layout: inv_x2_read takes the 16 locations (row k1, column
// q + 4 k2) that inv_x1_write of the same thread overwrites next, so no barrier separates them.
SPF_HD void inv_x2_write(const C2 (&v)[16], C2* buf, int u) {
  const int k1 = u & 15, q = u >> 4;
#pragma unroll
  for (int j = 0; j < 4; j++) {
#pragma unroll
    for (int qp = 0; qp < 4; qp++) buf[k1 * kXPad + qp + 4 * q + 16 * j] = v[4 * j + qp];
  }
}
SPF_HD void inv_x2_read(C2 (&v)[16], const C2* buf, int u) {
  const int k1 = u & 15, q = u >> 4;
#pragma unroll
  for (int k2 = 0; k2 < 16; k2++) v[k2] = buf[k1 * kXPad + q + 4 * k2];
}
SPF_HD void inv_pass2(C2 (&v)[16], int u, const C2* T2) {
  const int q = u >> 4;
#pragma unroll
  for (int k2 = 1; k2 < 16; k2++) v[k2] = cmul_conj(v[k2], T2[q * kT2Pad + k2]);
  dft16<true>(v);
}
SPF_HD void inv_x1_write(const C2 (&v)[16], C2* buf, int u) {
  const int k1 = u & 15, q = u >> 4;
#pragma unroll
  for (int mp = 0; mp < 16; mp++) buf[k1 * kXPad + q + 4 * mp] = v[mp];
}
SPF_HD void inv_x1_read(C2 (&v)[16], const C2* buf, int a) {
#pragma unroll
  for (int k1 = 0; k1 < 16; k1++) v[k1] = buf[k1 * kXPad + a];
}
// Inverse pass 1 with the untwist left as a deferred scale: true outputs are s[m] * v[m]
// (consumed by f64_to_torus_s, whose first two operations absorb the factor as FMAs).
template <class KP>
SPF_HD void inv_pass1_core_s_k(C2 (&v)[16], double (&s)[16], KP& kp) {
#pragma unroll
  for (int i = 0; i < 16; i++) s[i] = 1.0;
  dft16_s<true>(v, s, kp);
#pragma unroll
  for (int m = 1; m < 16; m++) rot_s(v[m], s[m], 64 - m, kp);
#pragma unroll
  for (int m = 1; m < 16; m++) s[m] = kp(s[m]);  // the output scales come from the provider too (consumed as FMA factors)
}
SPF_HD void inv_pass1_core_s(C2 (&v)[16], double (&s)[16]) {
  KLit kp;
  inv_pass1_core_s_k(v, s, kp);
}
SPF_HD void inv_pass1_core(C2 (&v)[16]) {
  double s[16];
  inv_pass1_core_s(v, s);
#pragma unroll
  for (int m = 1; m < 16; m++) v[m] = C2{v[m].x * s[m], v[m].y * s[m]};
}
SPF_HD void inv_pass1(C2 (&v)[16], int a, const C2* T1) {
#pragma unroll
  for (int k1 = 0; k1 < 16; k1++) v[k1] = cmul_conj(v[k1], T1[k1 * 64 + a]);
  inv_pass1_core(v);
}

// ------------------------------------------------------------------------------------------
// scalar conversions
// ------------------------------------------------------------------------------------------

// int32 -> f64
SPF_HD double i32_to_f64(int32_t x) {
#if defined(__CUDA_ARCH__)
  // the conversion pipe is idle in these kernels while the FP64 pipe and the issue slots are not: one I2F.F64.S32 instead of
  // an integer op, a move and a DADD (same value)
  return __int2double_rn(x);
#else
  // without a conversion: 2^52 + 2^31 + x is exact, subtract the bias
  uint64_t bits = 0x4330000000000000ull | (uint64_t)((uint32_t)x ^ 0x80000000u);
  double d;
  __builtin_memcpy(&d, &bits, 8);
  return d - 4503601774854144.0;  // 2^52 + 2^31
#endif
}

// int64 -> f64, round to nearest even (what `as f64` does; entities/polynomial.rs:264-268).
SPF_HD double i64_to_f64(int64_t x) {
#if defined(__CUDA_ARCH__)
  return __ll2double_rn((long long)x);
#else
  return (double)x;
#endif
}

SPF_HD uint64_t f64_bits(double x) {
#if defined(__CUDA_ARCH__)
  return (uint64_t)__double_as_longlong(x);
#else
  uint64_t b;
  __builtin_memcpy(&b, &x, 8);
  return b;
#endif
}
SPF_HD double bits_f64(uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __longlong_as_double((long long)b);
#else
  double x;
  __builtin_memcpy(&x, &b, 8);
  return x;
#endif
}
// f64 -> i64, truncating and saturating (Rust's `as i64`, math/torus.rs:181-185)
SPF_HD int64_t f64_to_i64_sat(double x) {
#if defined(__CUDA_ARCH__)
  return (int64_t)__double2ll_rz(x);
#else
  if (x != x) return 0;
  if (x >= 9223372036854775808.0) return INT64_MAX;
  if (x < -9223372036854775808.0) return INT64_MIN;
  return (int64_t)x;
#endif
}

// f64 -> torus: complex_untwist's round() (half away from zero, simd/scalar.rs:32-33) followed by
// vector_mod_pow2_q_f64 for q = 2^64 (scalar.rs:75-119) and the saturating `as i64`
// (math/torus.rs:181-185).  Four DP ops + one conversion instead of ~25 integer ops:
//   h  = rint(x / 2^64) * 2^64     (add/sub of 1.5*2^116, whose ulp is 2^64; |x| < 2^115, FFT
//                                   outputs are < 2^100)
//   lo = x - h                     (exact; |lo| <= 2^63)
//   r  = trunc(lo +- 0.5)          with the add rounded TOWARD ZERO: doubles >= 2^52 are integers
//                                   and keep their value, smaller ones get round-half-away exactly.
// The reference's saturating-cast corner (x = -+2^63 mod 2^64) is kept.
// f64_to_torus(sc * xs) with the scale absorbed into the first two operations as FMAs
// CORNER = false leaves the saturating-cast corner to the caller: *mag_max accumulates the largest
// |lo| exponent word seen, and a caller that finds kTorusCornerMag in it afterwards redoes its
// values with f64_to_torus_s (one test per 32 conversions instead of ~8 predicated instructions each).
constexpr uint32_t kTorusCornerMag = 0x43E00000u;  // high word of 2^63
template <bool SCALED, bool CORNER>
SPF_HD uint64_t f64_to_torus_impl(double xs, double sc, uint32_t* mag_max) {
  const double magic = 124615124604835863084731911901282304.0;  // 1.5 * 2^116
  const double hq = (SCALED ? spf_fma(sc, xs, magic) : xs + magic) - magic;
  const double lo = SCALED ? spf_fma(sc, xs, -hq) : xs - hq;
  const uint32_t hi = (uint32_t)(f64_bits(lo) >> 32);
  const double half = bits_f64((uint64_t)((hi & 0x80000000u) | 0x3FE00000u) << 32);  // copysign(0.5, lo)
#if defined(__CUDA_ARCH__)
  uint64_t r = (uint64_t)__double2ll_rz(__dadd_rz(lo, half));
#else
  const long double y = (long double)lo + (long double)half;  // exact in the 64-bit x87 significand
  uint64_t r;
  if (y != y) r = 0;
  else if (y >= 9223372036854775808.0L) r = (uint64_t)INT64_MAX;
  else if (y < -9223372036854775808.0L) r = (uint64_t)INT64_MIN;
  else r = (uint64_t)(int64_t)y;
#endif
  // |lo| <= 2^63 by construction, so exponent 0x43E means |lo| == 2^63 exactly: the reference's
  // result then follows the sign of x.  Probability ~2^-53 per coefficient.
  const uint32_t mag = hi & 0x7FFFFFFFu;
  if (CORNER) {
    if (__builtin_expect(mag == kTorusCornerMag, 0))
      r = ((f64_bits(xs) ^ (SCALED ? f64_bits(sc) : 0ull)) >> 63) ? 0x7FFFFFFFFFFFFFFFull : 0x8000000000000000ull;  // sign of sc * xs
  } else {
    *mag_max = mag > *mag_max ? mag : *mag_max;
  }
  return r;
}
SPF_HD uint64_t f64_to_torus(double x) { return f64_to_torus_impl<false, true>(x, 1.0, nullptr); }
SPF_HD uint64_t f64_to_torus_s(double xs, double sc) { return f64_to_torus_impl<true, true>(xs, sc, nullptr); }
SPF_HD uint64_t f64_to_torus_s_fast(double xs, double sc, uint32_t& mag_max) {
  return f64_to_torus_impl<true, false>(xs, sc, &mag_max);
}

// ------------------------------------------------------------------------------------------
// radix decomposition (math/radix.rs:67-114,155-162; simd/scalar.rs:52-72)
// ------------------------------------------------------------------------------------------
SPF_HD uint64_t radix_round(uint64_t x, int radix_log, int count) {
  const int shift = 64 - radix_log * count;
  return (x >> shift) + ((x >> (shift - 1)) & 1);
}
// Balanced digits without a carry chain: with r = radix_round(x) and r' = r + sum_t (B/2) B^t, the
// bit field t of r' is the UNSIGNED digit u_t = d_t + B/2 of the balanced representation
// (sum d_t B^t = r mod B^count, d_t in [-B/2, B/2)), which is unique -- so d_t = u_t - B/2 equals what
// PolynomialRadixIterator (math/radix.rs:81-113) emits LSB first with its carry.
SPF_HD uint64_t radix_offset(int radix_log, int count) {
  uint64_t o = 0;
  for (int t = 0; t < count; t++) o += (1ull << (radix_log - 1)) << (t * radix_log);
  return o;
}
// one vector_next_decomp step on a scalar; returns the signed digit
SPF_HD int32_t next_digit(uint64_t& s, int radix_log) {
  const uint64_t mask = (1ull << radix_log) - 1;
  uint64_t digit = s & mask;
  s >>= radix_log;
  const uint64_t carry = digit >> (radix_log - 1);
  s += carry;
  return (int32_t)((int64_t)digit - (int64_t)(carry << radix_log));
}

// (p * X^rot)[j] for 0 <= rot < 2N: entities/polynomial.rs:211-236 as a gather.
SPF_HD uint64_t rotated_coeff(const uint64_t* p, int j, int rot) {
  int idx = j - rot;          // in (-2N, N)
  bool neg = false;
  if (idx < 0) { idx += kN; neg = true; }
  if (idx < 0) { idx += kN; neg = false; }
  const uint64_t v = p[idx];
  return neg ? 0 - v : v;
}

}  // namespace spf
