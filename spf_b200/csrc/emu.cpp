// emu.cpp -- HOST EMULATOR of the device kernel bodies (team_ops.cuh / fft16.cuh).
// Test infrastructure: runs the exact __host__ __device__ code of the CUDA kernels with one
// host thread per virtual GPU thread (64 per team) and a pthread barrier in place of bar.sync,
// so the FFT factorisation, the register-slot <-> bin mapping and every index computation are checked against
// the oracle on machines without a GPU.  Built by g++ into libspf_emu.so; never shipped on the
// product path and never used as a fallback.
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#include <cmath>
#include <vector>

#include "tables.h"
#include "team_ops.cuh"

using namespace spf;

namespace {

struct HostCx {
  static constexpr bool kTmemTwiddles = false;
  int u;
  pthread_barrier_t* bar;
  void sync() { pthread_barrier_wait(bar); }
  uint64_t rp_stash[32];  // device: the thread's tensor-memory columns
  void rp_store(const uint64_t (&rp)[32]) { memcpy(rp_stash, rp, sizeof(rp_stash)); }
  void rp_load(uint64_t (&rp)[32]) { memcpy(rp, rp_stash, sizeof(rp_stash)); }
};

// pair of teams (pbs_pair_team): 128 host threads, one barrier per half and one for the pair
struct HostPairCx {
  int u, h;
  pthread_barrier_t* bar_half;
  pthread_barrier_t* bar_pair;
  void sync() { pthread_barrier_wait(bar_half); }
  void pair_sync() { pthread_barrier_wait(bar_pair); }
  // the device keeps the thread's 16 pass-1 twiddles in tensor memory; here they come from the table
  template <bool CONJ>
  void t1_mul(C2 (&v)[16], const C2* T1) {
    for (int k1 = 0; k1 < 16; k1++) v[k1] = CONJ ? cmul_conj(v[k1], T1[k1 * 64 + u]) : cmul(v[k1], T1[k1 * 64 + u]);
  }
  // reader-side pass-2 twiddles (device: the thread's constants sit in tensor memory; here they are recomputed, same arithmetic)
  void rt2_fwd(double (&tw)[12], const C2* T2) { rt2_fwd_consts(T2, u >> 4, h, tw); }
  void rt2_inv(C2 (&w)[6], const C2* T2) { rt2_inv_consts(T2, u >> 4, h, w); }
  // the BSK ring is device machinery: the host reads the key in place
  const C2* bsk_acquire(int, const C2* g) { return g; }
  void bsk_release(int) {}
  void bsk_skip(int) {}
  C2 bsk_load(const C2* p) { return *p; }
  // the device keeps a private copy of the thread's own accumulator coefficients in tensor memory
  uint64_t own_stash[32];
  void own_store(const uint64_t (&own)[32]) { memcpy(own_stash, own, sizeof(own_stash)); }
  void own_ld8(uint64_t (&o)[8], int c) { memcpy(o, own_stash + 8 * c, 64); }
  void own_ld4x2(uint64_t (&o)[8], int m4) { memcpy(o, own_stash + m4, 32); memcpy(o + 4, own_stash + m4 + 16, 32); }
  void own_st4x2(const uint64_t (&o)[8], int m4) { memcpy(own_stash + m4, o, 32); memcpy(own_stash + m4 + 16, o + 4, 32); }
  void own_st_wait() {}
  void f_store(const C2 (&)[2][8]) {}  // device: accumulators parked in tensor memory between digit levels
  void f_load(C2 (&)[2][8]) {}
};

template <class Cx, class Body>
struct PairLaunch {
  Body* body;
  Cx cx;
  static void* run(void* p) {
    PairLaunch* l = (PairLaunch*)p;
    (*l->body)(l->cx);
    return nullptr;
  }
};

template <class Cx, class Body>
void run_pair(Body body) {
  pthread_barrier_t half[2], pair;
  pthread_barrier_init(&half[0], nullptr, kTeam);
  pthread_barrier_init(&half[1], nullptr, kTeam);
  pthread_barrier_init(&pair, nullptr, 2 * kTeam);
  std::vector<PairLaunch<Cx, Body>> ls(2 * kTeam);
  std::vector<pthread_t> th(2 * kTeam);
  for (int t = 0; t < 2 * kTeam; t++) {
    ls[t].body = &body;
    ls[t].cx.u = t % kTeam;
    ls[t].cx.h = t / kTeam;
    ls[t].cx.bar_half = &half[t / kTeam];
    ls[t].cx.bar_pair = &pair;
    pthread_create(&th[t], nullptr, PairLaunch<Cx, Body>::run, &ls[t]);
  }
  for (int t = 0; t < 2 * kTeam; t++) pthread_join(th[t], nullptr);
  pthread_barrier_destroy(&half[0]);
  pthread_barrier_destroy(&half[1]);
  pthread_barrier_destroy(&pair);
}

template <class Body>
struct Launch {
  Body* body;
  HostCx cx;
  static void* run(void* p) {
    Launch* l = (Launch*)p;
    (*l->body)(l->cx);
    return nullptr;
  }
};

template <class Body>
void run_team(Body body) {
  pthread_barrier_t bar;
  pthread_barrier_init(&bar, nullptr, kTeam);
  std::vector<Launch<Body>> ls(kTeam);
  std::vector<pthread_t> th(kTeam);
  for (int u = 0; u < kTeam; u++) {
    ls[u].body = &body;
    ls[u].cx = HostCx{u, &bar, {}};
    pthread_create(&th[u], nullptr, Launch<Body>::run, &ls[u]);
  }
  for (int u = 0; u < kTeam; u++) pthread_join(th[u], nullptr);
  pthread_barrier_destroy(&bar);
}

// 8 teams of one CTA (cmux_wide): one barrier per team and one for all 512 threads
struct HostWideCx {
  int u, team;
  pthread_barrier_t* bar_team;
  pthread_barrier_t* bar_cta;
  void sync() { pthread_barrier_wait(bar_team); }
  void cta_sync() { pthread_barrier_wait(bar_cta); }
};
template <class Body>
struct WideLaunch {
  Body* body;
  HostWideCx cx;
  static void* run(void* p) {
    WideLaunch* l = (WideLaunch*)p;
    (*l->body)(l->cx);
    return nullptr;
  }
};
template <class Body>
void run_wide(Body body) {
  const int nt = kWideTeams * kTeam;
  pthread_barrier_t team[kWideTeams], cta;
  for (int i = 0; i < kWideTeams; i++) pthread_barrier_init(&team[i], nullptr, kTeam);
  pthread_barrier_init(&cta, nullptr, nt);
  std::vector<WideLaunch<Body>> ls(nt);
  std::vector<pthread_t> th(nt);
  for (int t = 0; t < nt; t++) {
    ls[t].body = &body;
    ls[t].cx = HostWideCx{t % kTeam, t / kTeam, &team[t / kTeam], &cta};
    pthread_create(&th[t], nullptr, WideLaunch<Body>::run, &ls[t]);
  }
  for (int t = 0; t < nt; t++) pthread_join(th[t], nullptr);
  for (int i = 0; i < kWideTeams; i++) pthread_barrier_destroy(&team[i]);
  pthread_barrier_destroy(&cta);
}

// four teams of one ciphertext (pbs_quad_team)
struct HostQuadCx {
  int u, h, t;
  pthread_barrier_t* bar_team;
  pthread_barrier_t* bar_quad;
  // split gather: the two teams of a polynomial swap 16 packed digits per thread (device: through tensor memory)
  pthread_barrier_t* bar_poly = nullptr;  // the 128 threads of teams (h, 0) and (h, 1)
  uint32_t* xchg = nullptr;               // [h][t][u][8]
  void digit_xchg(uint32_t (&pk)[8]) {
    memcpy(xchg + ((size_t)(h * 2 + t) * kTeam + u) * 8, pk, sizeof(pk));
    pthread_barrier_wait(bar_poly);
    memcpy(pk, xchg + ((size_t)(h * 2 + (1 - t)) * kTeam + u) * 8, sizeof(pk));
  }
  void rt2(double (&tw)[6], C2 (&wi)[3], const C2* T2) { rt2_group_consts(T2, u >> 4, 2 * h + t, tw, wi); }
  void sync() { pthread_barrier_wait(bar_team); }
  void quad_sync() { pthread_barrier_wait(bar_quad); }
  // the device stages the next BSK row in shared memory with a bulk copy; the host reads the key directly
  void row_prefetch(const C2*) {}
  const C2* row_wait(int, const C2* row) { return row; }
  C2 row_load(const C2* p) { return *p; }
  template <bool CONJ>
  void t1_mul(C2 (&v)[16], const C2* T1) {
    for (int k1 = 0; k1 < 16; k1++) v[k1] = CONJ ? cmul_conj(v[k1], T1[k1 * 64 + u]) : cmul(v[k1], T1[k1 * 64 + u]);
  }
};
template <class Body>
struct QuadLaunch {
  Body* body;
  HostQuadCx cx;
  static void* run(void* p) {
    QuadLaunch* l = (QuadLaunch*)p;
    (*l->body)(l->cx);
    return nullptr;
  }
};
template <class Body>
void run_quad(Body body) {
  const int nt = 4 * kTeam;
  pthread_barrier_t team[4], quad, poly[2];
  for (int i = 0; i < 4; i++) pthread_barrier_init(&team[i], nullptr, kTeam);
  for (int i = 0; i < 2; i++) pthread_barrier_init(&poly[i], nullptr, 2 * kTeam);
  pthread_barrier_init(&quad, nullptr, nt);
  std::vector<uint32_t> xchg(4 * kTeam * 8);
  std::vector<QuadLaunch<Body>> ls(nt);
  std::vector<pthread_t> th(nt);
  for (int t = 0; t < nt; t++) {
    const int tm = t / kTeam;
    ls[t].body = &body;
    ls[t].cx = HostQuadCx{t % kTeam, tm >> 1, tm & 1, &team[tm], &quad, &poly[tm >> 1], xchg.data()};
    pthread_create(&th[t], nullptr, QuadLaunch<Body>::run, &ls[t]);
  }
  for (int t = 0; t < nt; t++) pthread_join(th[t], nullptr);
  for (int i = 0; i < 4; i++) pthread_barrier_destroy(&team[i]);
  for (int i = 0; i < 2; i++) pthread_barrier_destroy(&poly[i]);
  pthread_barrier_destroy(&quad);
}

struct Tables {
  std::vector<C2> T1, T2;
  Tables() : T1(kT1Elems), T2(kT2Elems) { fill_twiddle_tables(T1.data(), T2.data()); }
};
const Tables& tables() {
  static Tables t;
  return t;
}

}  // namespace

extern "C" {

// reference-scale FFT-domain polys -> device scale (2^-10)
void emu_import_fft(const C2* src, C2* dst, size_t npoly) {
  for (size_t q = 0; q < npoly; q++) import_fft_poly(src + q * kM, dst + q * kM);
}
void emu_export_fft(const C2* src, C2* dst, size_t npoly) {
  for (size_t q = 0; q < npoly; q++) export_fft_poly(src + q * kM, dst + q * kM);
}

// PolynomialRef::fft in the reference's (natural order, unscaled) convention, via the team code.
void emu_poly_fft(const uint64_t* poly, C2* out_natural) {
  const Tables& t = tables();
  std::vector<C2> xbuf(kXBuf), dev(kM);
  run_team([&](HostCx& cx) {
    C2 v[16];
    team_poly_fft(cx, v, [&](int j) { return poly[j]; }, xbuf.data(), t.T1.data(), t.T2.data());
    for (int s = 0; s < 16; s++) dev[bin_of(cx.u, s)] = v[s];
  });
  export_fft_poly(dev.data(), out_natural);
}

// PolynomialFftRef::ifft (natural order, unscaled input) via the team code.
void emu_poly_ifft(const C2* in_natural, uint64_t* poly) {
  const Tables& t = tables();
  std::vector<C2> xbuf(kXBuf), dev(kM);
  import_fft_poly(in_natural, dev.data());
  run_team([&](HostCx& cx) {
    C2 v[16];
    for (int s = 0; s < 16; s++) v[s] = dev[bin_of(cx.u, s)];
    team_fft_inv(cx, v, xbuf.data(), t.T1.data(), t.T2.data());
    for (int m = 0; m < 16; m++) {
      poly[cx.u + 64 * m] = f64_to_torus(v[m].x);
      poly[cx.u + 64 * m + kM] = f64_to_torus(v[m].y);
    }
  });
}

uint64_t emu_f64_to_torus(double x) { return f64_to_torus(x); }
double emu_i32_to_f64(int32_t x) { return i32_to_f64(x); }

// cmux with the GGSW in device scale (2^-10); d0 may be null (external product)
void emu_cmux(uint64_t* out, const uint64_t* d0, const uint64_t* d1, const C2* ggsw_dev, int radix_log,
              int count) {
  const Tables& t = tables();
  std::vector<C2> xbuf(kXBuf);
  std::vector<uint64_t> st(32 * 64);
  run_team([&](HostCx& cx) {
    cmux_team(cx, out, d0, d1, ggsw_dev, st.data(), xbuf.data(), t.T1.data(), t.T2.data(), radix_log, count);
  });
}

// the latency-oriented 8-team version of the same op (count must be 4)
void emu_cmux_wide(uint64_t* out, const uint64_t* d0, const uint64_t* d1, const C2* ggsw_dev, int radix_log,
                   int count) {
  const Tables& t = tables();
  std::vector<C2> xbuf(kWideTeams * kXBuf);
  run_wide([&](HostWideCx& cx) {
    cmux_wide(cx, out, d0, d1, ggsw_dev, xbuf.data(), t.T1.data(), t.T2.data(), radix_log, count);
  });
}

// generalized PBS on the pair-team code the device runs; bsk in device scale (2^-10).  lut may be null (CBS mode).
void emu_pbs(uint64_t* glwe_out, const uint64_t* lwe_in, const uint64_t* lut, const C2* bsk_dev, int lwe_n,
             int log_chi, int log_v, int cbs_radix_log, int cbs_count) {
  const Tables& t = tables();
  std::vector<C2> xbuf(2 * kXBuf);
  PbsArgs A{lwe_in, lut, glwe_out, bsk_dev, lwe_n, log_chi, log_v, cbs_radix_log, cbs_count};
  run_pair<HostPairCx>([&](HostPairCx& cx) {
    int G = 0;
    pbs_pair_team(cx, A, xbuf.data(), t.T1.data(), t.T2.data(), G);
  });
}
// Part of the library's interface that tests/emu_util.py binds.  The transient and chunked forms it used to select all
// gave emu_pbs's output bit for bit; they are now the one form the device ships, so every flag pair runs emu_pbs.
void emu_pbs_variant(uint64_t* glwe_out, const uint64_t* lwe_in, const uint64_t* lut, const C2* bsk_dev, int lwe_n,
                     int log_chi, int log_v, int cbs_radix_log, int cbs_count, int /*transient*/, int /*chunked*/) {
  emu_pbs(glwe_out, lwe_in, lut, bsk_dev, lwe_n, log_chi, log_v, cbs_radix_log, cbs_count);
}

// the latency-mode (four-team) blind rotation
void emu_pbs_quad(uint64_t* glwe_out, const uint64_t* lwe_in, const uint64_t* lut, const C2* bsk_dev, int lwe_n,
                  int log_chi, int log_v, int cbs_radix_log, int cbs_count) {
  const Tables& t = tables();
  std::vector<C2> xbuf(4 * kXBuf);
  std::vector<uint64_t> acc(2 * kN);
  PbsArgs A{lwe_in, lut, glwe_out, bsk_dev, lwe_n, log_chi, log_v, cbs_radix_log, cbs_count};
  run_quad([&](HostQuadCx& cx) {
    int executed = 0;
    pbs_quad_team(cx, A, acc.data(), xbuf.data(), t.T1.data(), t.T2.data(), executed);
  });
}

// trace / CBS tail for one level.  mode: 0 CBS pre-process + trace (+SS), 1 plain trace, 2 SS only.
void emu_trace_ss(const uint64_t* glwe_in, uint64_t* glev_out, C2* ggsw_out_dev, const C2* ak_dev,
                  const C2* ssk_dev, int level, int mode, int cbs_radix_log, int cbs_count, int tr_radix_log,
                  int tr_count, int ss_radix_log, int ss_count) {
  const Tables& t = tables();
  std::vector<C2> xbuf(kXBuf);
  std::vector<uint64_t> g(2 * kN);
  uint32_t kinv[11];
  fill_kinv(kinv);
  TraceSsArgs A{glwe_in, glev_out, ggsw_out_dev, ak_dev, ssk_dev, kinv, level, mode, cbs_radix_log,
                cbs_count, tr_radix_log, tr_count, ss_radix_log, ss_count, 1.0};
  run_team([&](HostCx& cx) { trace_ss_team(cx, A, g.data(), xbuf.data(), t.T1.data(), t.T2.data()); });
}

}  // extern "C"
