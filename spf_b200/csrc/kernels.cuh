// kernels.cuh -- sm_100a __global__ kernels for the circuit-bootstrapping hot path.
// The per-team bodies live in team_ops.cuh (shared with the host emulator); this file adds the
// CTA organisation: shared-memory carve-up, named barriers, grid mapping.
#pragma once
#include <cuda_runtime.h>

#include "team_ops.cuh"

namespace spf {

// One team = 2 warps.  Team-private named barrier ids 1..15 (0 is __syncthreads).
__device__ __forceinline__ void tmem_ld16(uint32_t (&r)[16], uint32_t taddr);
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]);
__device__ __forceinline__ void tmem_wait_ld();
__device__ __forceinline__ void tmem_wait_st();

struct DevCx {
  static constexpr bool kTmemTwiddles = false;
  int u;
  int bar;
  uint32_t rp_taddr;  // 64 private tensor-memory columns of this warp (trace / scheme-switch kernel only)
  __device__ __forceinline__ void sync() const {
    asm volatile("bar.sync %0, 64;" ::"r"(bar) : "memory");
  }
  __device__ __forceinline__ void rp_store(const uint64_t (&rp)[32]) const {
#pragma unroll
    for (int c = 0; c < 4; c++) {
      uint32_t r[16];
#pragma unroll
      for (int i = 0; i < 8; i++) { r[2 * i] = (uint32_t)rp[8 * c + i]; r[2 * i + 1] = (uint32_t)(rp[8 * c + i] >> 32); }
      tmem_st16(rp_taddr + 16 * c, r);
    }
    tmem_wait_st();
  }
  __device__ __forceinline__ void rp_load(uint64_t (&rp)[32]) const {
    uint32_t r[4][16];
#pragma unroll
    for (int c = 0; c < 4; c++) tmem_ld16(r[c], rp_taddr + 16 * c);
    tmem_wait_ld();
#pragma unroll
    for (int c = 0; c < 4; c++)
#pragma unroll
      for (int i = 0; i < 8; i++) rp[8 * c + i] = ((uint64_t)r[c][2 * i + 1] << 32) | r[c][2 * i];
  }
};

struct DevTables {
  const C2* T1;  // global copies of the twiddle tables
  const C2* T2;
};

__device__ __forceinline__ void load_tables(C2* sT1, C2* sT2, const DevTables& t) {
  for (int i = threadIdx.x; i < kT1Elems; i += blockDim.x) sT1[i] = t.T1[i];
  for (int i = threadIdx.x; i < kT2Elems; i += blockDim.x) sT2[i] = t.T2[i];
  __syncthreads();
}

constexpr int kTableBytes = (kT1Elems + kT2Elems) * 16;  // 17472

// Programmatic dependent launch (griddepcontrol): a kernel launched with the programmatic-stream-
// serialization attribute may start while its predecessor in the stream is still running; everything
// before pdl_wait() must therefore touch only data no earlier kernel of the stream writes (twiddle
// tables, the pointer tables uploaded at graph build) -- pdl_wait() returns once the predecessor has
// completed and its writes are visible.  pdl_launch_dependents() lets the successor's CTAs be
// scheduled as soon as every CTA of this grid has passed it.  Both are no-ops for ordinary launches.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ------------------------------------------------------------------------------------------
// K3: batched programmable bootstrap (blind rotation), throughput mode.  3 ciphertexts per CTA,
// each owned by a PAIR of teams (128 threads, see pbs_pair_team), one persistent CTA per SM:
// 12 warps, <= 168 registers.  Resident pairs walk the 637 BSK rows roughly in step, so a row is
// fetched from HBM once per sweep and then served from L2 to all CTAs.  The per-thread constants
// and parked values of a pair live in TENSOR MEMORY (tcgen05.ld/st); DESIGN.md section 7 lists the
// alternatives that were measured and what each was worth.
// ------------------------------------------------------------------------------------------
constexpr int kPbsPairs = 3;
// Per pair: the two exchange buffers (one per half).  The accumulator image lives in the half's exchange buffer
// (pbs_pair_team), so a pair needs no persistent accumulator in shared memory: the BSK ring lives in what that frees.
constexpr int kPbsPairBytes = 2 * kXBuf * 16;
// tensor-memory columns: [0,64) T1 | own coefficients 64 per pair | parked accumulators 64 per pair while they fit
// in the 512 columns | [448,512) reader-side pass-2 twiddles; pairs beyond that park their accumulators in shared memory
constexpr int kPbsTmemOwn0 = 64;
constexpr int kPbsTmemF0 = kPbsTmemOwn0 + 64 * kPbsPairs;
constexpr int kPbsTmemFPairs = (512 - kPbsTmemF0) / 64 < kPbsPairs ? (512 - kPbsTmemF0) / 64 : kPbsPairs;
constexpr int kPbsFParkBytes = (kPbsPairs - kPbsTmemFPairs) * 2 * kTeam * 16 * 16;  // 32 KiB per pair parked in smem
// The bootstrapping key is staged through a shared-memory ring by bulk copies, one copy per chunk and CTA.
constexpr int kRingStages = 3;
constexpr int kRingChunkElems = 2 * kM;                  // one (row, level) GLEV row of the BSK: [p][bin]
constexpr int kRingChunkBytes = kRingChunkElems * 16;    // 32768
constexpr int kPbsPairOff = kTableBytes;
constexpr int kPbsRingOff = kPbsPairOff + kPbsPairs * kPbsPairBytes + kPbsFParkBytes;
constexpr int kPbsRingBytes = kRingStages * kRingChunkBytes + 64;  // + full barriers, release counters
constexpr int kPbsSmem = kPbsRingOff + kPbsRingBytes;
static_assert(kPbsSmem <= 232448, "pbs_kernel shared memory");

// tensor-memory helpers (32x32b shape: thread i of a warp <-> TMEM lane 32*(warp%4)+i, one
// 32-bit word per column)
__device__ __forceinline__ void tmem_ld16(uint32_t (&r)[16], uint32_t taddr) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}
__device__ __forceinline__ void tmem_st2(uint32_t taddr, uint32_t a, uint32_t b) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

constexpr int kPbsTmemCols = 512;
__device__ __forceinline__ void tmem_ld8(uint32_t (&r)[8], uint32_t taddr) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// mbarrier wait that turns a lost wake-up into a trapped kernel instead of a hung GPU
__device__ __forceinline__ void mbar_wait_trap(uint32_t bar, uint32_t parity) {
  unsigned long long t_start = 0;
  for (int spin = 0;; spin++) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) return;
    if ((spin & 1023) == 1023) {  // a chunk that has not landed after 2 s will never land
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t_start == 0) t_start = now;
      else if (now - t_start > 2000000000ull) __trap();
    }
  }
}
struct DevPairCx {
  // ---- reader-side pass-2 twiddles: 12 + 12 doubles of this thread in the columns [448, 496) (pair_tmem_init) ----
  __device__ __forceinline__ void rt2_fwd(double (&tw)[12], const C2*) const {
    uint32_t a[16], b[8];
    tmem_ld16(a, t1_taddr + 448);
    tmem_ld8(b, t1_taddr + 448 + 16);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 8; i++) tw[i] = __hiloint2double((int)a[2 * i + 1], (int)a[2 * i]);
#pragma unroll
    for (int i = 0; i < 4; i++) tw[8 + i] = __hiloint2double((int)b[2 * i + 1], (int)b[2 * i]);
  }
  __device__ __forceinline__ void rt2_inv(C2 (&w)[6], const C2*) const {
    uint32_t a[16], b[8];
    tmem_ld16(a, t1_taddr + 448 + 24);
    tmem_ld8(b, t1_taddr + 448 + 24 + 16);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 4; i++) w[i] = C2{__hiloint2double((int)a[4 * i + 1], (int)a[4 * i]), __hiloint2double((int)a[4 * i + 3], (int)a[4 * i + 2])};
#pragma unroll
    for (int i = 0; i < 2; i++) w[4 + i] = C2{__hiloint2double((int)b[4 * i + 1], (int)b[4 * i]), __hiloint2double((int)b[4 * i + 3], (int)b[4 * i + 2])};
  }
  int u, h;
  int bar_half, bar_pair;
  uint32_t t1_taddr;   // this warp's lane quarter, column 0 of the T1 block
  uint32_t own_taddr;  // this warp's private 64 columns (own coefficients)
  uint32_t f_taddr;    // this warp's 64 columns for the parked accumulators (unused when fpark != nullptr)
  C2* fpark;           // shared-memory parking [16][128] of a pair whose accumulators do not fit in tensor memory
  // ---- BSK ring (protocol in team_ops.cuh above pbs_pair_team) ----
  uint32_t ring_s = 0, full_s = 0;  // shared addresses of stage 0 / of full[0]
  unsigned* rel = nullptr;          // per-stage count of pairs that are done with the resident chunk
  const C2* bsk = nullptr;
  int lwe_n = 0, npairs = 0, total = 0;  // total: chunks this CTA consumes over the whole launch
  bool elected = false;             // one thread per pair counts the pair off
  // chunk G = 4 i + k: k = 2 t + row with digit level t <-> GLEV level 1 - t
  __device__ __forceinline__ void ring_issue(int Gn) const {
    const int i = (Gn >> 2) % lwe_n, k = Gn & 3, c = (k & 1) * 2 + (1 - (k >> 1)), st = Gn % kRingStages;
    const C2* src = bsk + ((size_t)i * 4 + c) * kRingChunkElems;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // in front of every refill of a ring stage
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full_s + 8 * st), "r"((uint32_t)kRingChunkBytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(ring_s + st * kRingChunkBytes), "l"(src), "r"((uint32_t)kRingChunkBytes), "r"(full_s + 8 * st) : "memory");
  }
  // returns the chunk's address: a shared-window address in a pointer's clothes (bsk_load)
  __device__ __forceinline__ const C2* bsk_acquire(int G, const C2*) const {
    const int st = G % kRingStages;
    mbar_wait_trap(full_s + 8 * st, (uint32_t)(G / kRingStages) & 1u);
    return reinterpret_cast<const C2*>((size_t)(ring_s + st * kRingChunkBytes));
  }
  __device__ __forceinline__ C2 bsk_load(const C2* p) const {
    C2 r;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "r"((uint32_t)(size_t)p) : "memory");
    return r;
  }
  __device__ __forceinline__ void bsk_release(int G) const {
    if (elected) {
      const int st = G % kRingStages;
      __threadfence_block();
      if (atomicAdd(rel + st, 1u) == (unsigned)npairs - 1u) {  // last pair out re-arms the stage
        atomicExch(rel + st, 0u);
        __threadfence_block();
        if (G + kRingStages < total) ring_issue(G + kRingStages);
      }
    }
  }
  __device__ __forceinline__ void bsk_skip(int G) const {  // a step whose rotation is the identity: count off unread chunks
    if (elected) {
#pragma unroll 1
      for (int k = 0; k < 4; k++) {
        mbar_wait_trap(full_s + 8 * ((G + k) % kRingStages), (uint32_t)((G + k) / kRingStages) & 1u);  // the copy has landed
        bsk_release(G + k);
      }
    }
  }
  __device__ __forceinline__ void sync() const { asm volatile("bar.sync %0, 64;" ::"r"(bar_half) : "memory"); }
  __device__ __forceinline__ void pair_sync() const { asm volatile("bar.sync %0, 128;" ::"r"(bar_pair) : "memory"); }
  // v[k1] *= T1[k1][u] (or its conjugate).  The 16 twiddles of a thread never change, so they sit
  // in the thread's tensor-memory columns instead of a shared-memory table: 16 LDS.128 per
  // transform (12 % of the kernel's shared-memory wavefronts) become 4 tcgen05.ld on a path the
  // LSU pipe does not see.  Four twiddles (16 registers) at a time: shorter live ranges, a better schedule.
  template <bool CONJ>
  __device__ __forceinline__ void t1_mul(C2 (&v)[16], const C2*) const {
#pragma unroll
    for (int g = 0; g < 4; g++) {
      uint32_t r[16];
      tmem_ld16(r, t1_taddr + 16 * g);
      tmem_wait_ld();
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const C2 w{__hiloint2double((int)r[4 * i + 1], (int)r[4 * i]), __hiloint2double((int)r[4 * i + 3], (int)r[4 * i + 2])};
        const int k = 4 * g + i;
        v[k] = CONJ ? cmul_conj(v[k], w) : cmul(v[k], w);
      }
    }
  }
  // accumulators parked in tensor memory while the second digit level is transformed
  __device__ __forceinline__ void f_store(const C2 (&f)[2][8]) const {
    if (fpark) {
#pragma unroll
      for (int c = 0; c < 16; c++) fpark[c * 2 * kTeam + h * kTeam + u] = f[c >> 3][c & 7];
      return;
    }
    // one double per store: a 16-register store makes ptxas gather the 64 words into consecutive registers first (64 moves)
#pragma unroll
    for (int c = 0; c < 16; c++) {
      const C2 x = f[c >> 3][c & 7];
      tmem_st2(f_taddr + 4 * c, (uint32_t)__double2loint(x.x), (uint32_t)__double2hiint(x.x));
      tmem_st2(f_taddr + 4 * c + 2, (uint32_t)__double2loint(x.y), (uint32_t)__double2hiint(x.y));
    }
    tmem_wait_st();
  }
  __device__ __forceinline__ void f_load(C2 (&f)[2][8]) const {
    if (fpark) {
#pragma unroll
      for (int c = 0; c < 16; c++) f[c >> 3][c & 7] = fpark[c * 2 * kTeam + h * kTeam + u];
      return;
    }
    uint32_t r[4][16];
#pragma unroll
    for (int c = 0; c < 4; c++) tmem_ld16(r[c], f_taddr + 16 * c);
    tmem_wait_ld();
#pragma unroll
    for (int c = 0; c < 4; c++) {
#pragma unroll
      for (int i = 0; i < 4; i++)
        f[c >> 1][4 * (c & 1) + i] = C2{__hiloint2double((int)r[c][4 * i + 1], (int)r[c][4 * i]),
                                        __hiloint2double((int)r[c][4 * i + 3], (int)r[c][4 * i + 2])};
    }
  }
  // the thread's own accumulator coefficients: a private copy in tensor memory, fetched 8 (gather) or 4 + 4 (update) at a time
  __device__ __forceinline__ void own_ld8(uint64_t (&o)[8], int c) const {
    uint32_t r[16];
    tmem_ld16(r, own_taddr + 16 * c);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 8; i++) o[i] = ((uint64_t)r[2 * i + 1] << 32) | r[2 * i];
  }
  __device__ __forceinline__ void own_ld4x2(uint64_t (&o)[8], int m4) const {
    uint32_t a[8], b[8];
    tmem_ld8(a, own_taddr + 2 * m4);
    tmem_ld8(b, own_taddr + 2 * (m4 + 16));
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 4; i++) {
      o[i] = ((uint64_t)a[2 * i + 1] << 32) | a[2 * i];
      o[4 + i] = ((uint64_t)b[2 * i + 1] << 32) | b[2 * i];
    }
  }
  __device__ __forceinline__ void own_st4x2(const uint64_t (&o)[8], int m4) const {
    uint32_t a[8], b[8];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      a[2 * i] = (uint32_t)o[i]; a[2 * i + 1] = (uint32_t)(o[i] >> 32);
      b[2 * i] = (uint32_t)o[4 + i]; b[2 * i + 1] = (uint32_t)(o[4 + i] >> 32);
    }
    tmem_st8(own_taddr + 2 * m4, a);
    tmem_st8(own_taddr + 2 * (m4 + 16), b);
  }
  __device__ __forceinline__ void own_st_wait() const { tmem_wait_st(); }
  __device__ __forceinline__ void own_store(const uint64_t (&own)[32]) const {
#pragma unroll
    for (int c = 0; c < 4; c++) {
      uint32_t r[16];
#pragma unroll
      for (int i = 0; i < 8; i++) { r[2 * i] = (uint32_t)own[8 * c + i]; r[2 * i + 1] = (uint32_t)(own[8 * c + i] >> 32); }
      tmem_st16(own_taddr + 16 * c, r);
    }
    tmem_wait_st();
  }
};

// Tensor-memory scratchpad of the pair / quad team kernels: one 512-column allocation per CTA.
// Columns [0,64) pass-1 twiddles of the thread (shared by the warps of a lane quarter, which have the same
// thread-in-team index), then the per-pair blocks of pbs_kernel (kPbsTmemOwn0, kPbsTmemF0); [448,512) pass-2
// twiddles.  Returns this warp's lane-quarter base address.
__device__ __forceinline__ uint32_t pair_tmem_init(const C2* sT1, const C2* sT2, uint32_t& alloc_base, bool reader_t2 = false) {
  __shared__ uint32_t tmem_base;
  const int warp = threadIdx.x >> 5;
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     (uint32_t)__cvta_generic_to_shared(&tmem_base)), "n"(kPbsTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  alloc_base = tmem_base;
  const uint32_t t1_taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
  if (warp < 4) {  // every lane quarter is shared by warps w, w+4, w+8, which have the same u
    const int uu = (warp & 1) * 32 + (threadIdx.x & 31);
#pragma unroll
    for (int k1 = 0; k1 < 16; k1++) {
      const C2 w = sT1[k1 * 64 + uu];
      tmem_st4(t1_taddr + 4 * k1, (uint32_t)__double2loint(w.x), (uint32_t)__double2hiint(w.x),
               (uint32_t)__double2loint(w.y), (uint32_t)__double2hiint(w.y));
    }
    if (reader_t2) {
      // pbs_kernel: the thread's reader-side pass-2 constants (warps 0..3 of a pair: half h = warp >> 1) instead of the table row
      double tw[12];
      C2 wi[6];
      rt2_fwd_consts(sT2, uu >> 4, (warp >> 1) & 1, tw);
      rt2_inv_consts(sT2, uu >> 4, (warp >> 1) & 1, wi);
#pragma unroll
      for (int i = 0; i < 6; i++)
        tmem_st4(t1_taddr + 448 + 4 * i, (uint32_t)__double2loint(tw[2 * i]), (uint32_t)__double2hiint(tw[2 * i]),
                 (uint32_t)__double2loint(tw[2 * i + 1]), (uint32_t)__double2hiint(tw[2 * i + 1]));
#pragma unroll
      for (int i = 0; i < 6; i++)
        tmem_st4(t1_taddr + 448 + 24 + 4 * i, (uint32_t)__double2loint(wi[i].x), (uint32_t)__double2hiint(wi[i].x),
                 (uint32_t)__double2loint(wi[i].y), (uint32_t)__double2hiint(wi[i].y));
    } else {
      // pbs_quad_kernel: the table row of pass-2 twiddles (it writes its reader-side constants over it)
#pragma unroll
      for (int k2 = 0; k2 < 16; k2++) {
        const C2 w = k2 ? sT2[(uu >> 4) * kT2Pad + k2] : C2{1.0, 0.0};
        tmem_st4(t1_taddr + 448 + 4 * k2, (uint32_t)__double2loint(w.x), (uint32_t)__double2hiint(w.x),
                 (uint32_t)__double2loint(w.y), (uint32_t)__double2hiint(w.y));
      }
    }
    tmem_wait_st();
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  return t1_taddr;
}
// every thread of the CTA must call this before exiting
__device__ __forceinline__ void pair_tmem_free(uint32_t alloc_base) {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if ((threadIdx.x >> 5) == 0)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(alloc_base), "n"(kPbsTmemCols) : "memory");
}

struct PbsBatch {
  const uint64_t* lwe_in;   // [B][n+1]
  const uint64_t* lut;      // shared GLWE LUT, or nullptr for CBS mode
  size_t lut_stride;        // 0: one LUT for the whole batch, else per-ciphertext stride (elements)
  uint64_t* glwe_out;       // [B][2][2048]
  const C2* bsk;
  const void* const* ptrs;  // optional device table: ptrs[c] = LWE input of item c (graph executor)
  int batch, lwe_n, log_chi, log_v, cbs_radix_log, cbs_count;
};

__global__ void __launch_bounds__(kPbsPairs * 2 * kTeam, 1) pbs_kernel(PbsBatch P, DevTables tabs) {
  extern __shared__ __align__(16) unsigned char smem[];
  C2* sT1 = reinterpret_cast<C2*>(smem);
  C2* sT2 = sT1 + kT1Elems;
  load_tables(sT1, sT2, tabs);
  uint32_t tmem_alloc;
  const uint32_t t1_taddr = pair_tmem_init(sT1, sT2, tmem_alloc, true);
  const int pair = threadIdx.x / (2 * kTeam);
  const int npairs = blockDim.x / (2 * kTeam);  // 1..kPbsPairs pairs per CTA (fewer for small batches)
  const int h = (threadIdx.x / kTeam) & 1;
  C2* xb = reinterpret_cast<C2*>(smem + kPbsPairOff + pair * kPbsPairBytes);
  C2* fpark = pair < kPbsTmemFPairs ? nullptr
                                    : reinterpret_cast<C2*>(smem + kPbsPairOff + kPbsPairs * kPbsPairBytes) + (pair - kPbsTmemFPairs) * 2 * kTeam * 16;
  DevPairCx cx{(int)(threadIdx.x % kTeam), h, 1 + pair * 3 + h, 3 + pair * 3, t1_taddr, t1_taddr + kPbsTmemOwn0 + 64 * pair,
               t1_taddr + kPbsTmemF0 + 64 * (pair < kPbsTmemFPairs ? pair : 0), fpark};
  int G = 0;        // chunk position of this pair in the CTA-wide BSK chunk sequence
  int rounds = 0;   // ciphertexts the busiest pair (pair 0) of this CTA processes
  {
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + kPbsRingOff + kRingStages * kRingChunkBytes);
    cx.ring_s = smem_u32(smem + kPbsRingOff);
    cx.full_s = smem_u32(full);
    cx.rel = reinterpret_cast<unsigned*>(full + kRingStages);
    cx.bsk = P.bsk;
    cx.lwe_n = P.lwe_n;
    cx.npairs = npairs;                             // participants that count themselves off a chunk
    cx.elected = (threadIdx.x % (2 * kTeam)) == 0;  // one thread per pair
    if ((int)blockIdx.x < P.batch) rounds = (P.batch - (int)blockIdx.x + (int)gridDim.x * npairs - 1) / ((int)gridDim.x * npairs);
    cx.total = rounds * 4 * P.lwe_n;
    if (threadIdx.x == 0) {
      for (int st = 0; st < kRingStages; st++) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(cx.full_s + 8 * st) : "memory");
        cx.rel[st] = 0;
      }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0)
      for (int g0 = 0; g0 < kRingStages && g0 < cx.total; g0++) cx.ring_issue(g0);
  }
  // Persistent pairs: slot (pair, CTA) takes ciphertexts slot, slot + slots, ...  Slots are numbered
  // pair-major so that a trailing partial round leaves at most one busy pair on as many SMs as
  // possible (a pair alone on an SM runs ~1.3x faster than one sharing it with two others).
  for (int c = pair * gridDim.x + blockIdx.x; c < P.batch; c += gridDim.x * npairs) {
    PbsArgs A;
    A.lwe_in = P.ptrs ? static_cast<const uint64_t*>(P.ptrs[c]) : P.lwe_in + (size_t)c * (P.lwe_n + 1);
    A.lut = P.lut ? P.lut + (size_t)c * P.lut_stride : nullptr;
    A.glwe_out = P.glwe_out + (size_t)c * 2 * kN;
    A.bsk = P.bsk;
    A.lwe_n = P.lwe_n;
    A.log_chi = P.log_chi;
    A.log_v = P.log_v;
    A.cbs_radix_log = P.cbs_radix_log;
    A.cbs_count = P.cbs_count;
    pbs_pair_team(cx, A, xb, sT1, sT2, G);
  }
  // a pair with fewer ciphertexts than pair 0 (the tail of the batch) still counts itself off the remaining chunks
  if (cx.elected)
    for (; G < cx.total; G++) {
      mbar_wait_trap(cx.full_s + 8 * (G % kRingStages), (uint32_t)(G / kRingStages) & 1u);
      cx.bsk_release(G);
    }
  pair_tmem_free(tmem_alloc);
}

// ------------------------------------------------------------------------------------------
// K3q: latency mode of the blind rotation, one ciphertext per CTA on 4 teams (pbs_quad_team);
// chosen by launch_pbs when the batch has at most one ciphertext per SM.
// ------------------------------------------------------------------------------------------
// smem: pass-2 twiddles | GLWE accumulator | 4 exchange buffers | one staged BSK row (128 KiB) | mbarrier.
// The pass-1 twiddles are only needed to fill tensor memory at start-up and borrow the row buffer.
constexpr int kQuadT2Bytes = kT2Elems * 16;                                         // 1088
constexpr int kQuadRowBytes = 8 * kM * 16;                                           // 131072: one GGSW of the BSK
constexpr int kQuadSmem = kQuadT2Bytes + 2 * kN * 8 + 4 * kXBuf * 16 + kQuadRowBytes + 16;  // 231504


struct DevQuadCx {
  // Split gather: the two teams of a polynomial gather half of the rounded differences each and swap digits.
  // Teams (h, 0) and (h, 1) are warps {2h, 2h+1} and {4 + 2h, 5 + 2h}: thread u of both sits on the same tensor-memory lane,
  // so 16 packed digits change hands through eight columns of that lane (columns [64, 72) written by t = 0, [72, 80) by
  // t = 1) and one 128-thread barrier -- no shared memory (the kernel has none left) and no second gather.
  __device__ __forceinline__ void digit_xchg(uint32_t (&pk)[8]) const {
    tmem_st8(t1_taddr + 64 + 8 * t, pk);
    tmem_wait_st();
    asm volatile("bar.sync %0, 128;" ::"r"(5 + h) : "memory");
    tmem_ld8(pk, t1_taddr + 64 + 8 * (1 - t));
    tmem_wait_ld();
  }
  // reader-side pass-2 twiddles (team_ops.cuh: rt2_group_consts): 12 doubles per thread in the columns [448 + 24 t, 472 + 24 t)
  // of its lane (warps w and w + 4 share a lane quarter and differ in t).  Measured against the producer-side twiddles: 3.52 -> 3.36 ms
  // at batch 1, 3.39 -> 3.31 at 64.
  __device__ __forceinline__ void rt2(double (&tw)[6], C2 (&wi)[3], const C2*) const {
    uint32_t a[16], b[8];
    tmem_ld16(a, t1_taddr + 448 + 24 * t);
    tmem_ld8(b, t1_taddr + 448 + 24 * t + 16);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 6; i++) tw[i] = __hiloint2double((int)a[2 * i + 1], (int)a[2 * i]);
    wi[0] = C2{__hiloint2double((int)a[13], (int)a[12]), __hiloint2double((int)a[15], (int)a[14])};
    wi[1] = C2{__hiloint2double((int)b[1], (int)b[0]), __hiloint2double((int)b[3], (int)b[2])};
    wi[2] = C2{__hiloint2double((int)b[5], (int)b[4]), __hiloint2double((int)b[7], (int)b[6])};
  }
  int u, h, t;
  uint32_t t1_taddr;
  C2* row;          // staged BSK row
  uint64_t* mbar;   // completes when the bulk copy into `row` has landed
  __device__ __forceinline__ void sync() const { asm volatile("bar.sync %0, 64;" ::"r"(1 + 2 * h + t) : "memory"); }
  __device__ __forceinline__ void quad_sync() const { __syncthreads(); }
  // one thread of the CTA starts the bulk copy (TMA) of the next step's 128 KiB BSK row
  __device__ __forceinline__ void row_prefetch(const C2* src) const {
    if (threadIdx.x == 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)), "r"((uint32_t)kQuadRowBytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(smem_u32(row)), "l"(src), "r"((uint32_t)kQuadRowBytes), "r"(smem_u32(mbar)) : "memory");
    }
  }
  // k-th completed copy: mbarrier phase parity k & 1
  __device__ __forceinline__ const C2* row_wait(int k, const C2*) const {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "ROW_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra ROW_DONE;\n\t"
        "bra ROW_WAIT;\n\t"
        "ROW_DONE:\n\t"
        "}" ::"r"(smem_u32(mbar)), "r"((uint32_t)(k & 1)) : "memory");
    return row;
  }
  __device__ __forceinline__ C2 row_load(const C2* p) const {
    C2 r;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "r"(smem_u32(p)) : "memory");
    return r;
  }
  template <bool CONJ>
  __device__ __forceinline__ void t1_mul(C2 (&v)[16], const C2* T1) const {
#pragma unroll
    for (int half = 0; half < 2; half++) {
      uint32_t r0[16], r1[16];
      tmem_ld16(r0, t1_taddr + 32 * half);
      tmem_ld16(r1, t1_taddr + 32 * half + 16);
      tmem_wait_ld();
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const C2 w0{__hiloint2double((int)r0[4 * i + 1], (int)r0[4 * i]), __hiloint2double((int)r0[4 * i + 3], (int)r0[4 * i + 2])};
        const C2 w1{__hiloint2double((int)r1[4 * i + 1], (int)r1[4 * i]), __hiloint2double((int)r1[4 * i + 3], (int)r1[4 * i + 2])};
        const int ka = 8 * half + i, kb = 8 * half + 4 + i;
        v[ka] = CONJ ? cmul_conj(v[ka], w0) : cmul(v[ka], w0);
        v[kb] = CONJ ? cmul_conj(v[kb], w1) : cmul(v[kb], w1);
      }
    }
  }
};

__global__ void __launch_bounds__(4 * kTeam, 1) pbs_quad_kernel(PbsBatch P, DevTables tabs) {
  extern __shared__ __align__(16) unsigned char smem[];
  C2* sT2 = reinterpret_cast<C2*>(smem);
  uint64_t* acc = reinterpret_cast<uint64_t*>(smem + kQuadT2Bytes);
  C2* xb = reinterpret_cast<C2*>(smem + kQuadT2Bytes + 2 * kN * 8);
  C2* row = reinterpret_cast<C2*>(smem + kQuadT2Bytes + 2 * kN * 8 + 4 * kXBuf * 16);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + kQuadT2Bytes + 2 * kN * 8 + 4 * kXBuf * 16 + kQuadRowBytes);
  C2* sT1 = row;  // borrowed until tensor memory holds the pass-1 twiddles
  load_tables(sT1, sT2, tabs);
  uint32_t tmem_alloc;
  const uint32_t t1_taddr = pair_tmem_init(sT1, sT2, tmem_alloc);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(mbar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  {  // every thread's reader-side pass-2 constants over the table row pair_tmem_init left in [448, 512)
    const int tm = threadIdx.x / kTeam, uu = threadIdx.x % kTeam;
    double tw[6];
    C2 wi[3];
    rt2_group_consts(sT2, uu >> 4, 2 * (tm & 1) + (tm >> 1), tw, wi);
    const uint32_t base = t1_taddr + 448 + 24 * (tm >> 1);
#pragma unroll
    for (int i = 0; i < 3; i++)
      tmem_st4(base + 4 * i, (uint32_t)__double2loint(tw[2 * i]), (uint32_t)__double2hiint(tw[2 * i]), (uint32_t)__double2loint(tw[2 * i + 1]),
               (uint32_t)__double2hiint(tw[2 * i + 1]));
#pragma unroll
    for (int i = 0; i < 3; i++)
      tmem_st4(base + 12 + 4 * i, (uint32_t)__double2loint(wi[i].x), (uint32_t)__double2hiint(wi[i].x), (uint32_t)__double2loint(wi[i].y),
               (uint32_t)__double2hiint(wi[i].y));
    tmem_wait_st();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  }
  const int team = threadIdx.x / kTeam;
  // team w = (h, t) with h = w & 1, t = w >> 1: the two teams that run the inverse transforms (t = 0) are warps
  // 0..3, one per SM sub-partition (warp % 4) -- with h = w >> 1 they were warps 0,1,4,5, i.e. the FP64-issue-bound
  // inverse phase ran on two of the four sub-partitions.
  DevQuadCx cx{(int)(threadIdx.x % kTeam), team & 1, team >> 1, t1_taddr, row, mbar};
  int copies = 0;  // bulk copies completed so far on this CTA's mbarrier (phase parity bookkeeping)
  for (int c = blockIdx.x; c < P.batch; c += gridDim.x) {
    PbsArgs A;
    A.lwe_in = P.ptrs ? static_cast<const uint64_t*>(P.ptrs[c]) : P.lwe_in + (size_t)c * (P.lwe_n + 1);
    A.lut = P.lut ? P.lut + (size_t)c * P.lut_stride : nullptr;
    A.glwe_out = P.glwe_out + (size_t)c * 2 * kN;
    A.bsk = P.bsk;
    A.lwe_n = P.lwe_n;
    A.log_chi = P.log_chi;
    A.log_v = P.log_v;
    A.cbs_radix_log = P.cbs_radix_log;
    A.cbs_count = P.cbs_count;
    pbs_quad_team(cx, A, acc, xb, sT1, sT2, copies);
    cx.quad_sync();
  }
  pair_tmem_free(tmem_alloc);
}

// ------------------------------------------------------------------------------------------
// K5+K6: trace (+ CBS pre-processing) and scheme switch, one team per (ciphertext, level).
// ------------------------------------------------------------------------------------------
// DevCx of the trace / scheme-switch kernel: tensor-memory columns [0,64) T1 | [64,128) T2 (per lane quarter, shared by the
// two warps of the quarter: warps w and w + 4 have the same thread-in-team index) | 64 columns per warp of parked states
struct DevTrCx : DevCx {
  static constexpr bool kTmemTwiddles = true;  // twiddles of both passes in tensor memory
  uint32_t tw_taddr;
  template <bool CONJ>
  __device__ __forceinline__ void t1_mul(C2 (&v)[16]) const {
#pragma unroll
    for (int g = 0; g < 4; g++) {
      uint32_t r[16];
      tmem_ld16(r, tw_taddr + 16 * g);
      tmem_wait_ld();
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const C2 w{__hiloint2double((int)r[4 * i + 1], (int)r[4 * i]), __hiloint2double((int)r[4 * i + 3], (int)r[4 * i + 2])};
        const int k = 4 * g + i;
        v[k] = CONJ ? cmul_conj(v[k], w) : cmul(v[k], w);
      }
    }
  }
  template <bool CONJ>
  __device__ __forceinline__ void t2_mul(C2 (&v)[16]) const {
#pragma unroll
    for (int g = 0; g < 4; g++) {
      uint32_t r[16];
      tmem_ld16(r, tw_taddr + 64 + 16 * g);
      tmem_wait_ld();
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const C2 w{__hiloint2double((int)r[4 * i + 1], (int)r[4 * i]), __hiloint2double((int)r[4 * i + 3], (int)r[4 * i + 2])};
        const int k = 4 * g + i;
        if (k) v[k] = CONJ ? cmul_conj(v[k], w) : cmul(v[k], w);
      }
    }
  }
};
constexpr int kTrTmemCols = 256;  // [0,128) twiddles | [128,256) parked states, 64 columns per warp of a lane quarter
constexpr int kTrTeams = 4;  // teams (ciphertext levels) per CTA: four fit the shared memory of one CTA per SM
constexpr int kTrTeamBytes = 2 * kN * 8 + kXBuf * 16;                 // g + xbuf = 49408 (digits are stateless)
constexpr int kTrSmem = kTableBytes + kTrTeams * kTrTeamBytes;        // 215104

// Peer arenas of a sharded graph (graph.cuh): byte offsets from this rank's arena to the arenas of the other
// ranks as mapped into this process (CUDA IPC), and the ranks they belong to.
constexpr int kMaxPeers = 7;
struct PeerOffsets {
  int n;
  int rank_of[kMaxPeers];
  long long off[kMaxPeers];
};

struct TraceSsBatch {
  const uint64_t* glwe_in;  // mode 0: [B][2][2048] PBS outputs; mode 1: [B][...] GLWEs; mode 2: [B][l][2][2048] GLEVs
  uint64_t* glev_out;       // optional [B][levels][2][2048] (mode 0/1)
  C2* ggsw_out;             // optional [B][2][l][2][1024]
  const C2* ak;
  const C2* ssk;
  const uint32_t* kinv;
  const void* const* ptrs;  // optional device table: ptrs[c] = input (GLWE or GLEV base) of item c
  int batch, levels, mode;
  int cbs_radix_log, cbs_count, tr_radix_log, tr_count, ss_radix_log, ss_count;
  double out_scale;
  PeerOffsets peers;       // n = 0: GGSWs are stored locally only
};

template <bool PEERS>
__global__ void __launch_bounds__(kTrTeams * kTeam, 1) trace_ss_kernel(const __grid_constant__ TraceSsBatch P, DevTables tabs) {
  extern __shared__ __align__(16) unsigned char smem[];
  C2* sT1 = reinterpret_cast<C2*>(smem);
  C2* sT2 = sT1 + kT1Elems;
  load_tables(sT1, sT2, tabs);
  // tensor memory: 64 columns per warp for the parked decomposition states (warps w and w + 4 share a lane quarter)
  __shared__ uint32_t tmem_base;
  const int warp = threadIdx.x >> 5;
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     (uint32_t)__cvta_generic_to_shared(&tmem_base)), "n"(kTrTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_alloc = tmem_base;
  const uint32_t tw_taddr = tmem_alloc + ((uint32_t)((warp & 3) * 32) << 16);
  if (warp < 4) {  // twiddles of thread-in-team index uu = 32 (warp & 1) + lane, for both warps of this lane quarter
    const int uu = (warp & 1) * 32 + (threadIdx.x & 31);
#pragma unroll
    for (int k = 0; k < 16; k++) {
      const C2 w1 = sT1[k * 64 + uu];
      tmem_st4(tw_taddr + 4 * k, (uint32_t)__double2loint(w1.x), (uint32_t)__double2hiint(w1.x), (uint32_t)__double2loint(w1.y),
               (uint32_t)__double2hiint(w1.y));
      const C2 w2 = k ? sT2[(uu >> 4) * kT2Pad + k] : C2{1.0, 0.0};
      tmem_st4(tw_taddr + 64 + 4 * k, (uint32_t)__double2loint(w2.x), (uint32_t)__double2hiint(w2.x), (uint32_t)__double2loint(w2.y),
               (uint32_t)__double2hiint(w2.y));
    }
    tmem_wait_st();
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const int team = threadIdx.x / kTeam;
  const int item = blockIdx.x * (blockDim.x / kTeam) + team;
  if (item < P.batch * P.levels) {  // no early return: every thread must reach the deallocation barrier
    const int c = item / P.levels, level = item % P.levels;
    unsigned char* base = smem + kTableBytes + team * kTrTeamBytes;
    uint64_t* g = reinterpret_cast<uint64_t*>(base);
    C2* xbuf = reinterpret_cast<C2*>(base + 2 * kN * 8);
    DevTrCx cx;
    cx.u = (int)(threadIdx.x % kTeam);
    cx.bar = team + 1;
    cx.rp_taddr = tw_taddr + 128u + (uint32_t)(warp >> 2) * 64;
    cx.tw_taddr = tw_taddr;
    TraceSsArgs A;
    const size_t glwe = 2 * kN;
    if (P.ptrs) A.glwe_in = static_cast<const uint64_t*>(P.ptrs[c]) + (P.mode == 2 ? (size_t)level * glwe : 0);
    else if (P.mode == 0) A.glwe_in = P.glwe_in + (size_t)c * glwe;
    else A.glwe_in = P.glwe_in + (size_t)item * glwe;
    A.glev_out = P.glev_out ? P.glev_out + (size_t)item * glwe : nullptr;
    A.ggsw_out = P.ggsw_out ? P.ggsw_out + (size_t)c * 2 * P.cbs_count * 2 * kM : nullptr;
    A.ak = P.ak;
    A.ssk = P.ssk;
    A.kinv = P.kinv;
    A.level = level;
    A.mode = P.mode;
    A.cbs_radix_log = P.cbs_radix_log;
    A.cbs_count = P.cbs_count;
    A.tr_radix_log = P.tr_radix_log;
    A.tr_count = P.tr_count;
    A.ss_radix_log = P.ss_radix_log;
    A.ss_count = P.ss_count;
    A.out_scale = P.out_scale;
    A.n_peers = P.peers.n;
    A.peer_off = P.peers.off;
    trace_ss_team<PEERS>(cx, A, g, xbuf, sT1, sT2);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_alloc), "n"(kTrTmemCols) : "memory");
}

// ------------------------------------------------------------------------------------------
// Peer-memory level barrier and broadcast of a sharded graph run (no NCCL on the data path).
// flags[world] (u64) sit at the start of every rank's arena: flags[src] on rank dst = the last epoch rank src
// has signalled to dst.  One warp: thread i signals peer i (after a system-scope fence that orders the P2P stores
// of the preceding kernels before the flag), then waits for peer i's signal.  A rank that never arrives trips the
// timeout and sets *err instead of hanging the GPU.
// ------------------------------------------------------------------------------------------
__global__ void peer_barrier_kernel(unsigned long long* flags, PeerOffsets peers, int rank, unsigned long long epoch, int* err,
                                    unsigned long long timeout_ns) {
  const int i = threadIdx.x;
  __threadfence_system();
  if (*reinterpret_cast<volatile int*>(err)) return;  // an earlier barrier of this run timed out: do not wait again
  if (i < peers.n) {
    volatile unsigned long long* theirs = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(flags) + peers.off[i]) + rank;
    *theirs = epoch;
    __threadfence_system();
    volatile unsigned long long* mine = flags + peers.rank_of[i];
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (*mine < epoch) {
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > timeout_ns) { atomicExch(err, 1); break; }
      __nanosleep(200);
    }
  }
  __threadfence_system();
}

// Gathers the ciphertexts behind a graph's Output nodes into one contiguous staging buffer, so that they leave
// the device in as few copies as their host buffers allow: item k = n8[k] 8-byte words from src[k] to dst + off8[k]
// (every ciphertext is a whole number of u64 words; an L1 LWE is 2049 of them).
__global__ void gather_outputs_kernel(unsigned long long* dst, const void* const* src, const unsigned long long* off8, const unsigned* n8) {
  const int k = blockIdx.y;
  const unsigned long long* s = static_cast<const unsigned long long*>(src[k]);
  unsigned long long* d = dst + off8[k];
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n8[k]; i += gridDim.x * blockDim.x) d[i] = s[i];
}

// dst_r[i] = src[i] for every peer r (the keyswitch outputs of this rank's trees: 5 KB each)
__global__ void peer_bcast_kernel(const uint4* src, size_t n16, PeerOffsets peers) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) {
    const uint4 v = src[i];
    for (int r = 0; r < peers.n; r++)
      *reinterpret_cast<uint4*>(reinterpret_cast<char*>(const_cast<uint4*>(src + i)) + peers.off[r]) = v;
  }
}

// All box-ciphertext-handle traffic of one rank in one run phase (box.cuh): item k copies n8 u64 words from src to
// each of its n_dst destinations -- this rank's arena, its own replica, or the replicas of the other ranks (peer
// stores over NVLink).  The table travels as a __grid_constant__ parameter, so every launch works on its own snapshot
// of the bindings.  Items whose pointers are all 16-byte aligned move 16-byte words (an L1 LWE is 2049 u64 words:
// the odd word goes in the tail loop); the others move u64 words.
constexpr int kBoxCopyMaxDst = 8;
struct BoxCopyItem {
  const unsigned long long* src;
  unsigned long long* dst[kBoxCopyMaxDst];
  unsigned n8;
  int n_dst;
};
template <int N>
struct BoxCopyTable {
  BoxCopyItem item[N];
};
constexpr int kBoxCopySmall = 32;   // 2.6 KB of parameters
constexpr int kBoxCopyLarge = 400;  // 32 000 bytes: within the 32 764-byte kernel parameter limit (CUDA >= 12.1)
static_assert(sizeof(BoxCopyTable<kBoxCopyLarge>) <= 32764, "box copy table exceeds the kernel parameter limit");

template <int N>
__global__ void __launch_bounds__(256) box_copy_kernel(const __grid_constant__ BoxCopyTable<N> t) {
  const BoxCopyItem& it = t.item[blockIdx.y];
  const int nd = it.n_dst;
  bool v16 = (reinterpret_cast<uintptr_t>(it.src) & 15) == 0;
  for (int d = 0; d < nd; d++) v16 &= (reinterpret_cast<uintptr_t>(it.dst[d]) & 15) == 0;
  const size_t n16 = v16 ? it.n8 / 2 : 0;
  const size_t stride = (size_t)gridDim.x * blockDim.x, first = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  for (size_t i = first; i < n16; i += stride) {
    const uint4 v = reinterpret_cast<const uint4*>(it.src)[i];
    for (int d = 0; d < nd; d++) reinterpret_cast<uint4*>(it.dst[d])[i] = v;
  }
  for (size_t i = 2 * n16 + first; i < it.n8; i += stride) {
    const unsigned long long v = it.src[i];
    for (int d = 0; d < nd; d++) it.dst[d][i] = v;
  }
}

// ------------------------------------------------------------------------------------------
// K2: runtime CMUX / external product, one team per GLWE output.
// ------------------------------------------------------------------------------------------
constexpr int kCmuxTeams = 4;
constexpr int kCmuxTeamBytes = 32 * 64 * 8 + kXBuf * 16;          // state + xbuf = 33024
constexpr int kCmuxSmem = kTableBytes + kCmuxTeams * kCmuxTeamBytes;  // 149568

struct CmuxBatch {
  uint64_t* out;          // [B][glwe_per_item][2][2048]
  const uint64_t* d0;     // nullptr: plain external product of d1
  const uint64_t* d1;
  const C2* ggsw;         // 2^-10 scaled
  size_t ggsw_stride;     // elements between consecutive items' GGSWs (0 = shared)
  const void* const* ptrs;  // optional device table, 3 per item: {ggsw, d0 (may be null), d1} (graph executor)
  void* const* out_ptrs;    // optional device table: out_ptrs[c] = output of GLWE c (recycled slots of the graph arena)
  int batch;              // number of GLWE outputs
  int glwe_per_item;      // 1 for cmux, l_cbs for glev_cmux (GLWEs sharing one GGSW)
  int radix_log, count;
};

__global__ void __launch_bounds__(kCmuxTeams * kTeam, 1) cmux_kernel(CmuxBatch P, DevTables tabs) {
  extern __shared__ __align__(16) unsigned char smem[];
  C2* sT1 = reinterpret_cast<C2*>(smem);
  C2* sT2 = sT1 + kT1Elems;
  pdl_launch_dependents();
  load_tables(sT1, sT2, tabs);
  pdl_wait();  // the ciphertexts come from earlier kernels of the stream
  const int team = threadIdx.x / kTeam;
  const int c = blockIdx.x * (blockDim.x / kTeam) + team;
  if (c >= P.batch) return;
  unsigned char* base = smem + kTableBytes + team * kCmuxTeamBytes;
  uint64_t* st = reinterpret_cast<uint64_t*>(base);
  C2* xbuf = reinterpret_cast<C2*>(base + 32 * 64 * 8);
  DevCx cx{(int)(threadIdx.x % kTeam), team + 1};
  const size_t glwe = 2 * kN;
  if (P.ptrs) {
    const int item = c / P.glwe_per_item;
    const size_t off = (size_t)(c % P.glwe_per_item) * glwe;
    const uint64_t* d0 = static_cast<const uint64_t*>(P.ptrs[3 * item + 1]);
    cmux_team(cx, P.out_ptrs ? static_cast<uint64_t*>(P.out_ptrs[c]) : P.out + (size_t)c * glwe, d0 ? d0 + off : nullptr,
              static_cast<const uint64_t*>(P.ptrs[3 * item + 2]) + off, static_cast<const C2*>(P.ptrs[3 * item]), st,
              xbuf, sT1, sT2, P.radix_log, P.count);
    return;
  }
  cmux_team(cx, P.out + (size_t)c * glwe, P.d0 ? P.d0 + (size_t)c * glwe : nullptr, P.d1 + (size_t)c * glwe,
            P.ggsw + (size_t)(c / P.glwe_per_item) * P.ggsw_stride, st, xbuf, sT1, sT2, P.radix_log, P.count);
}

// ------------------------------------------------------------------------------------------
// K2w: latency-oriented CMUX, one CTA of 8 teams per GLWE output (cmux_wide); chosen by
// launch_cmux when there are fewer outputs than SMs (the ripple MUX chain of a Parasol program).
// ------------------------------------------------------------------------------------------
// Both GLWE inputs (2 x 32 KiB) are staged in shared memory by two bulk copies (TMA): the four teams
// that decompose the same polynomial would otherwise each pull it through L2 (256 KiB per CMUX instead
// of 64 KiB, which made the load phase L2->SM bandwidth bound: 6.9 k of the kernel's 22 k clocks).
constexpr int kWideGlweBytes = 2 * kN * 8;
constexpr int kWideSmem = kTableBytes + kWideTeams * kXBuf * 16 + 2 * kWideGlweBytes + 16;  // 216144
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity);

struct DevWideCx {
  int u, team;
  __device__ __forceinline__ void sync() const { asm volatile("bar.sync %0, 64;" ::"r"(team + 1) : "memory"); }
  __device__ __forceinline__ void cta_sync() const { __syncthreads(); }
};

__global__ void __launch_bounds__(kWideTeams * kTeam, 1) cmux_wide_kernel(CmuxBatch P, DevTables tabs) {
  extern __shared__ __align__(16) unsigned char smem[];
  C2* sT1 = reinterpret_cast<C2*>(smem);
  C2* sT2 = sT1 + kT1Elems;
  pdl_launch_dependents();
  const int c = blockIdx.x;
  {  // the selector GGSW (256 KiB) is pulled towards L2 while the predecessor level still runs
    const C2* gg = P.ptrs ? static_cast<const C2*>(P.ptrs[3 * (c / P.glwe_per_item)]) : P.ggsw + (size_t)(c / P.glwe_per_item) * P.ggsw_stride;
    const char* q = reinterpret_cast<const char*>(gg);
    for (int i = threadIdx.x; i < (int)(2 * 2 * 4 * kM * sizeof(C2) / 128) && P.count == 4; i += blockDim.x) prefetch_l2(q + (size_t)i * 128);
  }
  C2* xb = reinterpret_cast<C2*>(smem + kTableBytes);
  uint64_t* sd1 = reinterpret_cast<uint64_t*>(smem + kTableBytes + kWideTeams * kXBuf * 16);
  uint64_t* sd0 = sd1 + 2 * kN;
  uint64_t* mbar = sd0 + 2 * kN;
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(mbar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  load_tables(sT1, sT2, tabs);  // ends with a CTA barrier: the mbarrier is initialised for everyone
  const size_t glwe = 2 * kN;
  const int item = c / P.glwe_per_item;
  const size_t off = P.ptrs ? (size_t)(c % P.glwe_per_item) * glwe : (size_t)c * glwe;
  const uint64_t* d0 = P.ptrs ? static_cast<const uint64_t*>(P.ptrs[3 * item + 1]) : P.d0;
  const uint64_t* d1 = P.ptrs ? static_cast<const uint64_t*>(P.ptrs[3 * item + 2]) : P.d1;
  const C2* ggsw = P.ptrs ? static_cast<const C2*>(P.ptrs[3 * item]) : P.ggsw + (size_t)item * P.ggsw_stride;
  pdl_wait();  // the GLWE inputs come from earlier kernels of the stream
  if (threadIdx.x == 0) {
    const uint32_t bytes = d0 ? 2 * kWideGlweBytes : kWideGlweBytes;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(sd1)), "l"(d1 + off), "r"((uint32_t)kWideGlweBytes), "r"(smem_u32(mbar)) : "memory");
    if (d0)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(smem_u32(sd0)), "l"(d0 + off), "r"((uint32_t)kWideGlweBytes), "r"(smem_u32(mbar)) : "memory");
  }
  DevWideCx cx{(int)(threadIdx.x % kTeam), (int)(threadIdx.x / kTeam)};
  mbar_wait(smem_u32(mbar), 0);
  cmux_wide(cx, P.out_ptrs ? static_cast<uint64_t*>(P.out_ptrs[c]) : P.out + (size_t)c * glwe, d0 ? sd0 : nullptr, sd1, ggsw, xb, sT1, sT2,
            P.radix_log, P.count);
}

// ------------------------------------------------------------------------------------------
// K4: LWE keyswitch L1 -> L0 (ops/keyswitch/lwe_keyswitch.rs:23-62), integer only.
// out = (0, b) - sum_i sum_t digit_t(a_i) * KSK[i][l-1-t].  A CTA owns kKsBatch inputs, all n0+1
// output columns and a contiguous slice of the mask index i (grid.y = split-K over i, so small
// batches still spread the 62.7 MB KSK sweep over the whole GPU); each KSK row is read once per
// kKsBatch ciphertexts.  The rows of mask element i+1 are prefetched into registers while
// element i is accumulated.  With more than one slice the partial sums are combined with u64
// atomics into a zero-initialised output (wrapping adds commute, so the result is bit-exact).
//
// Balanced digits d in [-B/2, B/2) are handled as UNSIGNED digits u = d + B/2 read straight out of
// the bit fields of round(a_i) + sum_t (B/2) B^t (no carry chain, see radix_offset), so that one
// u64 multiply-add is two 32-bit IMADs (IMAD.WIDE.U32 for the low word, IMAD for the high word);
// the surplus (B/2) * sum_{i,t} KSK[i][t] is a constant of the key, precomputed per block of
// kKsBlock mask elements (ksk_colsum_kernel) and subtracted once per CTA.
// ------------------------------------------------------------------------------------------
constexpr int kKsBatch = 16;
constexpr int kKsThreads = 320;
constexpr int kKsMaxLevels = 8;
constexpr int kKsBlock = 32;  // mask elements per precomputed column-sum block; slices are multiples of it

struct KsBatch {
  uint64_t* out;        // [B][n0+1]
  const uint64_t* in;   // [B][n1+1]
  const uint64_t* ksk;  // [n1][l][n0+1]
  const uint64_t* colsum;  // [ceil(n1 / kKsBlock)][n0+1]: sum over the block's i and all levels of ksk
  const void* const* ptrs;  // optional device table: ptrs[b] = L1 LWE input of item b
  int batch, n1, n0, radix_log, count;
  int slice;            // mask elements per grid.y slice (n1 when not split), a multiple of kKsBlock
};

// colsum[blk][c] = sum_{i in block blk} sum_t ksk[i][t][c]   (one thread per (blk, c); run once per key)
__global__ void ksk_colsum_kernel(uint64_t* colsum, const uint64_t* ksk, int n1, int levels, int cols) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, blk = blockIdx.y;
  if (c >= cols) return;
  uint64_t acc = 0;
  const int i1 = min(n1, (blk + 1) * kKsBlock);
  for (int i = blk * kKsBlock; i < i1; i++)
    for (int t = 0; t < levels; t++) acc += ksk[((size_t)i * levels + t) * cols + c];
  colsum[(size_t)blk * cols + c] = acc;
}

// acc += k * u (mod 2^64) for a 32-bit u as two IMADs: the compiler does not form the accumulating
// IMAD.WIDE from C (it multiplies, then adds with carry: 5 instructions).
__device__ __forceinline__ void mad_u64_u32(uint64_t& acc, uint64_t k, uint32_t u) {
  asm("{\n\t"
      ".reg .u32 klo, khi, alo, ahi;\n\t"
      "mov.b64 {klo, khi}, %1;\n\t"
      "mad.wide.u32 %0, klo, %2, %0;\n\t"
      "mov.b64 {alo, ahi}, %0;\n\t"
      "mad.lo.u32 ahi, khi, %2, ahi;\n\t"
      "mov.b64 %0, {alo, ahi};\n\t"
      "}"
      : "+l"(acc)
      : "l"(k), "r"(u));
}

template <int L>
__global__ void __launch_bounds__(kKsThreads) keyswitch_kernel(KsBatch P) {
  extern __shared__ __align__(16) unsigned char smem[];
  uint32_t* st = reinterpret_cast<uint32_t*>(smem);  // [kKsBatch][slice] rounded + offset states (l*logB <= 31 bits)
  const int b0 = blockIdx.x * kKsBatch;
  const int nb = min(kKsBatch, P.batch - b0);
  const int i_begin = blockIdx.y * P.slice;
  const int ni = min(P.slice, P.n1 - i_begin);
  const bool split = gridDim.y > 1;
  const uint32_t off = (uint32_t)radix_offset(P.radix_log, P.count);
  for (int idx = threadIdx.x; idx < kKsBatch * ni; idx += blockDim.x) {
    const int b = idx / ni, i = idx % ni;
    const uint64_t* src = b < nb ? (P.ptrs ? static_cast<const uint64_t*>(P.ptrs[b0 + b]) : P.in + (size_t)(b0 + b) * (P.n1 + 1)) : nullptr;
    // padding rows of a ragged tile get the all-(B/2) state: unsigned digits B/2 = signed digits 0
    st[b * P.slice + i] = (src ? (uint32_t)radix_round(src[i_begin + i], P.radix_log, P.count) : 0u) + off;
  }
  __syncthreads();
  const int cols = P.n0 + 1;
  const int c0 = threadIdx.x, c1 = threadIdx.x + kKsThreads;
  const bool has0 = c0 < cols, has1 = c1 < cols;
  uint64_t acc0[kKsBatch], acc1[kKsBatch];
#pragma unroll
  for (int b = 0; b < kKsBatch; b++) { acc0[b] = 0; acc1[b] = 0; }
  const uint32_t mask = (1u << P.radix_log) - 1;
  uint64_t k0[L], k1[L], n0v[L], n1v[L];
  auto load_rows = [&](int i, uint64_t (&r0)[L], uint64_t (&r1)[L]) {
    const uint64_t* row = P.ksk + (size_t)(i_begin + i) * L * cols;
#pragma unroll
    for (int t = 0; t < L; t++) {  // digit t (LSB first) pairs with level l-1-t (lev_ciphertext_ops.rs:36)
      const uint64_t* r = row + (size_t)(L - 1 - t) * cols;
      r0[t] = has0 ? __ldg(reinterpret_cast<const unsigned long long*>(r + c0)) : 0;
      r1[t] = has1 ? __ldg(reinterpret_cast<const unsigned long long*>(r + c1)) : 0;
    }
  };
  if (ni > 0) load_rows(0, k0, k1);
  for (int i = 0; i < ni; i++) {
    if (i + 1 < ni) load_rows(i + 1, n0v, n1v);
#pragma unroll
    for (int b = 0; b < kKsBatch; b++) {
      uint32_t s = st[b * P.slice + i];
#pragma unroll
      for (int t = 0; t < L; t++) {
        const uint32_t u = s & mask;  // unsigned digit = signed digit + B/2
        s >>= P.radix_log;
        mad_u64_u32(acc0[b], k0[t], u);
        mad_u64_u32(acc1[b], k1[t], u);
      }
    }
#pragma unroll
    for (int t = 0; t < L; t++) { k0[t] = n0v[t]; k1[t] = n1v[t]; }
  }
  // (B/2) * sum of this slice's KSK rows
  uint64_t s0 = 0, s1 = 0;
  for (int blk = i_begin / kKsBlock; blk * kKsBlock < i_begin + ni; blk++) {
    if (has0) s0 += P.colsum[(size_t)blk * cols + c0];
    if (has1) s1 += P.colsum[(size_t)blk * cols + c1];
  }
  s0 <<= P.radix_log - 1;
  s1 <<= P.radix_log - 1;
#pragma unroll
  for (int b = 0; b < kKsBatch; b++) {
    if (b >= nb) break;
    uint64_t* o = P.out + (size_t)(b0 + b) * cols;
    uint64_t body = 0;
    if (blockIdx.y == 0)
      body = (P.ptrs ? static_cast<const uint64_t*>(P.ptrs[b0 + b]) : P.in + (size_t)(b0 + b) * (P.n1 + 1))[P.n1];
    const uint64_t v0 = (c0 == P.n0 ? body : 0) - (acc0[b] - s0);
    const uint64_t v1 = (c1 == P.n0 ? body : 0) - (acc1[b] - s1);
    if (split) {
      if (has0) atomicAdd(reinterpret_cast<unsigned long long*>(o + c0), (unsigned long long)v0);
      if (has1) atomicAdd(reinterpret_cast<unsigned long long*>(o + c1), (unsigned long long)v1);
    } else {
      if (has0) o[c0] = v0;
      if (has1) o[c1] = v1;
    }
  }
}

// ------------------------------------------------------------------------------------------
// K4u: the keyswitch as a dense integer contraction on the 5th-generation tensor cores (tcgen05.mma kind::i8,
// TMEM accumulators).
//   out[b][c] = (0, body_b) - sum_{k=(i,t)} d[b][k] * KSK[k][c]   is   [B x 12288] x [12288 x 638] mod 2^64.
// With unsigned digits u = d + B/2 in {0..B-1} (see K4) and the KSK split into its 8 BYTE PLANES,
//   sum_k u[b][k] * KSK[k][c] = sum_j 2^(8j) * (U x P_j)[b][c],   P_j[k][c] = byte j of KSK[k][c],
// every U x P_j is an exact u8 x u8 -> s32 GEMM (12288 * 3 * 255 < 2^24), i.e. 8 int8 tensor-core
// GEMMs whose results are recombined with shifts in the epilogue; the surplus (B/2) * sum_k KSK[k][c]
// is the same per-key constant as in K4.  K is walked in chunks of (kKtIC mask elements, one digit level).
// ------------------------------------------------------------------------------------------
constexpr int kKtIC = 512;

// colsum[c * levels + t][col] = sum_{i in chunk c} ksk[i][levels-1-t][col]
__global__ void ks_tc_colsum_kernel(uint64_t* colsum, const uint64_t* ksk, int n1, int levels, int cols) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x, chunk = blockIdx.y;
  if (col >= cols) return;
  const int c = chunk / levels, t = chunk % levels;
  uint64_t acc = 0;
  for (int i = c * kKtIC; i < (c + 1) * kKtIC && i < n1; i++) acc += ksk[((size_t)i * levels + (levels - 1 - t)) * cols + col];
  colsum[(size_t)chunk * cols + col] = acc;
}

// st16[b][i] = round(a_i of input b) + radix_offset: the digit source of K4u, computed once per
// launch instead of once per column block
__global__ void ks_tc_states_kernel(uint16_t* st16, const uint64_t* in, const void* const* ptrs, int batch, int n1,
                                    int radix_log, int count) {
  const uint32_t off = (uint32_t)radix_offset(radix_log, count);
  const size_t total = (size_t)batch * n1;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const size_t b = e / n1;
    const int i = (int)(e % n1);
    const uint64_t* src = ptrs ? static_cast<const uint64_t*>(ptrs[b]) : in + b * (size_t)(n1 + 1);
    st16[e] = (uint16_t)((uint32_t)radix_round(src[i], radix_log, count) + off);
  }
}

// CTA tile 128 ciphertexts x 64 columns x 8 planes = 8 accumulators of 64 TMEM columns (all 512).
// Per k-step (32 digits): the 16 KiB of B (8 planes x 64 columns x 32 bytes, stored by
// ks_umma_prepare_kernel in the canonical K-major core-matrix layout) arrive by ONE bulk copy
// (cp.async.bulk -> mbarrier), the 4 KiB A tile is cut out of the u16 digit states by 128 producer
// threads (thread = ciphertext row), one thread issues the 8 MMAs and commits them to the stage's
// "empty" barrier.  6-stage ring; warps 0-3 produce A and run the epilogue (TMEM lane = row),
// warp 4 feeds B, warp 5 issues the MMAs.  Epilogue: recombine the planes with shifts, remove the
// digit offset (per-key column sums), subtract from (0, body); grid.z splits K (u64 atomics).
constexpr int kKuM = 128, kKuN = 64, kKuStages = 6;
constexpr int kKuATile = kKuM * 32, kKuBPlane = kKuN * 32, kKuBTile = 8 * kKuBPlane;   // 4096, 2048, 16384
constexpr int kKuSmem = kKuStages * (kKuATile + kKuBTile) + 1024;                      // + barriers, surplus table

struct KsUBatch {
  uint64_t* out;
  const uint64_t* in;
  const void* const* ptrs;
  const uint16_t* st16;     // [B][n1] rounded + offset states
  const uint8_t* btiles;    // [n_blocks][k_steps][8 planes][2 kc][8 col-groups][8 cols][16 B]
  const uint64_t* colsum;   // [chunks][n0+1], chunk = c * L + t  (ks_tc_colsum_kernel)
  int batch, n1, n0, radix_log, count;
  int chunks_per_cta;
};

// One thread per 16-byte row piece: btiles[...][col % 8] = bytes of plane j of KSK for 16 consecutive k
__global__ void ks_umma_prepare_kernel(uint8_t* btiles, const uint64_t* ksk, int n1, int levels, int cols, int n_blocks) {
  const int ks_total = n1 * levels / 32;
  const size_t slot = blockIdx.x * (size_t)blockDim.x + threadIdx.x;  // (nb, ks, j, kc, cg, cr)
  const size_t total = (size_t)n_blocks * ks_total * 8 * 2 * 8 * 8;
  if (slot >= total) return;
  const int cr = (int)(slot & 7), cg = (int)((slot >> 3) & 7), kc = (int)((slot >> 6) & 1), j = (int)((slot >> 7) & 7);
  const int ks = (int)((slot >> 10) % ks_total), nb = (int)((slot >> 10) / ks_total);
  const int col = nb * kKuN + cg * 8 + cr;
  uint32_t w[4] = {0, 0, 0, 0};
  if (col < cols) {
    for (int e = 0; e < 16; e++) {
      const int k = ks * 32 + kc * 16 + e, t = k / n1, i = k % n1;  // digit t <-> KSK level levels-1-t
      const uint64_t v = ksk[((size_t)i * levels + (levels - 1 - t)) * cols + col];
      w[e >> 2] |= (uint32_t)((v >> (8 * j)) & 0xFF) << (8 * (e & 3));
    }
  }
  reinterpret_cast<uint4*>(btiles)[slot] = make_uint4(w[0], w[1], w[2], w[3]);
}

__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  // K-major, no swizzle: ((8, n), 2) : ((16 B, SBO), LBO); version 1 (cute/arch/mma_sm100_desc.hpp layout)
  return (uint64_t)((addr & 0x3FFFF) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "KU_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra KU_DONE;\n\t"
      "bra KU_WAIT;\n\t"
      "KU_DONE:\n\t"
      "}" ::"r"(bar), "r"(parity) : "memory");
}

__global__ void __launch_bounds__(192, 1) keyswitch_umma_kernel(KsUBatch P) {
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* sA = smem;                                  // [stage][4096]
  unsigned char* sB = smem + kKuStages * kKuATile;           // [stage][16384]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kKuStages * (kKuATile + kKuBTile));  // full[4], empty[4], done
  uint64_t* surplus = bars + 16;                             // [64] (after 2 * stages + 1 barriers)
  __shared__ uint32_t tmem_base;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int L = P.count, chunks_per_t = P.n1 / kKtIC, total_chunks = chunks_per_t * L;
  const int ks_per_t = P.n1 / 32, ks_total = ks_per_t * L, ks_per_chunk = kKtIC / 32;
  const int kc_begin = blockIdx.z * P.chunks_per_cta, kc_end = min(kc_begin + P.chunks_per_cta, total_chunks);
  const int n_ksteps = (kc_end - kc_begin) * ks_per_chunk;
  const int b0 = blockIdx.x * kKuM, cols = P.n0 + 1;
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + kKuStages), done = smem_u32(bars + 2 * kKuStages);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&tmem_base)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) {
    for (int s = 0; s < kKuStages; s++) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(full0 + 8 * s), "r"(kKuM + 1) : "memory");  // 128 A producers + the TMA thread
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(empty0 + 8 * s) : "memory");
    }
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(done) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < kKuN) {  // (B/2) * sum of the KSK rows this CTA covers, per column
    const int col = blockIdx.y * kKuN + tid;
    uint64_t sp = 0;
    if (col < cols)
      for (int kc = kc_begin; kc < kc_end; kc++) sp += P.colsum[(size_t)kc * cols + col];
    surplus[tid] = sp << (P.radix_log - 1);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tacc = tmem_base;

  if (warp < 4) {
    // ===== A producers: thread = ciphertext row =====
    const int r = tid;
    const bool live = b0 + r < P.batch;
    const uint32_t off = (uint32_t)radix_offset(P.radix_log, L);
    const uint32_t dmask = ((1u << P.radix_log) - 1) * 0x00010001u;
    const uint16_t* row = P.st16 + (size_t)(live ? b0 + r : 0) * P.n1;
    const uint32_t a_dst = smem_u32(sA) + (r / 8) * 128 + (r % 8) * 16;
    const uint4 pad = make_uint4(off * 0x00010001u, off * 0x00010001u, off * 0x00010001u, off * 0x00010001u);
    auto load_states = [&](int it, uint4 (&w)[4]) {  // the 32 states of this row for k-step `it`
      const int kc = kc_begin + it / ks_per_chunk, c = kc / L, kk = it % ks_per_chunk;
      const uint4* src = reinterpret_cast<const uint4*>(row + c * kKtIC + kk * 32);
#pragma unroll
      for (int x = 0; x < 4; x++) w[x] = live ? __ldg(src + x) : pad;
    };
    uint4 w[4], wn[4];
    if (n_ksteps > 0) load_states(0, w);
    for (int it = 0; it < n_ksteps; it++) {
      const int kc = kc_begin + it / ks_per_chunk, t = kc % L;
      const int stage = it % kKuStages;
      if (it + 1 < n_ksteps) load_states(it + 1, wn);  // one k-step ahead: the L2 latency stays off the ring's critical path
      const int shift = P.radix_log * t;
      uint32_t o[8];
#pragma unroll
      for (int x = 0; x < 4; x++) {
        o[2 * x] = __byte_perm((w[x].x >> shift) & dmask, (w[x].y >> shift) & dmask, 0x6420);
        o[2 * x + 1] = __byte_perm((w[x].z >> shift) & dmask, (w[x].w >> shift) & dmask, 0x6420);
      }
      if (it >= kKuStages) mbar_wait(empty0 + 8 * stage, ((it / kKuStages) - 1) & 1);  // the MMAs that read this stage are done
      const uint32_t dst = a_dst + stage * kKuATile;
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst + (kKuM / 8) * 128), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(full0 + 8 * stage) : "memory");
#pragma unroll
      for (int x = 0; x < 4; x++) w[x] = wn[x];
    }
    // ===== epilogue: TMEM lane = row =====
    mbar_wait(done, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const bool split = gridDim.z > 1;
    const uint64_t* inrow = live ? (P.ptrs ? static_cast<const uint64_t*>(P.ptrs[b0 + r]) : P.in + (size_t)(b0 + r) * (P.n1 + 1)) : nullptr;
    for (int cc = 0; cc < kKuN / 8; cc++) {
      uint32_t v[8][8];
#pragma unroll
      for (int j = 0; j < 8; j++)
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(v[j][0]), "=r"(v[j][1]), "=r"(v[j][2]), "=r"(v[j][3]), "=r"(v[j][4]), "=r"(v[j][5]), "=r"(v[j][6]), "=r"(v[j][7])
                     : "r"(tacc + ((uint32_t)(warp * 32) << 16) + j * kKuN + cc * 8));
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      if (live) {
#pragma unroll
        for (int x = 0; x < 8; x++) {
          const int col = blockIdx.y * kKuN + cc * 8 + x;
          if (col < cols) {
            uint64_t sum = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) sum += (uint64_t)v[j][x] << (8 * j);
            uint64_t body = (col == P.n0 && blockIdx.z == 0) ? inrow[P.n1] : 0;
            const uint64_t val = body - (sum - surplus[cc * 8 + x]);
            uint64_t* o = P.out + (size_t)(b0 + r) * cols + col;
            if (split) atomicAdd(reinterpret_cast<unsigned long long*>(o), (unsigned long long)val);
            else *o = val;
          }
        }
      }
    }
  } else if (warp == 4) {
    // ===== B producer: one bulk copy of 16 KiB per k-step =====
    if ((tid & 31) == 0) {
      for (int it = 0; it < n_ksteps; it++) {
        const int kc = kc_begin + it / ks_per_chunk, c = kc / L, t = kc % L, kk = it % ks_per_chunk;
        const int stage = it % kKuStages;
        const size_t ksg = (size_t)t * ks_per_t + (size_t)c * ks_per_chunk + kk;
        const uint8_t* src = P.btiles + ((size_t)blockIdx.y * ks_total + ksg) * kKuBTile;
        if (it >= kKuStages) mbar_wait(empty0 + 8 * stage, ((it / kKuStages) - 1) & 1);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full0 + 8 * stage), "r"((uint32_t)kKuBTile) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(sB) + stage * kKuBTile), "l"(src), "r"((uint32_t)kKuBTile), "r"(full0 + 8 * stage) : "memory");
      }
    }
  } else {
    // ===== MMA issuer =====
    if ((tid & 31) == 0) {
      const uint32_t idesc = (2u << 4) | ((uint32_t)(kKuN >> 3) << 17) | ((uint32_t)(kKuM >> 4) << 24);  // s32 += u8 x u8, K-major
      for (int it = 0; it < n_ksteps; it++) {
        const int stage = it % kKuStages;
        mbar_wait(full0 + 8 * stage, (it / kKuStages) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint64_t da = umma_smem_desc(smem_u32(sA) + stage * kKuATile, (kKuM / 8) * 128, 128);
        const uint32_t acc = it > 0;
#pragma unroll
        for (int j = 0; j < 8; j++) {
          const uint64_t db = umma_smem_desc(smem_u32(sB) + stage * kKuBTile + j * kKuBPlane, (kKuN / 8) * 128, 128);
          asm volatile(
              "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
              "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
              ::"r"(tacc + j * kKuN), "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(empty0 + 8 * stage) : "memory");
      }
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(done) : "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tacc) : "memory");
}

// ------------------------------------------------------------------------------------------
// K7: small integer ops
// ------------------------------------------------------------------------------------------
// sample_extract (ops/ciphertext/glwe_ciphertext_ops.rs:31-76), k = 1
__global__ void sample_extract_kernel(uint64_t* out, const uint64_t* glwe, const void* const* ptrs, const uint32_t* idx,
                                      uint32_t idx_const, int batch) {
  const int c = blockIdx.y;
  if (c >= batch) return;
  const int h = idx ? (int)idx[c] : (int)idx_const;
  const uint64_t* a = ptrs ? static_cast<const uint64_t*>(ptrs[c]) : glwe + (size_t)c * 2 * kN;
  uint64_t* o = out + (size_t)c * (kN + 1);
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j <= kN; j += gridDim.x * blockDim.x) {
    if (j == kN) o[j] = a[kN + h];
    else o[j] = j <= h ? a[h - j] : 0 - a[h + kN - j];
  }
}

// op 0: out = a + b (xor, evaluation.rs:53-55); op 1: out = a + trivial_one (not, :48-50);
// op 2: out = a * X^n (mul_xn, :58-65)
__global__ void glwe_elementwise_kernel(uint64_t* out, const uint64_t* a, const uint64_t* b, const void* const* ptrs,
                                        const uint32_t* nvec, int op, uint32_t n, size_t batch) {
  const size_t total = batch * 2 * kN;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const size_t c = e / (2 * kN);
    const int r = (int)(e % (2 * kN)) / kN, j = (int)(e % kN);
    const uint64_t* pa = (ptrs ? static_cast<const uint64_t*>(ptrs[2 * c]) : a + c * 2 * kN) + r * kN;
    uint64_t v;
    if (op == 0) v = pa[j] + (ptrs ? static_cast<const uint64_t*>(ptrs[2 * c + 1])[r * kN + j] : b[e]);
    else if (op == 1) v = pa[j] + ((r == 1 && j == 0) ? (1ull << 63) : 0ull);
    else v = rotated_coeff(pa, j, (int)((nvec ? nvec[c] : n) & (2 * kN - 1)));
    out[e] = v;
  }
}

// ------------------------------------------------------------------------------------------
// K8: RLWE public-key encryption, the "double-LWE trick" of rlwe_encrypt_public_impl
// (ops/encryption/rlwe_encryption.rs:125-160; Encryption::encrypt_rlwe_l1 / encrypt_rlev_l1,
// parasol_runtime/src/crypto/encryption.rs:205-249), with the randomness (u, e0, e1) supplied by the caller:
//   ct = (p0 * u + e0, p1 * u + e1 + m)   over Z_2^64[X]/(X^N + 1), k = 1
// Both products are the EXACT negacyclic ones of polynomial_external_mad (integer work, bit-exact against the oracle),
// for any u64 multiplier -- not only the binary u the reference samples.  One CTA per ciphertext, 256 threads.
// Shared memory: the public key with the negacyclic sign folded in, pe[p][i] = p[i], pe[p][i + N] = -p[i]
// (so (p * u)[k] = sum_i u[i] * pe[(k - i) mod 2N], no sign logic in the loop), and u.  Thread t owns the outputs
// k = t + 256 kk, kk = 0..7, and walks the multiplier in groups i = ib + 256 ii, ii = 0..7: then
// k - i = (t - ib) + 256 (kk - ii) -- the 64 products of a group need only 15 key values per polynomial, 256 apart,
// and consecutive threads read consecutive addresses (conflict-free): 38 shared loads per 128 multiply-adds.
constexpr int kRlweThreads = 256;
constexpr int kRlweSmem = (2 * 2 * kN + kN) * 8;  // 81920
struct RlweBatch {
  uint64_t* out;        // [B][2][N]
  const uint64_t* pk;   // [2][N], shared by the batch
  const uint64_t* msg;  // [B][N] encoded message (torus)
  const uint64_t* u;    // [B][N]
  const uint64_t* e0;   // [B][N]
  const uint64_t* e1;   // [B][N]
  int batch;
};
__global__ void __launch_bounds__(kRlweThreads, 2) rlwe_encrypt_public_kernel(RlweBatch P) {
  extern __shared__ __align__(16) unsigned char smem[];
  uint64_t* pe = reinterpret_cast<uint64_t*>(smem);  // [2][2N]
  uint64_t* su = pe + 2 * 2 * kN;                    // [N]
  const int t = threadIdx.x;
  for (int i = t; i < 2 * kN; i += kRlweThreads) {
    const uint64_t v = P.pk[i];
    const int p = i / kN, j = i % kN;
    pe[p * 2 * kN + j] = v;
    pe[p * 2 * kN + kN + j] = 0 - v;
  }
  for (int c = blockIdx.x; c < P.batch; c += gridDim.x) {
    __syncthreads();  // the previous ciphertext's reads of su are done (and pe is complete)
    for (int i = t; i < kN; i += kRlweThreads) su[i] = P.u[(size_t)c * kN + i];
    __syncthreads();
    uint64_t acc[2][8];
#pragma unroll
    for (int p = 0; p < 2; p++)
#pragma unroll
      for (int kk = 0; kk < 8; kk++) acc[p][kk] = 0;
#pragma unroll 1
    for (int ib = 0; ib < 256; ib++) {
      uint64_t uu[8], w0[15], w1[15];
#pragma unroll
      for (int ii = 0; ii < 8; ii++) uu[ii] = su[ib + 256 * ii];
      const int base = t - ib;  // in (-256, 256)
#pragma unroll
      for (int d = 0; d < 15; d++) {
        const int idx = (base + 256 * (d - 7)) & (2 * kN - 1);
        w0[d] = pe[idx];
        w1[d] = pe[2 * kN + idx];
      }
#pragma unroll
      for (int kk = 0; kk < 8; kk++)
#pragma unroll
        for (int ii = 0; ii < 8; ii++) {
          acc[0][kk] += w0[kk - ii + 7] * uu[ii];
          acc[1][kk] += w1[kk - ii + 7] * uu[ii];
        }
    }
    uint64_t* o = P.out + (size_t)c * 2 * kN;
#pragma unroll
    for (int kk = 0; kk < 8; kk++) {
      const int k = t + 256 * kk;
      const size_t e = (size_t)c * kN + k;
      o[k] = acc[0][kk] + P.e0[e];
      o[kN + k] = acc[1][kk] + P.e1[e] + P.msg[e];
    }
  }
}

// one thread waits `ns` nanoseconds (capi.cu::launch_cbs: lets a concurrently submitted kernel be seated first)
__global__ void pause_kernel(unsigned ns) {
  unsigned long long t0, t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  do { asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); } while (t - t0 < ns);
}

// FFT-domain polynomials: dst = src * scale (2^-10 to import reference-scale data, 2^10 to export)
__global__ void fft_scale_kernel(C2* dst, const C2* src, size_t n, double scale) {
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const C2 x = src[e];
    dst[e] = C2{x.x * scale, x.y * scale};
  }
}

// FP64 peak probe: dependent-free DFMA chains on every SM (SURVEY 8(d): MEASURED_PEAKS.json has
// no FP64 figure, the builder measures one).
__global__ void dfma_probe_kernel(double* out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
         a7 = a0 + 7;
  const double m = 1.0000000001, c = 1e-12;
  for (int i = 0; i < iters; i++) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

}  // namespace spf
