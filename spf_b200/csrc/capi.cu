// capi.cu -- C ABI of libspf_b200.so (include/spf_b200.h): context, key upload, batched ops.
// No CPU fallback anywhere: every op launches the sm_100a kernels of kernels.cuh or fails.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_set>
#include <vector>

#include "../../include/spf_b200.h"
#include "kernels.cuh"
#include "tables.h"

using namespace spf;

namespace {

thread_local std::string g_create_err;

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
};

}  // namespace

struct spf_b200_ctx {
  int device = 0;
  spf_params p{};
  C2 *bsk = nullptr, *ak = nullptr, *ssk = nullptr;
  uint64_t* ksk = nullptr;
  uint64_t* ksk_colsum = nullptr;  // keyswitch_kernel's per-block column sums of the KSK
  uint64_t* ks_tc_colsum = nullptr;  // keyswitch_umma_kernel: per-(chunk, level) column sums
  uint8_t* ks_btiles = nullptr;      // keyswitch_umma_kernel: KSK byte planes as canonical K-major UMMA tiles (nullptr: shape unsupported)
  C2 *T1 = nullptr, *T2 = nullptr;
  uint32_t* kinv = nullptr;
  cudaStream_t stream[2] = {nullptr, nullptr};
  cudaEvent_t ev[2] = {nullptr, nullptr};
  cudaEvent_t ev_copied[2] = {nullptr, nullptr};  // host-pointer CBS pipeline: staging buffer of a slot is free again
  cudaStream_t aux = nullptr;                      // launch_cbs: the partial last wave of the blind rotation (high priority)
  cudaEvent_t ev_cbs_main = nullptr, ev_cbs_tail = nullptr;
  DevBuf scratch[2][7];  // per pipeline slot: grow-only device scratch ([6]: keyswitch digit states)
  std::string err;
  std::atomic<uint64_t> launches{0};
  int sm_count = 148;
  // lifetime: graphs built on this context keep it alive (spf_b200_destroy only drops the owner's reference)
  std::atomic<int> refs{1};
  // flow control of the asynchronous executor (graph.cuh: spf_b200_graph_spawn): at most max_in_flight spawned graphs
  // between dispatch and completion, as the bounded channel of CircuitProcessor::new (circuit_processor/mod.rs:95-123)
  std::mutex fc_mu;
  std::condition_variable fc_cv;
  int in_flight = 0, max_in_flight = 4;
  // device constants for the graph executor's Zero*/One* nodes (graph.cuh::ensure_constants)
  void* consts = nullptr;
  char *c_lwe0[2] = {nullptr, nullptr}, *c_glwe[2] = {nullptr, nullptr}, *c_glev[2] = {nullptr, nullptr},
       *c_ggsw[2] = {nullptr, nullptr};
};

namespace {

#define CU(call)                                                                            \
  do {                                                                                      \
    cudaError_t e_ = (call);                                                                \
    if (e_ != cudaSuccess) {                                                                \
      return fail(ctx, SPF_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));     \
    }                                                                                       \
  } while (0)

int fail(spf_b200_ctx* ctx, int code, const std::string& msg) {
  if (ctx) ctx->err = msg;
  else g_create_err = msg;
  return code;
}

size_t len_glwe(const spf_params* p) { return (size_t)(p->glwe_k + 1) * p->glwe_n; }
size_t len_ggsw(const spf_params* p, spf_radix r) { return len_glwe(p) * r.count * (p->glwe_k + 1) / 2; }
uint32_t ilog2u(uint32_t x) { uint32_t l = 0; while ((1u << (l + 1)) <= x) l++; return l; }
uint32_t cbs_log_v(const spf_params* p) {
  uint32_t lv = ilog2u(p->cbs.count);
  if ((1u << lv) != p->cbs.count) lv++;
  return lv;
}

int ensure(spf_b200_ctx* ctx, DevBuf& b, size_t bytes) {
  if (b.cap >= bytes) return 0;
  if (b.p) CU(cudaFree(b.p));
  b.p = nullptr; b.cap = 0;
  CU(cudaMalloc(&b.p, bytes));
  b.cap = bytes;
  return 0;
}

DevTables tabs(const spf_b200_ctx* ctx) { return DevTables{ctx->T1, ctx->T2}; }
cudaStream_t pick(spf_b200_ctx* ctx, void* stream) { return stream ? (cudaStream_t)stream : ctx->stream[0]; }

int check_launch(spf_b200_ctx* ctx, const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(ctx, SPF_E_CUDA, std::string(what) + " launch: " + cudaGetErrorString(e));
  ctx->launches.fetch_add(1);
  return 0;
}

// The sm_100a kernels are specialised for the shapes of DEFAULT_128 (SURVEY.md section 5:
// "specialised for DEFAULT_128 but must read sizes from Params"); radix parameters other than
// pbs_radix are runtime values.
int validate_params(const spf_params* p) {
  if (!p) return fail(nullptr, SPF_E_INVALID, "params is NULL");
  if (p->glwe_n != (uint32_t)kN || p->glwe_k != 1)
    return fail(nullptr, SPF_E_UNSUPPORTED, "kernels are specialised for l1_params = GLWE_1_2048 (k=1, N=2048)");
  if (p->pbs.radix_log != 16 || p->pbs.count != 2)
    return fail(nullptr, SPF_E_UNSUPPORTED, "blind-rotation kernel is specialised for pbs_radix = (log 16, count 2)");
  if (p->lwe_n == 0 || p->lwe_n > 4096) return fail(nullptr, SPF_E_INVALID, "l0 dimension out of range");
  const spf_radix rs[4] = {p->cbs, p->ks, p->ss, p->tr};
  for (const spf_radix& r : rs) {
    if (r.radix_log == 0 || r.count == 0 || r.radix_log * r.count >= 64 || r.radix_log > 30)
      return fail(nullptr, SPF_E_INVALID, "invalid radix decomposition");
  }
  if (p->ks.radix_log * p->ks.count > 32) return fail(nullptr, SPF_E_UNSUPPORTED, "ks_radix needs log*count <= 32");
  if (p->cbs.count >= 8) return fail(nullptr, SPF_E_INVALID, "cbs_radix.count must be < 8 (circuit_bootstrapping.rs:399)");
  if (p->cbs.radix_log * p->cbs.count + 1 >= 64) return fail(nullptr, SPF_E_INVALID, "cbs_radix too wide");
  return 0;
}

// Work items per CTA: the full complement when the batch fills the GPU, fewer for small batches
// so that every item gets an SM (and its shared-memory / FP64 pipes) to itself.
int per_cta(const spf_b200_ctx* ctx, size_t items, int max_per_cta) {
  int per = max_per_cta;
  while (per > 1 && items <= (size_t)ctx->sm_count * (per - 1)) per--;
  return per;
}

int launch_scale(spf_b200_ctx* ctx, C2* dst, const C2* src, size_t n, double scale, cudaStream_t s) {
  if (n == 0) return 0;
  const int threads = 256;
  const int blocks = (int)std::min<size_t>((n + threads - 1) / threads, (size_t)ctx->sm_count * 16);
  fft_scale_kernel<<<blocks, threads, 0, s>>>(dst, src, n, scale);
  return check_launch(ctx, "fft_scale_kernel");
}

int create_common(const spf_params* params, const double* bsk, size_t bsk_len, const uint64_t* ksk, size_t ksk_len,
                  const double* ssk, size_t ssk_len, const double* ak, size_t ak_len, int device, bool on_device,
                  spf_b200_ctx** out) {
  if (!out) return fail(nullptr, SPF_E_INVALID, "out is NULL");
  *out = nullptr;
  if (int rc = validate_params(params)) return rc;
  if (!bsk || !ksk || !ssk || !ak) return fail(nullptr, SPF_E_INVALID, "NULL key array");
  if (bsk_len != spf_b200_len_bsk(params) || ksk_len != spf_b200_len_ksk(params) ||
      ssk_len != spf_b200_len_ssk(params) || ak_len != spf_b200_len_ak(params))
    return fail(nullptr, SPF_E_INVALID, "key length does not match params (ComputeKey::check_is_valid, keys.rs:190-206)");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, SPF_E_CUDA, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(nullptr, SPF_E_INVALID, "device index out of range");
  spf_b200_ctx* ctx = new spf_b200_ctx();
  ctx->device = device;
  ctx->p = *params;
  auto bail = [&](int rc) { g_create_err = ctx->err; spf_b200_destroy(ctx); return rc; };
#define CUB(call)                                                                        \
  do {                                                                                   \
    cudaError_t e_ = (call);                                                             \
    if (e_ != cudaSuccess) {                                                             \
      ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                     \
      return bail(SPF_E_CUDA);                                                           \
    }                                                                                    \
  } while (0)
  CUB(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUB(cudaGetDeviceProperties(&prop, device));
  ctx->sm_count = prop.multiProcessorCount;
  if (prop.major < 10) { ctx->err = "spf_b200 requires an sm_100a (Blackwell) GPU"; return bail(SPF_E_UNSUPPORTED); }
  for (int i = 0; i < 2; i++) {
    CUB(cudaStreamCreateWithFlags(&ctx->stream[i], cudaStreamNonBlocking));
    CUB(cudaEventCreateWithFlags(&ctx->ev[i], cudaEventDisableTiming));
    CUB(cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming));
  }
  {
    int lo = 0, hi = 0;
    CUB(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    CUB(cudaStreamCreateWithPriority(&ctx->aux, cudaStreamNonBlocking, hi));
    CUB(cudaEventCreateWithFlags(&ctx->ev_cbs_main, cudaEventDisableTiming));
    CUB(cudaEventCreateWithFlags(&ctx->ev_cbs_tail, cudaEventDisableTiming));
  }
  CUB(cudaFuncSetAttribute(pbs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPbsSmem));
  CUB(cudaFuncSetAttribute(pbs_quad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kQuadSmem));
  CUB(cudaFuncSetAttribute(trace_ss_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTrSmem));
  CUB(cudaFuncSetAttribute(trace_ss_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTrSmem));
  CUB(cudaFuncSetAttribute(cmux_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCmuxSmem));
  CUB(cudaFuncSetAttribute(cmux_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kWideSmem));
  {
    const int ks_smem = kKsBatch * (int)(params->glwe_k * params->glwe_n + kKsBlock) * 4;
    switch (params->ks.count) {
#define SPF_KS_CASE(L) case L: CUB(cudaFuncSetAttribute(keyswitch_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, ks_smem)); break;
      SPF_KS_CASE(1) SPF_KS_CASE(2) SPF_KS_CASE(3) SPF_KS_CASE(4) SPF_KS_CASE(5) SPF_KS_CASE(6) SPF_KS_CASE(7) SPF_KS_CASE(8)
#undef SPF_KS_CASE
      default: break;
    }
  }
  // constant tables
  {
    std::vector<C2> T1(kT1Elems), T2(kT2Elems);
    fill_twiddle_tables(T1.data(), T2.data());
    uint32_t kinv[11];
    fill_kinv(kinv);
    CUB(cudaMalloc(&ctx->T1, sizeof(C2) * kT1Elems));
    CUB(cudaMalloc(&ctx->T2, sizeof(C2) * kT2Elems));
    CUB(cudaMalloc(&ctx->kinv, sizeof(kinv)));
    CUB(cudaMemcpy(ctx->T1, T1.data(), sizeof(C2) * kT1Elems, cudaMemcpyHostToDevice));
    CUB(cudaMemcpy(ctx->T2, T2.data(), sizeof(C2) * kT2Elems, cudaMemcpyHostToDevice));
    CUB(cudaMemcpy(ctx->kinv, kinv, sizeof(kinv), cudaMemcpyHostToDevice));
  }
  // keys: FFT-domain keys are rescaled by 2^-10 in place on the device (exact)
  const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  CUB(cudaMalloc(&ctx->bsk, sizeof(C2) * bsk_len));
  CUB(cudaMalloc(&ctx->ssk, sizeof(C2) * ssk_len));
  CUB(cudaMalloc(&ctx->ak, sizeof(C2) * ak_len));
  CUB(cudaMalloc(&ctx->ksk, sizeof(uint64_t) * ksk_len));
  CUB(cudaMemcpyAsync(ctx->bsk, bsk, sizeof(C2) * bsk_len, kind, ctx->stream[0]));
  CUB(cudaMemcpyAsync(ctx->ssk, ssk, sizeof(C2) * ssk_len, kind, ctx->stream[0]));
  CUB(cudaMemcpyAsync(ctx->ak, ak, sizeof(C2) * ak_len, kind, ctx->stream[0]));
  CUB(cudaMemcpyAsync(ctx->ksk, ksk, sizeof(uint64_t) * ksk_len, kind, ctx->stream[0]));
  if (launch_scale(ctx, ctx->bsk, ctx->bsk, bsk_len, 1.0 / 1024.0, ctx->stream[0]) ||
      launch_scale(ctx, ctx->ssk, ctx->ssk, ssk_len, 1.0 / 1024.0, ctx->stream[0]) ||
      launch_scale(ctx, ctx->ak, ctx->ak, ak_len, 1.0 / 1024.0, ctx->stream[0]))
    return bail(SPF_E_CUDA);
  {  // per-block column sums of the KSK for the unsigned-digit keyswitch (kernels.cuh K4)
    const int n1 = (int)(params->glwe_k * params->glwe_n), cols = (int)params->lwe_n + 1;
    const int nblk = (n1 + kKsBlock - 1) / kKsBlock;
    CUB(cudaMalloc(&ctx->ksk_colsum, sizeof(uint64_t) * (size_t)nblk * cols));
    ksk_colsum_kernel<<<dim3((cols + 127) / 128, nblk), 128, 0, ctx->stream[0]>>>(ctx->ksk_colsum, ctx->ksk, n1,
                                                                                   (int)params->ks.count, cols);
    CUB(cudaGetLastError());
    // tensor-core keyswitch (kernels.cuh K4u): per-chunk column sums + the KSK byte planes as UMMA tiles
    const int L = (int)params->ks.count, lb = (int)params->ks.radix_log;
    // byte-plane GEMMs accumulate in s32: (B - 1) * 255 per term, n1 * L terms
    const bool s32_ok = (uint64_t)n1 * L * ((1u << lb) - 1) * 255ull < (1ull << 31);
    if (n1 % kKtIC == 0 && L * lb + 1 <= 16 && lb <= 8 && s32_ok) {
      const int ks_total = n1 * L / 32, chunks = n1 / kKtIC * L;
      CUB(cudaMalloc(&ctx->ks_tc_colsum, sizeof(uint64_t) * (size_t)chunks * cols));
      ks_tc_colsum_kernel<<<dim3((cols + 127) / 128, chunks), 128, 0, ctx->stream[0]>>>(ctx->ks_tc_colsum, ctx->ksk, n1, L, cols);
      CUB(cudaGetLastError());
      // the KSK byte planes as canonical K-major UMMA tiles, 16 KiB per (column block, k-step)
      const int n_blocks = (cols + kKuN - 1) / kKuN;
      const size_t tile_bytes = (size_t)n_blocks * ks_total * kKuBTile;
      CUB(cudaMalloc(&ctx->ks_btiles, tile_bytes));
      ks_umma_prepare_kernel<<<(unsigned)((tile_bytes / 16 + 255) / 256), 256, 0, ctx->stream[0]>>>(ctx->ks_btiles, ctx->ksk, n1, L, cols, n_blocks);
      CUB(cudaGetLastError());
      CUB(cudaFuncSetAttribute(keyswitch_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kKuSmem));
    }
  }
  CUB(cudaStreamSynchronize(ctx->stream[0]));
#undef CUB
  *out = ctx;
  return 0;
}

// ---- kernel launch helpers (device pointers) ---------------------------------------------

int launch_pbs(spf_b200_ctx* ctx, uint64_t* d_glwe_out, const uint64_t* d_lwe_in, const uint64_t* d_lut, bool cbs,
               uint32_t log_chi, uint32_t log_v, size_t batch, cudaStream_t s, const void* const* ptrs = nullptr,
               bool packed = false) {
  if (batch == 0) return 0;
  PbsBatch P;
  P.lwe_in = d_lwe_in;
  P.lut = cbs ? nullptr : d_lut;
  P.lut_stride = 0;
  P.glwe_out = d_glwe_out;
  P.bsk = ctx->bsk;
  P.ptrs = ptrs;
  P.batch = (int)batch;
  P.lwe_n = (int)ctx->p.lwe_n;
  P.log_chi = (int)log_chi;
  P.log_v = (int)log_v;
  P.cbs_radix_log = (int)ctx->p.cbs.radix_log;
  P.cbs_count = (int)ctx->p.cbs.count;
  // A pair (one ciphertext) is largely latency-bound: alone on an SM it takes ~7 ms per PBS, ~9 ms
  // when three share the SM; small batches get one ciphertext per SM so they do not queue behind
  // each other, large ones run as persistent pairs (see pbs_kernel).
  if (packed) {  // launch_cbs: kPbsPairs ciphertexts per SM on as few SMs as possible, the rest of the GPU is busy elsewhere
    const int grid = (int)std::min<size_t>((batch + kPbsPairs - 1) / kPbsPairs, (size_t)ctx->sm_count);
    pbs_kernel<<<grid, kPbsPairs * 2 * kTeam, kPbsSmem, s>>>(P, tabs(ctx));
    return check_launch(ctx, "pbs_kernel");
  }
  if (batch <= (size_t)ctx->sm_count) {  // latency mode: one ciphertext per SM on four teams
    pbs_quad_kernel<<<(int)batch, 4 * kTeam, kQuadSmem, s>>>(P, tabs(ctx));
    return check_launch(ctx, "pbs_quad_kernel");
  }
  // Tail wave: a batch is a whole number of waves (sm_count x kPbsPairs ciphertexts) plus a remainder.  A remainder of
  // at most one ciphertext per SM would run as one pair per SM after everything else has finished (5.1 ms for e.g. the
  // last 100 of 4096 ciphertexts); the four-team latency kernel does the same work in 3.5 ms, so the remainder goes
  // there (same stream, right behind the full waves).
  const size_t wave = (size_t)ctx->sm_count * kPbsPairs;
  const size_t rem = batch % wave;
  if (batch > wave && rem > 0 && rem <= (size_t)ctx->sm_count && !P.lut_stride) {
    const size_t full = batch - rem;
    P.batch = (int)full;
    pbs_kernel<<<ctx->sm_count, kPbsPairs * 2 * kTeam, kPbsSmem, s>>>(P, tabs(ctx));
    if (int rc = check_launch(ctx, "pbs_kernel")) return rc;
    PbsBatch T = P;
    T.batch = (int)rem;
    T.glwe_out = d_glwe_out + full * 2 * kN;
    if (ptrs) T.ptrs = ptrs + full;
    else T.lwe_in = d_lwe_in + full * (size_t)(P.lwe_n + 1);
    pbs_quad_kernel<<<(int)rem, 4 * kTeam, kQuadSmem, s>>>(T, tabs(ctx));
    return check_launch(ctx, "pbs_quad_kernel");
  }
  const int per = per_cta(ctx, batch, kPbsPairs);
  const int grid = (int)std::min<size_t>((batch + per - 1) / per, (size_t)ctx->sm_count);  // persistent pairs
  pbs_kernel<<<grid, per * 2 * kTeam, kPbsSmem, s>>>(P, tabs(ctx));
  return check_launch(ctx, "pbs_kernel");
}

int launch_trace_ss(spf_b200_ctx* ctx, const uint64_t* d_glwe_in, uint64_t* d_glev_out, C2* d_ggsw_out, int mode,
                    int levels, double out_scale, size_t batch, cudaStream_t s, const void* const* ptrs = nullptr,
                    const PeerOffsets* peers = nullptr) {
  if (batch == 0) return 0;
  TraceSsBatch P;
  if (peers) P.peers = *peers;
  else P.peers.n = 0;
  P.glwe_in = d_glwe_in;
  P.glev_out = d_glev_out;
  P.ggsw_out = d_ggsw_out;
  P.ak = ctx->ak;
  P.ssk = ctx->ssk;
  P.kinv = ctx->kinv;
  P.ptrs = ptrs;
  P.batch = (int)batch;
  P.levels = levels;
  P.mode = mode;
  P.cbs_radix_log = (int)ctx->p.cbs.radix_log;
  P.cbs_count = (int)ctx->p.cbs.count;
  P.tr_radix_log = (int)ctx->p.tr.radix_log;
  P.tr_count = (int)ctx->p.tr.count;
  P.ss_radix_log = (int)ctx->p.ss.radix_log;
  P.ss_count = (int)ctx->p.ss.count;
  P.out_scale = out_scale;
  const size_t items = batch * (size_t)levels;
  const int per = per_cta(ctx, items, kTrTeams);
  const int grid = (int)((items + per - 1) / per);
  if (P.peers.n > 0) trace_ss_kernel<true><<<grid, per * kTeam, kTableBytes + per * kTrTeamBytes, s>>>(P, tabs(ctx));
  else trace_ss_kernel<false><<<grid, per * kTeam, kTableBytes + per * kTrTeamBytes, s>>>(P, tabs(ctx));
  return check_launch(ctx, "trace_ss_kernel");
}

// Circuit bootstrap = blind rotation (pbs_kernel) then trace + scheme switch (trace_ss_kernel) per ciphertext.
// The blind rotation runs in waves of sm_count x kPbsPairs ciphertexts; a batch such as 4096 = 9 x 444 + 100 ends in a
// remainder that cannot fill the GPU.  Run alone, that remainder costs a whole extra pass of the latency kernel
// (3.5 ms for 100 ciphertexts on 100 SMs while 48 idle, then 8.7 ms of trace kernels).  Here it is packed three to an SM
// onto ceil(rem / 3) SMs (the throughput configuration: 2.4 instead of 3.5 SM-ms per ciphertext) on a high-priority
// side stream and runs CONCURRENTLY with the trace / scheme-switch kernel of the full waves, whose thousands of short
// CTAs fill the remaining SMs: the step ends after (all work) / (all SMs) instead of after the sum of three under-filled
// phases.  Only scheduling depends on the first event (the remainder reads nothing the full waves write); the second one
// orders the remainder's trace kernel behind its blind rotation.
int launch_cbs(spf_b200_ctx* ctx, C2* d_ggsw_out, uint64_t* d_glwe, const uint64_t* d_lwe_in, const void* const* ptrs,
               double out_scale, size_t batch, cudaStream_t s, const PeerOffsets* peers = nullptr) {
  if (batch == 0) return 0;
  const int levels = (int)ctx->p.cbs.count;
  const size_t wave = (size_t)ctx->sm_count * kPbsPairs, rem = batch % wave, full = batch - rem;
  const size_t lwe = (size_t)ctx->p.lwe_n + 1, ggsw = len_ggsw(&ctx->p, ctx->p.cbs);
  // Worth it only when the trace kernels of the full waves can keep the other SMs busy for the remainder's whole round;
  // otherwise the packed remainder (one round, R) becomes the critical path and the latency kernel (0.49 R) followed by
  // the trace kernels is shorter.  Measured ratios: trace + scheme switch of one ciphertext = 2.93e-4 R of the whole GPU.
  bool pays = false;
  if (full > 0 && rem > 0 && rem <= wave / 2) {
    const double c = 2.93e-4, sm = (double)ctx->sm_count;
    const double serial = (rem <= (size_t)ctx->sm_count ? 0.49 : 1.0) + (double)batch * c;
    const double tail_sms = (double)((rem + kPbsPairs - 1) / kPbsPairs);
    const double packed = std::max(1.0, ((double)full * c * sm + tail_sms) / sm) + (double)rem * c;
    pays = packed < serial;
  }
  if (!pays || s == ctx->aux) {
    if (int rc = launch_pbs(ctx, d_glwe, d_lwe_in, nullptr, true, 0, cbs_log_v(&ctx->p), batch, s, ptrs)) return rc;
    return launch_trace_ss(ctx, d_glwe, nullptr, d_ggsw_out, 0, levels, out_scale, batch, s, nullptr, peers);
  }
  if (int rc = launch_pbs(ctx, d_glwe, d_lwe_in, nullptr, true, 0, cbs_log_v(&ctx->p), full, s, ptrs)) return rc;
  CU(cudaEventRecord(ctx->ev_cbs_main, s));
  CU(cudaStreamWaitEvent(ctx->aux, ctx->ev_cbs_main, 0));
  if (int rc = launch_pbs(ctx, d_glwe + full * 2 * kN, ptrs ? nullptr : d_lwe_in + full * lwe, nullptr, true, 0, cbs_log_v(&ctx->p), rem,
                          ctx->aux, ptrs ? ptrs + full : nullptr, /*packed=*/true))
    return rc;
  CU(cudaEventRecord(ctx->ev_cbs_tail, ctx->aux));
  // Both successors of the full waves become runnable at the same instant.  The remainder's few long CTAs must be placed
  // first: if the trace kernel's 4 000 CTAs take every SM, the remainder trickles in behind them and the step gets LONGER
  // than the serial form (seen on one box in four: 77.3 instead of 75.7 ms; stream priority alone did not prevent it).
  // A 20 us single-thread pause in front of the trace kernel gives the block scheduler time to seat the remainder.
  pause_kernel<<<1, 1, 0, s>>>(20000u);
  if (int rc = check_launch(ctx, "pause_kernel")) return rc;
  if (int rc = launch_trace_ss(ctx, d_glwe, nullptr, d_ggsw_out, 0, levels, out_scale, full, s, nullptr, peers)) return rc;
  CU(cudaStreamWaitEvent(s, ctx->ev_cbs_tail, 0));
  return launch_trace_ss(ctx, d_glwe + full * 2 * kN, nullptr, d_ggsw_out + full * ggsw, 0, levels, out_scale, rem, s, nullptr, peers);
}

int launch_cmux(spf_b200_ctx* ctx, uint64_t* d_out, const uint64_t* d_d0, const uint64_t* d_d1, const C2* d_ggsw,
                size_t ggsw_stride, int glwe_per_item, size_t n_glwe, cudaStream_t s, const void* const* ptrs = nullptr,
                void* const* out_ptrs = nullptr) {
  if (n_glwe == 0) return 0;
  CmuxBatch P;
  P.out_ptrs = out_ptrs;
  P.out = d_out;
  P.d0 = d_d0;
  P.d1 = d_d1;
  P.ggsw = d_ggsw;
  P.ggsw_stride = ggsw_stride;
  P.ptrs = ptrs;
  P.batch = (int)n_glwe;
  P.glwe_per_item = glwe_per_item;
  P.radix_log = (int)ctx->p.cbs.radix_log;
  P.count = (int)ctx->p.cbs.count;
  // few outputs (a level of a MUX tree): one CTA of 8 teams per output, 3-5x lower latency
  // Programmatic dependent launch: consecutive levels of a MUX tree are back-to-back CMUX kernels; each
  // loads its tables (and prefetches its selector) while the previous level drains (kernels.cuh, pdl_wait).
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.stream = s;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  const DevTables T = tabs(ctx);
  // two waves of the wide kernel still beat one team per output (cold L2: 49 vs 59 us at 296 outputs; 4 x mul32 in one
  // graph 45.2 -> 42.2 ms); from three waves on the throughput kernel wins (profiles/r1_w_cmux_kernel_choice.json)
  const size_t wide_max = 2 * (size_t)ctx->sm_count;
  if (n_glwe <= wide_max && P.count == 4) {
    cfg.gridDim = dim3((unsigned)n_glwe);
    cfg.blockDim = dim3(kWideTeams * kTeam);
    cfg.dynamicSmemBytes = kWideSmem;
    cudaLaunchKernelEx(&cfg, cmux_wide_kernel, P, T);
    return check_launch(ctx, "cmux_wide_kernel");
  }
  const int per = per_cta(ctx, n_glwe, kCmuxTeams);
  cfg.gridDim = dim3((unsigned)((n_glwe + per - 1) / per));
  cfg.blockDim = dim3(per * kTeam);
  cfg.dynamicSmemBytes = kTableBytes + per * kCmuxTeamBytes;
  cudaLaunchKernelEx(&cfg, cmux_kernel, P, T);
  return check_launch(ctx, "cmux_kernel");
}

int launch_keyswitch(spf_b200_ctx* ctx, uint64_t* d_out, const uint64_t* d_in, size_t batch, cudaStream_t s,
                     const void* const* ptrs = nullptr, DevBuf* states = nullptr /* caller-owned digit-state scratch */) {
  if (batch == 0) return 0;
  KsBatch P;
  P.out = d_out;
  P.in = d_in;
  P.ksk = ctx->ksk;
  P.colsum = ctx->ksk_colsum;
  P.ptrs = ptrs;
  P.batch = (int)batch;
  P.n1 = (int)(ctx->p.glwe_k * ctx->p.glwe_n);
  P.n0 = (int)ctx->p.lwe_n;
  P.radix_log = (int)ctx->p.ks.radix_log;
  P.count = (int)ctx->p.ks.count;
  static const bool ks_no_tc = getenv("SPF_B200_KS_NO_TC") != nullptr;  // read once, not per launch
  if (ctx->ks_btiles && !ks_no_tc) {  // dense contraction on the int8 tensor cores (K4u)
    DevBuf& st16 = states ? *states : ctx->scratch[s == ctx->stream[1] ? 1 : 0][6];
    if (int rc = ensure(ctx, st16, batch * (size_t)P.n1 * 2)) return rc;
    ks_tc_states_kernel<<<std::min<int>((int)((batch * (size_t)P.n1 + 255) / 256), ctx->sm_count * 8), 256, 0, s>>>(
        (uint16_t*)st16.p, d_in, ptrs, P.batch, P.n1, P.radix_log, P.count);
    if (int rc = check_launch(ctx, "ks_tc_states_kernel")) return rc;
    KsUBatch U;
    U.out = d_out; U.in = d_in; U.ptrs = ptrs; U.st16 = (const uint16_t*)st16.p; U.btiles = ctx->ks_btiles; U.colsum = ctx->ks_tc_colsum;
    U.batch = P.batch; U.n1 = P.n1; U.n0 = P.n0; U.radix_log = P.radix_log; U.count = P.count;
    const int ux = (int)((batch + kKuM - 1) / kKuM), uy = (P.n0 + 1 + kKuN - 1) / kKuN;
    const int chunks = P.n1 / kKtIC * P.count;
    int z = std::max(1, std::min(chunks, (ctx->sm_count + ux * uy - 1) / (ux * uy)));  // split K until every SM has a CTA
    U.chunks_per_cta = (chunks + z - 1) / z;
    z = (chunks + U.chunks_per_cta - 1) / U.chunks_per_cta;
    if (z > 1) CU(cudaMemsetAsync(d_out, 0, batch * (size_t)(P.n0 + 1) * 8, s));
    keyswitch_umma_kernel<<<dim3(ux, uy, z), 192, kKuSmem, s>>>(U);
    return check_launch(ctx, "keyswitch_umma_kernel");
  }
  if (P.n0 + 1 > 2 * kKsThreads) return fail(ctx, SPF_E_UNSUPPORTED, "l0 dimension too large for the keyswitch kernel");
  if (P.count > kKsMaxLevels) return fail(ctx, SPF_E_UNSUPPORTED, "ks_radix.count too large for the keyswitch kernel");
  const int tiles = (int)((batch + kKsBatch - 1) / kKsBatch);
  // split the sweep over the n1 mask elements so that at least ~2 CTAs per SM are in flight even
  // for small batches (a single CTA streaming the whole 62.7 MB KSK is latency-bound)
  int splits = 1;
  while (tiles * splits < 2 * ctx->sm_count && splits < 64 && (P.n1 / (splits * 2)) >= kKsBlock) splits *= 2;
  P.slice = ((P.n1 + splits - 1) / splits + kKsBlock - 1) / kKsBlock * kKsBlock;  // whole column-sum blocks
  splits = (P.n1 + P.slice - 1) / P.slice;
  if (splits > 1) CU(cudaMemsetAsync(d_out, 0, batch * (size_t)(P.n0 + 1) * 8, s));
  dim3 grid(tiles, splits);
  const size_t smem = (size_t)kKsBatch * P.slice * 4;
  switch (P.count) {  // the level count is a template parameter (fully unrolled digit loop)
#define SPF_KS_CASE(L) case L: keyswitch_kernel<L><<<grid, kKsThreads, smem, s>>>(P); break;
    SPF_KS_CASE(1) SPF_KS_CASE(2) SPF_KS_CASE(3) SPF_KS_CASE(4) SPF_KS_CASE(5) SPF_KS_CASE(6) SPF_KS_CASE(7) SPF_KS_CASE(8)
#undef SPF_KS_CASE
  }
  return check_launch(ctx, "keyswitch_kernel");
}

int launch_sample_extract(spf_b200_ctx* ctx, uint64_t* d_out, const uint64_t* d_glwe, const uint32_t* d_idx,
                          uint32_t idx_all, size_t batch, cudaStream_t s, const void* const* ptrs = nullptr) {
  if (batch == 0) return 0;
  if (!d_idx && idx_all >= (uint32_t)kN) return fail(ctx, SPF_E_INVALID, "sample_extract index >= N");
  for (size_t off = 0; off < batch; off += 65535) {
    const int nb = (int)std::min<size_t>(65535, batch - off);
    dim3 grid(3, nb);
    sample_extract_kernel<<<grid, 256, 0, s>>>(d_out + off * (kN + 1), d_glwe ? d_glwe + off * 2 * kN : nullptr,
                                               ptrs ? ptrs + off : nullptr, d_idx ? d_idx + off : nullptr, idx_all, nb);
    if (int rc = check_launch(ctx, "sample_extract_kernel")) return rc;
  }
  return 0;
}

int launch_elementwise(spf_b200_ctx* ctx, uint64_t* d_out, const uint64_t* d_a, const uint64_t* d_b, int op,
                       uint32_t n, size_t batch, cudaStream_t s, const void* const* ptrs = nullptr,
                       const uint32_t* nvec = nullptr) {
  if (batch == 0) return 0;
  const size_t total = batch * 2 * kN;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)ctx->sm_count * 16);
  glwe_elementwise_kernel<<<blocks, 256, 0, s>>>(d_out, d_a, d_b, ptrs, nvec, op, n, batch);
  return check_launch(ctx, "glwe_elementwise_kernel");
}

int launch_rlwe_encrypt(spf_b200_ctx* ctx, uint64_t* d_out, const uint64_t* d_pk, const uint64_t* d_msg, const uint64_t* d_u,
                        const uint64_t* d_e0, const uint64_t* d_e1, size_t batch, cudaStream_t s) {
  if (batch == 0) return 0;
  if (ctx->p.glwe_k != 1 || ctx->p.glwe_n != (uint32_t)kN) return fail(ctx, SPF_E_UNSUPPORTED, "rlwe_encrypt_public: k = 1, N = 2048 only");
  static const bool attr = [] {
    return cudaFuncSetAttribute(rlwe_encrypt_public_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kRlweSmem) == cudaSuccess;
  }();
  if (!attr) return fail(ctx, SPF_E_CUDA, "rlwe_encrypt_public_kernel: shared memory attribute");
  for (size_t off = 0; off < batch; off += (size_t)1 << 30) {
    const size_t n = std::min<size_t>((size_t)1 << 30, batch - off);
    RlweBatch P{d_out + off * 2 * kN, d_pk, d_msg + off * kN, d_u + off * kN, d_e0 + off * kN, d_e1 + off * kN, (int)n};
    const int blocks = (int)std::min<size_t>(n, (size_t)ctx->sm_count * 2);
    rlwe_encrypt_public_kernel<<<blocks, kRlweThreads, kRlweSmem, s>>>(P);
    if (int rc = check_launch(ctx, "rlwe_encrypt_public_kernel")) return rc;
  }
  return 0;
}

// Largest chunk of a host-pointer batch processed per pipeline slot: one PBS
// wave (148 SMs x 3 ciphertexts) so chunking costs no tail.
size_t cbs_chunk(const spf_b200_ctx* ctx) { return (size_t)ctx->sm_count * kPbsPairs; }

// ---- host-pointer ops: chunked, double-buffered over the context's two streams ---------------

// Generic 2-slot pipeline: for each chunk [off, off+n): stage(slot, off, n) enqueues H2D copies,
// kernels and D2H copies on ctx->stream[slot].  A slot is reused only after its previous chunk
// has drained.
template <class Stage>
int run_chunks(spf_b200_ctx* ctx, size_t batch, size_t chunk, Stage stage) {
  CU(cudaSetDevice(ctx->device));
  int slot = 0;
  bool used[2] = {false, false};
  for (size_t off = 0; off < batch; off += chunk, slot ^= 1) {
    const size_t n = std::min(chunk, batch - off);
    if (used[slot]) CU(cudaStreamSynchronize(ctx->stream[slot]));
    used[slot] = true;
    if (int rc = stage(slot, off, n)) {
      cudaStreamSynchronize(ctx->stream[0]);
      cudaStreamSynchronize(ctx->stream[1]);
      return rc;
    }
  }
  CU(cudaStreamSynchronize(ctx->stream[0]));
  CU(cudaStreamSynchronize(ctx->stream[1]));
  return 0;
}

// shared body of cmux / glev_cmux / multiply_glwe_ggsw
int host_cmux_like(spf_b200_ctx* ctx, uint64_t* out, const double* ggsw_in, const uint64_t* a,
                          const uint64_t* b, size_t batch, int glwe_per_item) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!out || !ggsw_in || !b) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  const size_t glwe = len_glwe(&ctx->p) * glwe_per_item, ggsw = spf_b200_len_ggsw_l1(&ctx->p);
  return run_chunks(ctx, batch, 2048, [&](int slot, size_t off, size_t n) -> int {
    cudaStream_t s = ctx->stream[slot];
    DevBuf* sc = ctx->scratch[slot];
    if (int rc = ensure(ctx, sc[0], n * glwe * 8)) return rc;
    if (int rc = ensure(ctx, sc[1], n * glwe * 8)) return rc;
    if (int rc = ensure(ctx, sc[2], n * ggsw * 16)) return rc;
    if (int rc = ensure(ctx, sc[3], n * glwe * 8)) return rc;
    if (a) CU(cudaMemcpyAsync(sc[0].p, a + off * glwe, n * glwe * 8, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(sc[1].p, b + off * glwe, n * glwe * 8, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(sc[2].p, ggsw_in + off * ggsw * 2, n * ggsw * 16, cudaMemcpyHostToDevice, s));
    if (int rc = launch_scale(ctx, (C2*)sc[2].p, (const C2*)sc[2].p, n * ggsw, 1.0 / 1024.0, s)) return rc;
    if (int rc = launch_cmux(ctx, (uint64_t*)sc[3].p, a ? (const uint64_t*)sc[0].p : nullptr, (const uint64_t*)sc[1].p,
                             (const C2*)sc[2].p, ggsw, glwe_per_item, n * glwe_per_item, s))
      return rc;
    CU(cudaMemcpyAsync(out + off * glwe, sc[3].p, n * glwe * 8, cudaMemcpyDeviceToHost, s));
    return 0;
  });
}

int host_elementwise(spf_b200_ctx* ctx, uint64_t* out, const uint64_t* a, const uint64_t* b, int op, uint32_t n_rot,
                            size_t batch) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!out || !a || (op == 0 && !b)) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  const size_t glwe = len_glwe(&ctx->p);
  return run_chunks(ctx, batch, 8192, [&](int slot, size_t off, size_t n) -> int {
    cudaStream_t s = ctx->stream[slot];
    DevBuf* sc = ctx->scratch[slot];
    if (int rc = ensure(ctx, sc[0], n * glwe * 8)) return rc;
    if (int rc = ensure(ctx, sc[1], n * glwe * 8)) return rc;
    if (int rc = ensure(ctx, sc[3], n * glwe * 8)) return rc;
    CU(cudaMemcpyAsync(sc[0].p, a + off * glwe, n * glwe * 8, cudaMemcpyHostToDevice, s));
    if (op == 0) CU(cudaMemcpyAsync(sc[1].p, b + off * glwe, n * glwe * 8, cudaMemcpyHostToDevice, s));
    if (int rc = launch_elementwise(ctx, (uint64_t*)sc[3].p, (const uint64_t*)sc[0].p, (const uint64_t*)sc[1].p, op, n_rot, n, s))
      return rc;
    CU(cudaMemcpyAsync(out + off * glwe, sc[3].p, n * glwe * 8, cudaMemcpyDeviceToHost, s));
    return 0;
  });
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

void spf_b200_default_128(spf_params* p) {
  p->lwe_n = 637;  p->lwe_std = 7.25e-5;
  p->glwe_k = 1;   p->glwe_n = 2048;  p->glwe_std = 7e-16;
  p->cbs = {4, 4};
  p->pbs = {16, 2};
  p->ks = {2, 6};
  p->pfks = {17, 2};
  p->ss = {3, 15};
  p->tr = {7, 6};
}

size_t spf_b200_len_lwe_l0(const spf_params* p) { return (size_t)p->lwe_n + 1; }
size_t spf_b200_len_lwe_l1(const spf_params* p) { return (size_t)p->glwe_k * p->glwe_n + 1; }
size_t spf_b200_len_glwe_l1(const spf_params* p) { return len_glwe(p); }
size_t spf_b200_len_glev_l1(const spf_params* p) { return len_glwe(p) * p->cbs.count; }
size_t spf_b200_len_ggsw_l1(const spf_params* p) { return len_ggsw(p, p->cbs); }
size_t spf_b200_len_bsk(const spf_params* p) { return len_ggsw(p, p->pbs) * p->lwe_n; }
size_t spf_b200_len_ksk(const spf_params* p) {
  return (size_t)p->glwe_k * p->glwe_n * p->ks.count * ((size_t)p->lwe_n + 1);
}
size_t spf_b200_len_ssk(const spf_params* p) {
  return len_glwe(p) * p->ss.count / 2 * ((size_t)p->glwe_k * (p->glwe_k + 1) / 2);
}
size_t spf_b200_len_ak(const spf_params* p) {
  return len_glwe(p) * p->tr.count / 2 * p->glwe_k * ilog2u(p->glwe_n);
}

int spf_b200_create(const spf_params* params, const double* bsk_fft, size_t bsk_len, const uint64_t* ksk,
                    size_t ksk_len, const double* ssk_fft, size_t ssk_len, const double* ak_fft, size_t ak_len,
                    int device, spf_b200_ctx** out) {
  return create_common(params, bsk_fft, bsk_len, ksk, ksk_len, ssk_fft, ssk_len, ak_fft, ak_len, device, false, out);
}
int spf_b200_create_from_device(const spf_params* params, const double* d_bsk_fft, size_t bsk_len,
                                const uint64_t* d_ksk, size_t ksk_len, const double* d_ssk_fft, size_t ssk_len,
                                const double* d_ak_fft, size_t ak_len, int device, spf_b200_ctx** out) {
  return create_common(params, d_bsk_fft, bsk_len, d_ksk, ksk_len, d_ssk_fft, ssk_len, d_ak_fft, ak_len, device, true,
                       out);
}

void spf_b200_destroy(spf_b200_ctx* ctx) {
  if (!ctx) return;
  if (ctx->refs.fetch_sub(1) > 1) return;  // graphs built on this context are still alive: the last one frees it
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  cudaFree(ctx->bsk); cudaFree(ctx->ak); cudaFree(ctx->ssk); cudaFree(ctx->ksk); cudaFree(ctx->ksk_colsum); cudaFree(ctx->ks_tc_colsum); cudaFree(ctx->ks_btiles);
  cudaFree(ctx->T1); cudaFree(ctx->T2); cudaFree(ctx->kinv); cudaFree(ctx->consts);
  for (int i = 0; i < 2; i++) {
    for (DevBuf& b : ctx->scratch[i]) cudaFree(b.p);
    if (ctx->stream[i]) cudaStreamDestroy(ctx->stream[i]);
    if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->ev_copied[i]) cudaEventDestroy(ctx->ev_copied[i]);
  }
  if (ctx->aux) cudaStreamDestroy(ctx->aux);
  if (ctx->ev_cbs_main) cudaEventDestroy(ctx->ev_cbs_main);
  if (ctx->ev_cbs_tail) cudaEventDestroy(ctx->ev_cbs_tail);
  delete ctx;
}

const char* spf_b200_last_error(const spf_b200_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }
uint64_t spf_b200_kernel_launches(const spf_b200_ctx* ctx) { return ctx ? ctx->launches.load() : 0; }
int spf_b200_device(const spf_b200_ctx* ctx) { return ctx ? ctx->device : -1; }

int spf_b200_synchronize(spf_b200_ctx* ctx) {
  if (!ctx) return SPF_E_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream[0]));
  CU(cudaStreamSynchronize(ctx->stream[1]));
  return 0;
}

// ---- device-pointer ops -------------------------------------------------------------------

int spf_b200_dev_circuit_bootstrap(spf_b200_ctx* ctx, double* d_ggsw_out, const uint64_t* d_lwe0_in, size_t batch,
                                   int reference_scale, void* stream) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!d_ggsw_out || !d_lwe0_in) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t s = pick(ctx, stream);
  // PBS output scratch: slot 0 when running on the caller's stream
  DevBuf& g = ctx->scratch[0][5];
  if (int rc = ensure(ctx, g, batch * len_glwe(&ctx->p) * 8)) return rc;
  return launch_cbs(ctx, (C2*)d_ggsw_out, (uint64_t*)g.p, d_lwe0_in, nullptr, reference_scale ? 1024.0 : 1.0, batch, s);
}

int spf_b200_dev_programmable_bootstrap(spf_b200_ctx* ctx, uint64_t* d_glwe_out, const uint64_t* d_lwe0_in,
                                        const uint64_t* d_lut_glwe, uint32_t log_chi, uint32_t log_v, size_t batch,
                                        void* stream) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!d_glwe_out || !d_lwe0_in || !d_lut_glwe) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  if (log_chi + log_v >= 12 || log_chi >= 52) return fail(ctx, SPF_E_INVALID, "log_chi/log_v out of range");
  CU(cudaSetDevice(ctx->device));
  return launch_pbs(ctx, d_glwe_out, d_lwe0_in, d_lut_glwe, false, log_chi, log_v, batch, pick(ctx, stream));
}

int spf_b200_dev_cmux(spf_b200_ctx* ctx, uint64_t* d_glwe_out, const double* d_sel_ggsw, size_t ggsw_stride,
                      const uint64_t* d_a, const uint64_t* d_b, size_t batch, void* stream) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!d_glwe_out || !d_sel_ggsw || !d_a || !d_b) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  CU(cudaSetDevice(ctx->device));
  return launch_cmux(ctx, d_glwe_out, d_a, d_b, (const C2*)d_sel_ggsw, ggsw_stride, 1, batch, pick(ctx, stream));
}

int spf_b200_dev_keyswitch_lwe_l1_lwe_l0(spf_b200_ctx* ctx, uint64_t* d_lwe0_out, const uint64_t* d_lwe1_in,
                                         size_t batch, void* stream) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!d_lwe0_out || !d_lwe1_in) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  CU(cudaSetDevice(ctx->device));
  return launch_keyswitch(ctx, d_lwe0_out, d_lwe1_in, batch, pick(ctx, stream));
}

int spf_b200_dev_sample_extract_l1(spf_b200_ctx* ctx, uint64_t* d_lwe1_out, const uint64_t* d_glwe_in,
                                   const uint32_t* d_idx, uint32_t idx_all, size_t batch, void* stream) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!d_lwe1_out || !d_glwe_in) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  CU(cudaSetDevice(ctx->device));
  return launch_sample_extract(ctx, d_lwe1_out, d_glwe_in, d_idx, idx_all, batch, pick(ctx, stream));
}

int spf_b200_dev_fft_rescale(spf_b200_ctx* ctx, double* d_dst, const double* d_src, size_t n, int to_device,
                             void* stream) {
  if (!ctx) return SPF_E_INVALID;
  if (n == 0) return 0;
  if (!d_dst || !d_src) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  CU(cudaSetDevice(ctx->device));
  return launch_scale(ctx, (C2*)d_dst, (const C2*)d_src, n, to_device ? 1.0 / 1024.0 : 1024.0, pick(ctx, stream));
}

int spf_b200_circuit_bootstrap(spf_b200_ctx* ctx, double* ggsw_out, const uint64_t* lwe0_in, size_t batch) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!ggsw_out || !lwe0_in) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  const size_t lwe = spf_b200_len_lwe_l0(&ctx->p), glwe = len_glwe(&ctx->p), ggsw = spf_b200_len_ggsw_l1(&ctx->p);
  // Pipeline: every kernel on ONE compute stream (a second stream's bootstraps would only fight the
  // first one's for the SMs), the 256 KiB-per-ciphertext results leave on a copy stream from two
  // alternating staging buffers; events order the hand-over, the host never waits inside the loop.
  CU(cudaSetDevice(ctx->device));
  const size_t chunk = std::min(cbs_chunk(ctx), batch);
  cudaStream_t comp = ctx->stream[0], copy = ctx->stream[1];
  for (int slot = 0; slot < 2; slot++) {
    if (int rc = ensure(ctx, ctx->scratch[slot][0], chunk * lwe * 8)) return rc;
    if (int rc = ensure(ctx, ctx->scratch[slot][1], chunk * glwe * 8)) return rc;
    if (int rc = ensure(ctx, ctx->scratch[slot][2], chunk * ggsw * 16)) return rc;
  }
  int slot = 0, rc = 0;
  size_t k = 0;
  for (size_t off = 0; off < batch && rc == 0; off += chunk, slot ^= 1, k++) {
    const size_t n = std::min(chunk, batch - off);
    DevBuf* sc = ctx->scratch[slot];
    if (k >= 2) CU(cudaStreamWaitEvent(comp, ctx->ev_copied[slot], 0));  // staging buffer drained
    CU(cudaMemcpyAsync(sc[0].p, lwe0_in + off * lwe, n * lwe * 8, cudaMemcpyHostToDevice, comp));
    rc = launch_cbs(ctx, (C2*)sc[2].p, (uint64_t*)sc[1].p, (const uint64_t*)sc[0].p, nullptr, 1024.0, n, comp);
    if (rc) break;
    CU(cudaEventRecord(ctx->ev[slot], comp));
    CU(cudaStreamWaitEvent(copy, ctx->ev[slot], 0));
    CU(cudaMemcpyAsync(ggsw_out + off * ggsw * 2, sc[2].p, n * ggsw * 16, cudaMemcpyDeviceToHost, copy));
    CU(cudaEventRecord(ctx->ev_copied[slot], copy));
  }
  const cudaError_t e0 = cudaStreamSynchronize(comp), e1 = cudaStreamSynchronize(copy);
  if (rc) return rc;
  if (e0 != cudaSuccess || e1 != cudaSuccess)
    return fail(ctx, SPF_E_CUDA, std::string("circuit_bootstrap pipeline: ") + cudaGetErrorString(e0 != cudaSuccess ? e0 : e1));
  return 0;
}

int spf_b200_programmable_bootstrap(spf_b200_ctx* ctx, uint64_t* glwe_out, const uint64_t* lwe0_in,
                                    const uint64_t* lut_glwe, uint32_t log_chi, uint32_t log_v, size_t batch) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!glwe_out || !lwe0_in || !lut_glwe) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  if (log_chi + log_v >= 12 || log_chi >= 52) return fail(ctx, SPF_E_INVALID, "log_chi/log_v out of range");
  const size_t lwe = spf_b200_len_lwe_l0(&ctx->p), glwe = len_glwe(&ctx->p);
  return run_chunks(ctx, batch, cbs_chunk(ctx), [&](int slot, size_t off, size_t n) -> int {
    cudaStream_t s = ctx->stream[slot];
    DevBuf* sc = ctx->scratch[slot];
    if (int rc = ensure(ctx, sc[0], n * lwe * 8)) return rc;
    if (int rc = ensure(ctx, sc[1], n * glwe * 8)) return rc;
    if (int rc = ensure(ctx, sc[3], glwe * 8)) return rc;
    CU(cudaMemcpyAsync(sc[0].p, lwe0_in + off * lwe, n * lwe * 8, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(sc[3].p, lut_glwe, glwe * 8, cudaMemcpyHostToDevice, s));
    if (int rc = launch_pbs(ctx, (uint64_t*)sc[1].p, (const uint64_t*)sc[0].p, (const uint64_t*)sc[3].p, false, log_chi, log_v, n, s))
      return rc;
    CU(cudaMemcpyAsync(glwe_out + off * glwe, sc[1].p, n * glwe * 8, cudaMemcpyDeviceToHost, s));
    return 0;
  });
}

int spf_b200_cmux(spf_b200_ctx* ctx, uint64_t* glwe_out, const double* sel_ggsw, const uint64_t* a, const uint64_t* b,
                  size_t batch) {
  if (ctx && batch && !a) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  return host_cmux_like(ctx, glwe_out, sel_ggsw, a, b, batch, 1);
}
int spf_b200_glev_cmux(spf_b200_ctx* ctx, uint64_t* glev_out, const double* sel_ggsw, const uint64_t* a,
                       const uint64_t* b, size_t batch) {
  if (ctx && batch && !a) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  return host_cmux_like(ctx, glev_out, sel_ggsw, a, b, batch, ctx ? (int)ctx->p.cbs.count : 1);
}
int spf_b200_multiply_glwe_ggsw(spf_b200_ctx* ctx, uint64_t* glwe_out, const uint64_t* glwe, const double* ggsw,
                                size_t batch) {
  return host_cmux_like(ctx, glwe_out, ggsw, nullptr, glwe, batch, 1);
}

int spf_b200_keyswitch_lwe_l1_lwe_l0(spf_b200_ctx* ctx, uint64_t* lwe0_out, const uint64_t* lwe1_in, size_t batch) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!lwe0_out || !lwe1_in) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  const size_t l1 = spf_b200_len_lwe_l1(&ctx->p), l0 = spf_b200_len_lwe_l0(&ctx->p);
  return run_chunks(ctx, batch, 8192, [&](int slot, size_t off, size_t n) -> int {
    cudaStream_t s = ctx->stream[slot];
    DevBuf* sc = ctx->scratch[slot];
    if (int rc = ensure(ctx, sc[0], n * l1 * 8)) return rc;
    if (int rc = ensure(ctx, sc[1], n * l0 * 8)) return rc;
    CU(cudaMemcpyAsync(sc[0].p, lwe1_in + off * l1, n * l1 * 8, cudaMemcpyHostToDevice, s));
    if (int rc = launch_keyswitch(ctx, (uint64_t*)sc[1].p, (const uint64_t*)sc[0].p, n, s)) return rc;
    CU(cudaMemcpyAsync(lwe0_out + off * l0, sc[1].p, n * l0 * 8, cudaMemcpyDeviceToHost, s));
    return 0;
  });
}

int spf_b200_sample_extract_l1(spf_b200_ctx* ctx, uint64_t* lwe1_out, const uint64_t* glwe_in, const uint32_t* idx,
                               uint32_t idx_all, size_t batch) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!lwe1_out || !glwe_in) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  if (idx) { for (size_t i = 0; i < batch; i++) if (idx[i] >= (uint32_t)kN) return fail(ctx, SPF_E_INVALID, "sample_extract index >= N"); }
  else if (idx_all >= (uint32_t)kN) return fail(ctx, SPF_E_INVALID, "sample_extract index >= N");
  const size_t l1 = spf_b200_len_lwe_l1(&ctx->p), glwe = len_glwe(&ctx->p);
  return run_chunks(ctx, batch, 8192, [&](int slot, size_t off, size_t n) -> int {
    cudaStream_t s = ctx->stream[slot];
    DevBuf* sc = ctx->scratch[slot];
    if (int rc = ensure(ctx, sc[0], n * glwe * 8)) return rc;
    if (int rc = ensure(ctx, sc[1], n * l1 * 8)) return rc;
    if (int rc = ensure(ctx, sc[3], n * 4)) return rc;
    CU(cudaMemcpyAsync(sc[0].p, glwe_in + off * glwe, n * glwe * 8, cudaMemcpyHostToDevice, s));
    if (idx) CU(cudaMemcpyAsync(sc[3].p, idx + off, n * 4, cudaMemcpyHostToDevice, s));
    if (int rc = launch_sample_extract(ctx, (uint64_t*)sc[1].p, (const uint64_t*)sc[0].p, idx ? (const uint32_t*)sc[3].p : nullptr, idx_all, n, s))
      return rc;
    CU(cudaMemcpyAsync(lwe1_out + off * l1, sc[1].p, n * l1 * 8, cudaMemcpyDeviceToHost, s));
    return 0;
  });
}

int spf_b200_scheme_switch(spf_b200_ctx* ctx, double* ggsw_out, const uint64_t* glev_in, size_t batch) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!ggsw_out || !glev_in) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  const size_t glev = spf_b200_len_glev_l1(&ctx->p), ggsw = spf_b200_len_ggsw_l1(&ctx->p);
  return run_chunks(ctx, batch, 2048, [&](int slot, size_t off, size_t n) -> int {
    cudaStream_t s = ctx->stream[slot];
    DevBuf* sc = ctx->scratch[slot];
    if (int rc = ensure(ctx, sc[0], n * glev * 8)) return rc;
    if (int rc = ensure(ctx, sc[2], n * ggsw * 16)) return rc;
    CU(cudaMemcpyAsync(sc[0].p, glev_in + off * glev, n * glev * 8, cudaMemcpyHostToDevice, s));
    if (int rc = launch_trace_ss(ctx, (const uint64_t*)sc[0].p, nullptr, (C2*)sc[2].p, 2, (int)ctx->p.cbs.count, 1024.0, n, s))
      return rc;
    CU(cudaMemcpyAsync(ggsw_out + off * ggsw * 2, sc[2].p, n * ggsw * 16, cudaMemcpyDeviceToHost, s));
    return 0;
  });
}

int spf_b200_trace(spf_b200_ctx* ctx, uint64_t* glwe_out, const uint64_t* glwe_in, size_t batch) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!glwe_out || !glwe_in) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  const size_t glwe = len_glwe(&ctx->p);
  return run_chunks(ctx, batch, 4096, [&](int slot, size_t off, size_t n) -> int {
    cudaStream_t s = ctx->stream[slot];
    DevBuf* sc = ctx->scratch[slot];
    if (int rc = ensure(ctx, sc[0], n * glwe * 8)) return rc;
    if (int rc = ensure(ctx, sc[1], n * glwe * 8)) return rc;
    CU(cudaMemcpyAsync(sc[0].p, glwe_in + off * glwe, n * glwe * 8, cudaMemcpyHostToDevice, s));
    if (int rc = launch_trace_ss(ctx, (const uint64_t*)sc[0].p, (uint64_t*)sc[1].p, nullptr, 1, 1, 1.0, n, s)) return rc;
    CU(cudaMemcpyAsync(glwe_out + off * glwe, sc[1].p, n * glwe * 8, cudaMemcpyDeviceToHost, s));
    return 0;
  });
}

int spf_b200_not(spf_b200_ctx* ctx, uint64_t* glwe_out, const uint64_t* glwe_in, size_t batch) {
  return host_elementwise(ctx, glwe_out, glwe_in, nullptr, 1, 0, batch);
}
int spf_b200_xor(spf_b200_ctx* ctx, uint64_t* glwe_out, const uint64_t* a, const uint64_t* b, size_t batch) {
  return host_elementwise(ctx, glwe_out, a, b, 0, 0, batch);
}
int spf_b200_mul_xn(spf_b200_ctx* ctx, uint64_t* glwe_out, const uint64_t* glwe_in, uint32_t n, size_t batch) {
  return host_elementwise(ctx, glwe_out, glwe_in, nullptr, 2, n, batch);
}

int spf_b200_dev_rlwe_encrypt_public(spf_b200_ctx* ctx, uint64_t* d_glwe_out, const uint64_t* d_public_key,
                                     const uint64_t* d_encoded_msg, const uint64_t* d_u, const uint64_t* d_e0,
                                     const uint64_t* d_e1, size_t batch, void* stream) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!d_glwe_out || !d_public_key || !d_encoded_msg || !d_u || !d_e0 || !d_e1) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  CU(cudaSetDevice(ctx->device));
  return launch_rlwe_encrypt(ctx, d_glwe_out, d_public_key, d_encoded_msg, d_u, d_e0, d_e1, batch, pick(ctx, stream));
}

int spf_b200_rlwe_encrypt_public(spf_b200_ctx* ctx, uint64_t* glwe_out, const uint64_t* public_key,
                                 const uint64_t* encoded_msg, const uint64_t* u, const uint64_t* e0, const uint64_t* e1,
                                 size_t batch) {
  if (!ctx) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!glwe_out || !public_key || !encoded_msg || !u || !e0 || !e1) return fail(ctx, SPF_E_INVALID, "NULL buffer");
  const size_t n = ctx->p.glwe_n, glwe = len_glwe(&ctx->p);
  return run_chunks(ctx, batch, 4096, [&](int slot, size_t off, size_t cnt) -> int {
    cudaStream_t s = ctx->stream[slot];
    DevBuf* sc = ctx->scratch[slot];
    for (int b = 0; b < 4; b++)
      if (int rc = ensure(ctx, sc[b], cnt * n * 8)) return rc;
    if (int rc = ensure(ctx, sc[4], cnt * glwe * 8)) return rc;
    if (int rc = ensure(ctx, sc[5], glwe * 8)) return rc;
    CU(cudaMemcpyAsync(sc[5].p, public_key, glwe * 8, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(sc[0].p, encoded_msg + off * n, cnt * n * 8, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(sc[1].p, u + off * n, cnt * n * 8, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(sc[2].p, e0 + off * n, cnt * n * 8, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(sc[3].p, e1 + off * n, cnt * n * 8, cudaMemcpyHostToDevice, s));
    if (int rc = launch_rlwe_encrypt(ctx, (uint64_t*)sc[4].p, (const uint64_t*)sc[5].p, (const uint64_t*)sc[0].p,
                                     (const uint64_t*)sc[1].p, (const uint64_t*)sc[2].p, (const uint64_t*)sc[3].p, cnt, s))
      return rc;
    CU(cudaMemcpyAsync(glwe_out + off * glwe, sc[4].p, cnt * glwe * 8, cudaMemcpyDeviceToHost, s));
    return 0;
  });
}

int spf_b200_fp64_peak(spf_b200_ctx* ctx, double* tflops_out) {
  if (!ctx || !tflops_out) return SPF_E_INVALID;
  CU(cudaSetDevice(ctx->device));
  const int threads = 256, blocks = ctx->sm_count * 8, iters = 1 << 15;
  DevBuf& b = ctx->scratch[0][4];
  if (int rc = ensure(ctx, b, (size_t)threads * blocks * 8)) return rc;
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0));
  CU(cudaEventCreate(&e1));
  double best = 0;
  for (int rep = 0; rep < 5; rep++) {
    CU(cudaEventRecord(e0, ctx->stream[0]));
    dfma_probe_kernel<<<blocks, threads, 0, ctx->stream[0]>>>((double*)b.p, iters);
    if (int rc = check_launch(ctx, "dfma_probe_kernel")) return rc;
    CU(cudaEventRecord(e1, ctx->stream[0]));
    CU(cudaEventSynchronize(e1));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 8.0 * (double)iters * threads * blocks;
    if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *tflops_out = best;
  return 0;
}

}  // extern "C"

#include "graph.cuh"
#include "serial.inl"
#include "box.cuh"
