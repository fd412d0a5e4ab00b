// graph.cuh -- level-synchronous, batching executor for FheCircuit graphs (included by capi.cu).
//
// Replaces the one-rayon-task-per-op scheduling of CircuitProcessor::{dispatch,execute_task,
// exec_op} (parasol_runtime/src/circuit_processor/mod.rs:130-546) for a whole graph at a time:
// nodes are levelised by dependency depth, all nodes of one (level, op) group run as ONE batched
// kernel launch, every intermediate ciphertext stays in HBM (GGSWs in the 2^-10 device scale),
// and only Input*/Output* nodes touch host memory.  Validation mirrors Task::validate
// (circuit_processor/task.rs:24-179): wrong input kinds / missing inputs / illegal sample-extract
// index are reported as SPF_E_GRAPH with a message instead of a RuntimeError.
#pragma once

namespace {

enum CtType { T_NONE = 0, T_LWE0, T_LWE1, T_GLWE1, T_GGSW1, T_GLEV1 };

const char* kOpNames[] = {"InputLwe0", "InputLwe1", "InputGlwe1", "InputGgsw1", "InputGlev1", "OutputLwe0", "OutputLwe1",
                          "OutputGlwe1", "OutputGgsw1", "OutputGlev1", "SampleExtract", "KeyswitchL1toL0", "Not", "GlweAdd",
                          "CMux", "GlevCMux", "MultiplyGgswGlwe", "CircuitBootstrap", "SchemeSwitch", "ZeroLwe0", "OneLwe0",
                          "ZeroGlwe1", "OneGlwe1", "ZeroGgsw1", "OneGgsw1", "ZeroGlev1", "OneGlev1", "Retire", "Nop", "MulXN"};

struct OpInfo {
  CtType out;
  int n_in;
  CtType in[3];
};

OpInfo op_info(uint32_t op) {
  switch (op) {
    case SPF_OP_INPUT_LWE0: return {T_LWE0, 0, {}};
    case SPF_OP_INPUT_LWE1: return {T_LWE1, 0, {}};
    case SPF_OP_INPUT_GLWE1: return {T_GLWE1, 0, {}};
    case SPF_OP_INPUT_GGSW1: return {T_GGSW1, 0, {}};
    case SPF_OP_INPUT_GLEV1: return {T_GLEV1, 0, {}};
    case SPF_OP_OUTPUT_LWE0: return {T_NONE, 1, {T_LWE0}};
    case SPF_OP_OUTPUT_LWE1: return {T_NONE, 1, {T_LWE1}};
    case SPF_OP_OUTPUT_GLWE1: return {T_NONE, 1, {T_GLWE1}};
    case SPF_OP_OUTPUT_GGSW1: return {T_NONE, 1, {T_GGSW1}};
    case SPF_OP_OUTPUT_GLEV1: return {T_NONE, 1, {T_GLEV1}};
    case SPF_OP_SAMPLE_EXTRACT: return {T_LWE1, 1, {T_GLWE1}};
    case SPF_OP_KEYSWITCH_L1_TO_L0: return {T_LWE0, 1, {T_LWE1}};
    case SPF_OP_NOT: return {T_GLWE1, 1, {T_GLWE1}};
    case SPF_OP_GLWE_ADD: return {T_GLWE1, 2, {T_GLWE1, T_GLWE1}};
    case SPF_OP_CMUX: return {T_GLWE1, 3, {T_GGSW1, T_GLWE1, T_GLWE1}};
    case SPF_OP_GLEV_CMUX: return {T_GLEV1, 3, {T_GGSW1, T_GLEV1, T_GLEV1}};
    case SPF_OP_MULTIPLY_GGSW_GLWE: return {T_GLWE1, 2, {T_GLWE1, T_GGSW1}};
    case SPF_OP_CIRCUIT_BOOTSTRAP: return {T_GGSW1, 1, {T_LWE0}};
    case SPF_OP_SCHEME_SWITCH: return {T_GGSW1, 1, {T_GLEV1}};
    case SPF_OP_ZERO_LWE0: case SPF_OP_ONE_LWE0: return {T_LWE0, 0, {}};
    case SPF_OP_ZERO_GLWE1: case SPF_OP_ONE_GLWE1: return {T_GLWE1, 0, {}};
    case SPF_OP_ZERO_GGSW1: case SPF_OP_ONE_GGSW1: return {T_GGSW1, 0, {}};
    case SPF_OP_ZERO_GLEV1: case SPF_OP_ONE_GLEV1: return {T_GLEV1, 0, {}};
    case SPF_OP_MUL_XN: return {T_GLWE1, 1, {T_GLWE1}};
    default: return {T_NONE, 0, {}};  // Retire, Nop
  }
}

size_t ct_bytes(const spf_params* p, CtType t) {
  switch (t) {
    case T_LWE0: return spf_b200_len_lwe_l0(p) * 8;
    case T_LWE1: return spf_b200_len_lwe_l1(p) * 8;
    case T_GLWE1: return spf_b200_len_glwe_l1(p) * 8;
    case T_GGSW1: return spf_b200_len_ggsw_l1(p) * 16;
    case T_GLEV1: return spf_b200_len_glev_l1(p) * 8;
    default: return 0;
  }
}
size_t ct_host_bytes(const spf_params* p, CtType t) { return ct_bytes(p, t); }

struct Group {
  uint32_t op;
  int level;
  std::vector<int> ids;   // slot k of the group's output buffer holds node ids[k]; -1 = padding slot
  size_t ptr_off = 0;   // offset (entries) into the device pointer table
  size_t u32_off = 0;   // offset into the device u32 table
  char* out_base = nullptr;
  char* scratch = nullptr;  // CBS: PBS outputs
  // Sharded layout (world > 1): slots [all_start, all_start + all_cnt) are computed by every rank,
  // slots [r_start[r], r_start[r] + r_cnt[r]) by rank r only.  `gather_chunk` > 0: the first
  // world * gather_chunk slots are `world` equal chunks completed by an all-gather after the group.
  size_t all_start = 0, all_cnt = 0;
  std::vector<size_t> r_start, r_cnt;
  size_t gather_chunk = 0;
  bool slot_outputs = false;  // CMux / MultiplyGgswGlwe: every output has its own recycled GLWE slot (out pointer table)
};

}  // namespace

struct spf_b200_graph {
  spf_b200_ctx* ctx = nullptr;
  std::vector<spf_node> nodes;
  std::vector<CtType> type;
  std::vector<int> level;
  std::vector<char*> dptr;  // device address of each node's output ciphertext
  std::vector<Group> groups;
  std::vector<int> inputs, outputs;
  char* arena = nullptr;
  size_t arena_bytes = 0;
  void** d_ptrs = nullptr;
  uint32_t* d_u32 = nullptr;
  char* d_out_stage = nullptr;  // rescaled GGSW outputs
  // non-GGSW outputs are gathered (gather_outputs_kernel) into d_gather in g->outputs order before they are copied out
  char* d_gather = nullptr;
  void* d_gather_tab = nullptr;  // [src pointers | word offsets | word counts]
  std::vector<size_t> gather_off;  // byte offset of output k in d_gather, (size_t)-1 for GGSW outputs
  size_t gather_items = 0;
  int n_levels = 0;
  uint64_t launches_per_run = 0;
  int world = 1;  // CircuitBootstrap groups are laid out as `world` equal chunks (spf_b200_graph_build_sharded)
  std::vector<int> owner;  // rank that computes the node's ciphertext, -1 = every rank holds it
  std::vector<int> slot;   // CMux outputs: index of the node's GLWE slot in the recycled pool, -1 otherwise
  size_t pool_slots = 0;   // size of that pool: the largest number of CMux outputs alive at once
  // peer-memory exchange of a sharded run (spf_b200_graph_open_peers / set_peers): the first kArenaHeader bytes of
  // every arena hold the level-barrier flags (u64 per rank) and an error word
  PeerOffsets peers = {};
  bool peers_set = false;
  int peer_rank = -1;
  unsigned long long epoch = 0;
  std::vector<void*> ipc_opened;
  std::vector<void*> pinned;  // io buffers page-locked by this graph (cudaHostRegister), so that their copies are true DMAs
  // io kinds per node (Input* / Output* only): 0 = page-locked host memory (plain DMA), 1 = pageable host memory staged
  // through the graph's own page-locked slab (set_io on an unpinned buffer: registering costs 0.4 ms per buffer and call),
  // 2 = DEVICE memory: a ciphertext handle that never leaves HBM (another graph's output, a torch tensor, ...); GGSWs
  // behind device handles keep the device scale (2^-10), 3 = a box ciphertext handle (rank graphs of a box only: io is
  // the spf_b200_box_ciphertext, whose copies box.cuh enqueues; the single-context parts below skip these nodes)
  std::vector<char> io_kind;
  std::vector<unsigned long long> io_alloc;  // allocation that holds the node's io buffer (alloc_base_of), 0 = do not merge copies
  char* h_stage = nullptr;        // page-locked staging slab for kind-1 buffers
  size_t h_stage_bytes = 0;
  std::vector<size_t> stage_off;  // per node: offset of its ciphertext in h_stage (kind 1), (size_t)-1 otherwise
  // asynchronous execution (spf_b200_graph_spawn): the graph's own stream, an event recorded behind every run, the first
  // error latched by the current / last run, the digit-state scratch of its keyswitch levels
  cudaStream_t stream = nullptr;
  cudaEvent_t done = nullptr;
  std::atomic<int> status{0};
  std::string status_msg;
  DevBuf ks_states;
  bool poisoned = false;  // a failed peer-mode run leaves the ranks' barrier epochs out of step: rebuild the graphs
  // rank that writes the Output* nodes every rank holds (output rank -1); -1 = every rank writes them (one process per
  // rank: each has its own host buffers).  A box (box.cuh) runs all ranks into the same host buffers: rank 0 only.
  int replicated_writer = -1;
};

// one spawned run between dispatch and completion
struct SpawnRecord {
  spf_b200_graph* g;
  spf_completion_fn cb;
  void* user;
  int status;
  std::string msg;
};

namespace {

constexpr size_t kArenaHeader = 4096;  // flags[world] at 0, error word at 2048

// Addresses of the live box ciphertext handles (spf_b200_box_ciphertext_alloc .. _free).  A handle passed where a host
// buffer is expected would otherwise be page-locked and DMA'd as if its bytes were a ciphertext.
std::mutex g_box_handles_mu;
std::unordered_set<const void*> g_box_handles;

bool is_box_handle(const void* p) {
  if (!p) return false;
  std::lock_guard<std::mutex> lk(g_box_handles_mu);
  return g_box_handles.count(p) != 0;
}

// Device constants for Zero*/One* nodes (mod.rs:95-105,475-506).  ZeroGgsw1/OneGgsw1 are real CBS
// outputs of the trivial LWE 0/1, exactly as Evaluation::new computes them (evaluation.rs:161-197).
int ensure_constants(spf_b200_ctx* ctx) {
  if (ctx->consts) return 0;
  const spf_params* p = &ctx->p;
  const size_t lwe0 = ct_bytes(p, T_LWE0), glwe = ct_bytes(p, T_GLWE1), glev = ct_bytes(p, T_GLEV1), ggsw = ct_bytes(p, T_GGSW1);
  const size_t total = 2 * (lwe0 + glwe + glev + ggsw);
  std::vector<char> h(total, 0);
  char* q = h.data();
  // [lwe0 zero, lwe0 one, glwe zero, glwe one, glev zero, glev one, ggsw zero, ggsw one]
  reinterpret_cast<uint64_t*>(q + lwe0)[p->lwe_n] = 1ull << 63;                      // trivial_lwe_l0_one
  reinterpret_cast<uint64_t*>(q + 2 * lwe0 + glwe)[(size_t)p->glwe_k * p->glwe_n] = 1ull << 63;  // trivial one: b[0]
  {
    uint64_t* g1 = reinterpret_cast<uint64_t*>(q + 2 * lwe0 + 2 * glwe + glev);       // trivial_binary_glev(1)
    for (uint32_t j = 0; j < p->cbs.count; j++)
      g1[(size_t)j * spf_b200_len_glwe_l1(p) + (size_t)p->glwe_k * p->glwe_n] = 1ull << (64 - p->cbs.radix_log * (j + 1));
  }
  CU(cudaSetDevice(ctx->device));
  CU(cudaMalloc(&ctx->consts, total));
  CU(cudaMemcpy(ctx->consts, h.data(), total, cudaMemcpyHostToDevice));
  char* d = static_cast<char*>(ctx->consts);
  ctx->c_lwe0[0] = d; ctx->c_lwe0[1] = d + lwe0;
  ctx->c_glwe[0] = d + 2 * lwe0; ctx->c_glwe[1] = d + 2 * lwe0 + glwe;
  ctx->c_glev[0] = d + 2 * lwe0 + 2 * glwe; ctx->c_glev[1] = ctx->c_glev[0] + glev;
  ctx->c_ggsw[0] = d + 2 * lwe0 + 2 * glwe + 2 * glev; ctx->c_ggsw[1] = ctx->c_ggsw[0] + ggsw;
  // the two trivial LWEs are adjacent only if lwe0 is unpadded; bootstrap them one by one
  for (int b = 0; b < 2; b++) {
    if (int rc = spf_b200_dev_circuit_bootstrap(ctx, reinterpret_cast<double*>(ctx->c_ggsw[b]),
                                                reinterpret_cast<const uint64_t*>(ctx->c_lwe0[b]), 1, 0, nullptr))
      return rc;
  }
  CU(cudaStreamSynchronize(ctx->stream[0]));
  return 0;
}

int graph_fail(spf_b200_ctx* ctx, const std::string& msg) { return fail(ctx, SPF_E_GRAPH, msg); }

// Page-lock a host ciphertext buffer for the lifetime of the graph (best effort: a buffer that cannot
// be registered -- already pinned by the caller, read-only mapping -- is simply copied as pageable).
// Buffers that are page-locked already (spf_b200_host_alloc, cudaHostAlloc, a caller's own registration) are left
// alone: cudaHostRegister costs 0.4 ms per 32 KiB buffer and grows with the number of registrations (5 s for the 516
// buffers of four mul32 programs), so hosts should carve their ciphertext buffers out of ONE pinned slab.
// Base address of the allocation (cudaMalloc / cudaHostAlloc) that contains p, 0 when p is not inside ONE such
// allocation known to the driver (pageable memory, a range registered piecemeal).  Copies are only ever merged between
// buffers of the same allocation: a cudaMemcpyAsync that runs over the end of an allocation or registration is refused
// by the driver, and two numpy rows or two 32 KiB cudaMallocs are routinely adjacent.
unsigned long long alloc_base_of(const void* p, size_t* size_out = nullptr) {
  typedef int (*range_fn)(unsigned long long*, size_t*, unsigned long long);
  static range_fn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult st;
    if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &f, cudaEnableDefault, &st) != cudaSuccess || st != cudaDriverEntryPointSuccess) f = nullptr;
    cudaGetLastError();
    return reinterpret_cast<range_fn>(f);
  }();
  if (!fn || !p) return 0;
  unsigned long long base = 0;
  size_t size = 0;
  if (fn(&base, &size, (unsigned long long)(uintptr_t)p) != 0) return 0;
  if (size_out) *size_out = size;
  return base;
}

// Returns the io kind (see spf_b200_graph::io_kind).  `may_register`: page-lock an unpinned host buffer (graph build);
// otherwise (set_io on a built graph) unpinned buffers are staged through the graph's slab.
int pin_io(spf_b200_graph* g, void* p, size_t bytes, bool may_register = true) {
  if (!p) return 0;
  // both ends: a buffer that merely shares its first page with a neighbour's registration is not page-locked
  cudaPointerAttributes attr, attr_end;
  if (cudaPointerGetAttributes(&attr, p) == cudaSuccess &&
      cudaPointerGetAttributes(&attr_end, static_cast<char*>(p) + (bytes ? bytes - 1 : 0)) == cudaSuccess) {
    if (attr.type == cudaMemoryTypeHost && attr_end.type == cudaMemoryTypeHost) return 0;
    if ((attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged) && attr_end.type == attr.type) return 2;
  }
  cudaGetLastError();
  if (!may_register) return 1;
  if (cudaHostRegister(p, bytes, cudaHostRegisterDefault) == cudaSuccess) { g->pinned.push_back(p); return 0; }
  cudaGetLastError();  // clear the sticky-free error
  return 1;
}

// Items per rank of a sharded CircuitBootstrap group: equal chunks (the last ones may be short or
// empty) so that one all-gather of world * chunk items puts every GGSW on every rank.
size_t cbs_chunk_items(size_t n, int world) { return (n + (size_t)world - 1) / (size_t)world; }

// Runs slots [start, start + n) of a group.
int run_group_range(spf_b200_graph* g, const Group& G, cudaStream_t s, size_t start, size_t n, const PeerOffsets* peers = nullptr) {
  spf_b200_ctx* ctx = g->ctx;
  if (n == 0) return 0;
  const spf_params* p = &ctx->p;
  const size_t out_bytes = ct_bytes(p, op_info(G.op).out);
  char* out = G.out_base ? G.out_base + start * out_bytes : nullptr;
  const void* const* base = reinterpret_cast<const void* const*>(g->d_ptrs + G.ptr_off);
  const void* const* p1 = base + start;
  const void* const* p2 = base + 2 * start;
  const void* const* p3 = base + 3 * start;
  const uint32_t* u32 = g->d_u32 + G.u32_off + start;
  switch (G.op) {
    case SPF_OP_SAMPLE_EXTRACT:
      return launch_sample_extract(ctx, reinterpret_cast<uint64_t*>(out), nullptr, u32, 0, n, s, p1);
    case SPF_OP_KEYSWITCH_L1_TO_L0:
      return launch_keyswitch(ctx, reinterpret_cast<uint64_t*>(out), nullptr, n, s, p1, &g->ks_states);
    case SPF_OP_NOT:
      return launch_elementwise(ctx, reinterpret_cast<uint64_t*>(out), nullptr, nullptr, 1, 0, n, s, p2);
    case SPF_OP_GLWE_ADD:
      return launch_elementwise(ctx, reinterpret_cast<uint64_t*>(out), nullptr, nullptr, 0, 0, n, s, p2);
    case SPF_OP_MUL_XN:
      return launch_elementwise(ctx, reinterpret_cast<uint64_t*>(out), nullptr, nullptr, 2, 0, n, s, p2, u32);
    case SPF_OP_CMUX:
    case SPF_OP_MULTIPLY_GGSW_GLWE:  // pointer table: 3 inputs per slot for all slots, then one output pointer per slot
      return launch_cmux(ctx, nullptr, nullptr, nullptr, nullptr, 0, 1, n, s, p3,
                         reinterpret_cast<void* const*>(g->d_ptrs + G.ptr_off + 3 * G.ids.size() + start));
    case SPF_OP_GLEV_CMUX:
      return launch_cmux(ctx, reinterpret_cast<uint64_t*>(out), nullptr, nullptr, nullptr, 0, (int)p->cbs.count, n * p->cbs.count, s, p3);
    case SPF_OP_CIRCUIT_BOOTSTRAP: {
      const size_t glwe = ct_bytes(p, T_GLWE1);
      return launch_cbs(ctx, reinterpret_cast<C2*>(out), reinterpret_cast<uint64_t*>(G.scratch + start * glwe), nullptr, p1, 1.0, n, s,
                        peers);
    }
    case SPF_OP_SCHEME_SWITCH:
      return launch_trace_ss(ctx, nullptr, nullptr, reinterpret_cast<C2*>(out), 2, (int)p->cbs.count, 1.0, n, s, p1);
    default:
      return 0;
  }
}

// This rank's share of a group: the replicated slots, then its own slots.
int run_group(spf_b200_graph* g, const Group& G, cudaStream_t s, int rank, const PeerOffsets* peers = nullptr) {
  if (int rc = run_group_range(g, G, s, G.all_start, G.all_cnt)) return rc;
  return run_group_range(g, G, s, G.r_start[rank], G.r_cnt[rank], peers);
}

// One level barrier over peer memory (peer_barrier_kernel); epochs only grow, so flags never need resetting.
int peer_barrier(spf_b200_graph* g, cudaStream_t s) {
  g->epoch++;
  peer_barrier_kernel<<<1, 32, 0, s>>>(reinterpret_cast<unsigned long long*>(g->arena), g->peers, g->peer_rank, g->epoch,
                                       reinterpret_cast<int*>(g->arena + 2048), 5000000000ull);
  return check_launch(g->ctx, "peer_barrier_kernel");
}

// Host-only part of a graph build: validation, levelisation with bootstrap-stage alignment and (world > 1) the
// ownership partition.  Fills g->type / level / owner / n_levels; needs no GPU.  Errors go to `ectx` (may be NULL:
// then they are readable through spf_b200_last_error(NULL)).
int plan_graph(spf_b200_ctx* ectx, const spf_params* p, spf_b200_graph* g, int world, std::vector<int>& stage) {
  const size_t n = g->nodes.size();
  g->type.resize(n);
  g->level.assign(n, -1);
  g->dptr.assign(n, nullptr);
  // ---- validation (Task::validate_inputs / validate_op, task.rs:24-179) ----
  for (size_t i = 0; i < n; i++) {
    const spf_node& nd = g->nodes[i];
    if (nd.op > SPF_OP_MUL_XN) return graph_fail(ectx, "node " + std::to_string(i) + ": unknown op " + std::to_string(nd.op));
    const OpInfo oi = op_info(nd.op);
    g->type[i] = oi.out;
    for (int e = 0; e < 3; e++) {
      const int src = nd.in[e];
      if (e < oi.n_in) {
        if (src < 0 || (size_t)src >= n)
          return graph_fail(ectx, std::string("node ") + std::to_string(i) + " (" + kOpNames[nd.op] + "): missing ciphertext input on edge " + std::to_string(e));
      } else if (src >= 0) {  // also Nop / Retire: Task::validate_inputs rejects any edge on a 0-input op (task.rs:100-118)
        return graph_fail(ectx, std::string("node ") + std::to_string(i) + " (" + kOpNames[nd.op] + "): unexpected extra input edge");
      }
    }
    if (nd.op == SPF_OP_RETIRE)  // user graphs never contain Retire (circuit_processor/mod.rs:606-611, illegal_retire_op)
      return graph_fail(ectx, "node " + std::to_string(i) + ": illegal Retire op in a user graph");
    if (nd.op == SPF_OP_SAMPLE_EXTRACT && nd.arg >= p->glwe_n)
      return graph_fail(ectx, "illegal sample extract index " + std::to_string(nd.arg));
    const bool is_io = nd.op <= SPF_OP_OUTPUT_GLEV1;
    if (is_io && !nd.io) return graph_fail(ectx, std::string("node ") + std::to_string(i) + " (" + kOpNames[nd.op] + "): io pointer is NULL");
  }
  for (size_t i = 0; i < n; i++) {
    const spf_node& nd = g->nodes[i];
    const OpInfo oi = op_info(nd.op);
    for (int e = 0; e < oi.n_in; e++) {
      if (g->type[nd.in[e]] != oi.in[e])
        return graph_fail(ectx, std::string("node ") + std::to_string(i) + " (" + kOpNames[nd.op] + "): input " + std::to_string(e) +
                                   " from node " + std::to_string(nd.in[e]) + " (" + kOpNames[g->nodes[nd.in[e]].op] + ") has the wrong ciphertext kind");
    }
  }
  // ---- levelise (iterative DFS with cycle detection) ----
  {
    std::vector<int> state(n, 0);  // 0 new, 1 on stack, 2 done
    std::vector<std::pair<int, int>> stack;
    for (size_t r = 0; r < n; r++) {
      if (state[r]) continue;
      stack.push_back({(int)r, 0});
      state[r] = 1;
      while (!stack.empty()) {
        auto& [v, e] = stack.back();
        const OpInfo oi = op_info(g->nodes[v].op);
        if (e < oi.n_in) {
          const int w = g->nodes[v].in[e++];
          if (state[w] == 1) return graph_fail(ectx, "graph has a cycle through node " + std::to_string(w));
          if (state[w] == 0) { state[w] = 1; stack.push_back({w, 0}); }
        } else {
          int lv = 0;
          for (int k = 0; k < oi.n_in; k++) lv = std::max(lv, g->level[g->nodes[v].in[k]] + 1);
          g->level[v] = lv;
          state[v] = 2;
          stack.pop_back();
        }
      }
    }
  }
  // ---- align the expensive ops ----
  // ASAP levels scatter the refresh chains (SampleExtract -> KeyswitchL1toL0 -> CircuitBootstrap)
  // between two instructions of a program over as many levels as the producing MUX tree is deep
  // (a ripple-carry adder yields one sum bit per two levels), which would run w one-ciphertext
  // bootstraps back to back.  Nodes of those three ops that have the same number of circuit
  // bootstraps upstream (their "stage") are therefore delayed to the level of the latest one, so
  // that a stage bootstraps as ONE batch; delaying a node is always legal, consumers are re-levelled.
  stage.assign(n, 0);
  {
    std::vector<int> order(n);
    for (size_t i = 0; i < n; i++) order[i] = (int)i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return g->level[a] < g->level[b]; });  // topological
    for (int v : order) {
      const OpInfo oi = op_info(g->nodes[v].op);
      for (int k = 0; k < oi.n_in; k++) {
        const int w = g->nodes[v].in[k];
        stage[v] = std::max(stage[v], stage[w] + (g->nodes[w].op == SPF_OP_CIRCUIT_BOOTSTRAP ? 1 : 0));
      }
    }
    auto slot = [&](int v) -> int {  // alignment class of node v, or -1
      switch (g->nodes[v].op) {
        case SPF_OP_SAMPLE_EXTRACT: return 3 * stage[v];
        case SPF_OP_KEYSWITCH_L1_TO_L0: return 3 * stage[v] + 1;
        case SPF_OP_CIRCUIT_BOOTSTRAP: return 3 * stage[v] + 2;
        default: return -1;
      }
    };
    int n_slots = 0;
    for (size_t i = 0; i < n; i++) n_slots = std::max(n_slots, slot((int)i) + 1);
    std::vector<int> floor_lv(n_slots, 0);
    for (int iter = 0; iter < 3 * n_slots + 2; iter++) {
      bool changed = false;
      for (int v : order) {  // re-level with the current floors (order stays topological: levels only grow
        const OpInfo oi = op_info(g->nodes[v].op);  //  along edges, and inputs precede consumers in `order`)
        int lv = 0;
        for (int k = 0; k < oi.n_in; k++) lv = std::max(lv, g->level[g->nodes[v].in[k]] + 1);
        const int sl = slot(v);
        if (sl >= 0) lv = std::max(lv, floor_lv[sl]);
        g->level[v] = lv;
      }
      for (int v : order) {
        const int sl = slot(v);
        if (sl >= 0 && g->level[v] > floor_lv[sl]) { floor_lv[sl] = g->level[v]; changed = true; }
      }
      if (!changed) break;
    }
  }
  for (size_t i = 0; i < n; i++) g->n_levels = std::max(g->n_levels, g->level[i] + 1);
  // ---- ownership (sharded graphs) ----
  // The ops between two bootstrap levels (the MUX trees and the sample-extract / keyswitch chains behind
  // them) are partitioned by connected component of their data edges: a component -- one instruction's
  // tree -- runs on ONE rank (SURVEY.md 8(e): "run each instruction's tree on one GPU and shard across
  // trees"), components are spread over the ranks stage by stage by size.  Keyswitch outputs (5 KB) are
  // all-gathered, so every circuit-bootstrap level can still be split evenly whatever produced its inputs.
  // A component whose ciphertexts are consumed by an op outside this scheme stays replicated.
  g->owner.assign(n, -1);
  if (world > 1) {
    auto local = [](uint32_t op) {
      return op == SPF_OP_CMUX || op == SPF_OP_GLEV_CMUX || op == SPF_OP_MULTIPLY_GGSW_GLWE || op == SPF_OP_NOT ||
             op == SPF_OP_GLWE_ADD || op == SPF_OP_MUL_XN || op == SPF_OP_SAMPLE_EXTRACT || op == SPF_OP_KEYSWITCH_L1_TO_L0;
    };
    std::vector<int> parent(n);
    for (size_t i = 0; i < n; i++) parent[i] = (int)i;
    auto find = [&](int v) {
      while (parent[v] != v) { parent[v] = parent[parent[v]]; v = parent[v]; }
      return v;
    };
    std::vector<char> replicated(n, 0);
    for (size_t v = 0; v < n; v++) {
      const uint32_t op = g->nodes[v].op;
      const OpInfo oi = op_info(op);
      const bool is_output = op >= SPF_OP_OUTPUT_LWE0 && op <= SPF_OP_OUTPUT_GLEV1;
      for (int e = 0; e < oi.n_in; e++) {
        const int w = g->nodes[v].in[e];
        if (!local(g->nodes[w].op)) continue;
        if (local(op)) parent[find((int)v)] = find(w);
        else if (!is_output && g->nodes[w].op != SPF_OP_KEYSWITCH_L1_TO_L0) replicated[w] = 1;
      }
    }
    struct Comp { int root, stage, first; size_t weight; bool replicated; };
    std::map<int, Comp> comps;
    for (size_t v = 0; v < n; v++) {
      if (!local(g->nodes[v].op)) continue;
      const int r = find((int)v);
      auto it = comps.find(r);
      if (it == comps.end()) it = comps.emplace(r, Comp{r, 0, (int)v, 0, false}).first;
      it->second.weight++;
      it->second.stage = std::max(it->second.stage, stage[v]);
      it->second.replicated |= replicated[v] != 0;
    }
    std::vector<Comp> list;
    for (auto& kv : comps) list.push_back(kv.second);
    std::sort(list.begin(), list.end(), [](const Comp& a, const Comp& b) {
      if (a.stage != b.stage) return a.stage < b.stage;
      if (a.weight != b.weight) return a.weight > b.weight;
      return a.first < b.first;
    });
    std::map<int, int> rank_of;
    std::vector<size_t> load(world, 0);
    int cur_stage = -1;
    for (const Comp& c : list) {
      if (c.stage != cur_stage) { cur_stage = c.stage; std::fill(load.begin(), load.end(), 0); }
      if (c.replicated) { rank_of[c.root] = -1; continue; }
      const int r = (int)(std::min_element(load.begin(), load.end()) - load.begin());
      load[r] += c.weight;
      rank_of[c.root] = r;
    }
    for (size_t v = 0; v < n; v++)
      if (local(g->nodes[v].op)) g->owner[v] = rank_of[find((int)v)];
  }
  return 0;
}

}  // namespace

extern "C" {

void spf_b200_graph_destroy(spf_b200_graph* g);
int spf_b200_graph_run_sharded(spf_b200_graph* g, int rank, int world, spf_exchange_fn exchange, void* user);
int spf_b200_graph_set_io(spf_b200_graph* g, size_t node, void* io);
int spf_b200_graph_output_rank(const spf_b200_graph* g, size_t node);

static int graph_build_sharded_impl(spf_b200_ctx* ctx, const spf_node* nodes, size_t n, int world, spf_b200_graph** out,
                                    bool box_handles);
// C++ exceptions (std::bad_alloc / length_error on a huge graph) never cross the C ABI.  `box_handles`: the rank graph
// of a box graph, whose io nodes may name box ciphertext handles (io kind 3); every other graph refuses them.
static int graph_build_checked(spf_b200_ctx* ctx, const spf_node* nodes, size_t n, int world, spf_b200_graph** out,
                               bool box_handles) {
  try {
    return graph_build_sharded_impl(ctx, nodes, n, world, out, box_handles);
  } catch (const std::exception& e) {
    return fail(ctx, SPF_E_GRAPH, std::string("graph build: ") + e.what());
  } catch (...) {
    return fail(ctx, SPF_E_GRAPH, "graph build: unknown exception");
  }
}
int spf_b200_graph_build_sharded(spf_b200_ctx* ctx, const spf_node* nodes, size_t n, int world, spf_b200_graph** out) {
  return graph_build_checked(ctx, nodes, n, world, out, false);
}
static int graph_build_sharded_impl(spf_b200_ctx* ctx, const spf_node* nodes, size_t n, int world, spf_b200_graph** out,
                                    bool box_handles) {
  if (!ctx) return SPF_E_INVALID;
  if (!out || (!nodes && n)) return fail(ctx, SPF_E_INVALID, "NULL argument");
  if (world < 1 || world > 1024) return fail(ctx, SPF_E_INVALID, "world must be in 1..1024");
  *out = nullptr;
  if (!box_handles)
    for (size_t i = 0; i < n; i++)
      if (is_box_handle(nodes[i].io))
        return fail(ctx, SPF_E_INVALID, "node " + std::to_string(i) + ": a box ciphertext handle is the io of box graphs only (spf_b200_box_graph_build)");
  const spf_params* p = &ctx->p;
  std::unique_ptr<spf_b200_graph, void (*)(spf_b200_graph*)> g(new spf_b200_graph(), spf_b200_graph_destroy);
  g->ctx = ctx;
  ctx->refs.fetch_add(1);  // released by spf_b200_graph_destroy: a graph may outlive its owner's spf_b200_destroy
  g->world = world;
  g->nodes.assign(nodes, nodes + n);
  g->io_kind.assign(n, 0);
  g->io_alloc.assign(n, 0);
  g->stage_off.assign(n, (size_t)-1);
  static const bool build_timing = getenv("SPF_B200_GRAPH_TIMING") != nullptr;
  auto now_ms = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t_start = now_ms();
  std::vector<int> stage;
  if (int rc = plan_graph(ctx, p, g.get(), world, stage)) return rc;
  const double t_plan = now_ms();
  if (int rc = ensure_constants(ctx)) return rc;
  const double t_consts = now_ms();
  // ---- groups, arena layout, pointer tables ----
  std::vector<std::vector<int>> by_level(g->n_levels);
  for (size_t i = 0; i < n; i++) by_level[g->level[i]].push_back((int)i);
  size_t arena = kArenaHeader, n_ptrs = 0, n_u32 = 0, out_stage = 0;
  auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
  std::vector<size_t> out_off, scratch_off;
  // CMux / MultiplyGgswGlwe outputs (the bulk of a MUX tree: 45 k of the 46 k nodes of a 32-bit multiply) do not get
  // a buffer each: they take a GLWE slot from a pool and give it back once the last level that reads them has
  // run.  last_use = the highest level of a consumer; ciphertexts that feed an Output node stay until the end.
  // Levels run in stream order (a programmatically launched CMUX level writes only after griddepcontrol.wait),
  // and no other rank ever stores into these slots, so a slot freed after level L can be rewritten at level L + 1.
  auto pooled = [](uint32_t op) { return op == SPF_OP_CMUX || op == SPF_OP_MULTIPLY_GGSW_GLWE; };
  g->slot.assign(n, -1);
  std::vector<int> last_use(n, -1);
  for (size_t v = 0; v < n; v++) {
    const OpInfo oi = op_info(g->nodes[v].op);
    const bool is_out = g->nodes[v].op >= SPF_OP_OUTPUT_LWE0 && g->nodes[v].op <= SPF_OP_OUTPUT_GLEV1;
    for (int e = 0; e < oi.n_in; e++) {
      const int w = g->nodes[v].in[e];
      last_use[w] = std::max(last_use[w], is_out ? g->n_levels : g->level[v]);
    }
  }
  std::vector<std::vector<int>> release_at(g->n_levels + 2);
  std::vector<int> free_slots;
  for (int lv = 0; lv < g->n_levels; lv++) {
    for (int v : release_at[lv]) free_slots.push_back(g->slot[v]);  // last read at level lv - 1
    std::map<uint32_t, std::vector<int>> ops;
    for (int id : by_level[lv]) ops[g->nodes[id].op].push_back(id);
    for (int id : by_level[lv]) {
      if (!pooled(g->nodes[id].op)) continue;
      if (free_slots.empty()) g->slot[id] = (int)g->pool_slots++;
      else { g->slot[id] = free_slots.back(); free_slots.pop_back(); }
      release_at[std::min(std::max(last_use[id], lv) + 1, g->n_levels + 1)].push_back(id);
    }
    for (auto& kv : ops) {
      const uint32_t op = kv.first;
      if (op == SPF_OP_RETIRE || op == SPF_OP_NOP) continue;
      Group G;
      G.op = op;
      G.level = lv;
      G.r_start.assign(world, 0);
      G.r_cnt.assign(world, 0);
      const OpInfo oi = op_info(op);
      const bool is_const = op >= SPF_OP_ZERO_LWE0 && op <= SPF_OP_ONE_GLEV1;
      const bool is_output = op >= SPF_OP_OUTPUT_LWE0 && op <= SPF_OP_OUTPUT_GLEV1;
      if (world == 1 || is_const || is_output || op <= SPF_OP_INPUT_GLEV1) {
        G.ids = kv.second;  // computed (or simply present) on every rank
        G.all_cnt = G.ids.size();
      } else if (op == SPF_OP_CIRCUIT_BOOTSTRAP) {
        // `world` equal chunks by index (the last ones may be short or empty), completed by an all-gather
        G.ids = kv.second;
        G.gather_chunk = cbs_chunk_items(G.ids.size(), world);
        for (int r = 0; r < world; r++) {
          G.r_start[r] = std::min(G.ids.size(), G.gather_chunk * (size_t)r);
          G.r_cnt[r] = std::min(G.ids.size() - G.r_start[r], G.gather_chunk);
        }
        G.ids.resize(G.gather_chunk * (size_t)world, -1);
      } else {
        std::vector<std::vector<int>> by_rank(world);
        std::vector<int> everyone;
        for (int id : kv.second) (g->owner[id] < 0 ? everyone : by_rank[g->owner[id]]).push_back(id);
        size_t widest = 0;
        for (auto& v : by_rank) widest = std::max(widest, v.size());
        // keyswitch outputs are all-gathered: pad every rank's share to the widest one
        const bool gather = op == SPF_OP_KEYSWITCH_L1_TO_L0 && widest > 0;
        if (gather) G.gather_chunk = widest;
        for (int r = 0; r < world; r++) {
          G.r_start[r] = G.ids.size();
          G.r_cnt[r] = by_rank[r].size();
          G.ids.insert(G.ids.end(), by_rank[r].begin(), by_rank[r].end());
          if (gather) G.ids.resize(G.r_start[r] + widest, -1);
        }
        G.all_start = G.ids.size();
        G.all_cnt = everyone.size();
        G.ids.insert(G.ids.end(), everyone.begin(), everyone.end());
      }
      size_t o = (size_t)-1, sc = (size_t)-1;
      G.slot_outputs = pooled(op);
      if (!is_const && !is_output && !G.slot_outputs) {
        o = arena;
        arena = align(arena + ct_bytes(p, oi.out) * G.ids.size());
        if (op == SPF_OP_CIRCUIT_BOOTSTRAP) { sc = arena; arena = align(arena + ct_bytes(p, T_GLWE1) * G.ids.size()); }
      }
      if (op == SPF_OP_OUTPUT_GGSW1) out_stage += ct_bytes(p, T_GGSW1) * G.ids.size();
      G.ptr_off = n_ptrs;
      G.u32_off = n_u32;
      if (G.slot_outputs) n_ptrs += 4 * G.ids.size();  // {sel, low, high} per slot, then the output pointers
      else if (op == SPF_OP_GLEV_CMUX) n_ptrs += 3 * G.ids.size();
      else if (op == SPF_OP_NOT || op == SPF_OP_GLWE_ADD || op == SPF_OP_MUL_XN) n_ptrs += 2 * G.ids.size();
      else if (oi.n_in == 1 && !is_output) n_ptrs += G.ids.size();
      if (op == SPF_OP_SAMPLE_EXTRACT || op == SPF_OP_MUL_XN) n_u32 += G.ids.size();
      out_off.push_back(o);
      scratch_off.push_back(sc);
      g->groups.push_back(std::move(G));
    }
  }
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&g->done, cudaEventDisableTiming));
  const size_t pool_off = arena;
  arena = align(arena + g->pool_slots * ct_bytes(p, T_GLWE1));
  g->arena_bytes = std::max<size_t>(arena, 256);
  const double t_layout = now_ms();
  CU(cudaMalloc(&g->arena, g->arena_bytes));
  CU(cudaMemset(g->arena, 0, kArenaHeader));
  const double t_malloc = now_ms();
  CU(cudaMalloc(&g->d_ptrs, std::max<size_t>(n_ptrs, 1) * sizeof(void*)));
  CU(cudaMalloc(&g->d_u32, std::max<size_t>(n_u32, 1) * 4));
  if (out_stage) CU(cudaMalloc(&g->d_out_stage, out_stage));
  // device addresses of every node output (groups are in level order, so producers come first)
  for (size_t gi = 0; gi < g->groups.size(); gi++) {
    Group& G = g->groups[gi];
    const OpInfo oi = op_info(G.op);
    if (out_off[gi] != (size_t)-1) G.out_base = g->arena + out_off[gi];
    if (scratch_off[gi] != (size_t)-1) G.scratch = g->arena + scratch_off[gi];
    for (size_t k = 0; k < G.ids.size(); k++) {
      const int id = G.ids[k];
      if (id < 0) continue;  // padding slot
      switch (G.op) {
        case SPF_OP_ZERO_LWE0: g->dptr[id] = ctx->c_lwe0[0]; break;
        case SPF_OP_ONE_LWE0: g->dptr[id] = ctx->c_lwe0[1]; break;
        case SPF_OP_ZERO_GLWE1: g->dptr[id] = ctx->c_glwe[0]; break;
        case SPF_OP_ONE_GLWE1: g->dptr[id] = ctx->c_glwe[1]; break;
        case SPF_OP_ZERO_GGSW1: g->dptr[id] = ctx->c_ggsw[0]; break;
        case SPF_OP_ONE_GGSW1: g->dptr[id] = ctx->c_ggsw[1]; break;
        case SPF_OP_ZERO_GLEV1: g->dptr[id] = ctx->c_glev[0]; break;
        case SPF_OP_ONE_GLEV1: g->dptr[id] = ctx->c_glev[1]; break;
        default:
          if (G.slot_outputs) g->dptr[id] = g->arena + pool_off + (size_t)g->slot[id] * ct_bytes(p, T_GLWE1);
          else if (G.out_base) g->dptr[id] = G.out_base + k * ct_bytes(p, oi.out);
      }
      const bool handle = box_handles && G.op <= SPF_OP_OUTPUT_GLEV1 && is_box_handle(g->nodes[id].io);
      if (G.op <= SPF_OP_INPUT_GLEV1) {
        g->inputs.push_back(id);
        g->io_kind[id] = handle ? 3 : (char)pin_io(g.get(), g->nodes[id].io, ct_host_bytes(p, g->type[id]));
        g->io_alloc[id] = handle ? 0 : alloc_base_of(g->nodes[id].io);
      }
      if (G.op >= SPF_OP_OUTPUT_LWE0 && G.op <= SPF_OP_OUTPUT_GLEV1) {
        g->outputs.push_back(id);
        g->io_kind[id] = handle ? 3 : (char)pin_io(g.get(), g->nodes[id].io, ct_host_bytes(p, g->type[g->nodes[id].in[0]]));
        g->io_alloc[id] = handle ? 0 : alloc_base_of(g->nodes[id].io);
      }
    }
  }
  const double t_pin = now_ms();
  std::vector<void*> h_ptrs(std::max<size_t>(n_ptrs, 1), nullptr);
  std::vector<uint32_t> h_u32(std::max<size_t>(n_u32, 1), 0);
  for (Group& G : g->groups) {
    const OpInfo oi = op_info(G.op);
    for (size_t k = 0; k < G.ids.size(); k++) {
      if (G.ids[k] < 0) continue;  // padding slot
      const spf_node& nd = g->nodes[G.ids[k]];
      switch (G.op) {
        case SPF_OP_CMUX:
        case SPF_OP_GLEV_CMUX:  // in[0] = Sel, in[1] = Low (a), in[2] = High (b): out = sel ? b : a
          h_ptrs[G.ptr_off + 3 * k + 0] = g->dptr[nd.in[0]];
          h_ptrs[G.ptr_off + 3 * k + 1] = g->dptr[nd.in[1]];
          h_ptrs[G.ptr_off + 3 * k + 2] = g->dptr[nd.in[2]];
          if (G.slot_outputs) h_ptrs[G.ptr_off + 3 * G.ids.size() + k] = g->dptr[G.ids[k]];
          break;
        case SPF_OP_MULTIPLY_GGSW_GLWE:  // in[0] = Glwe, in[1] = Ggsw
          h_ptrs[G.ptr_off + 3 * k + 0] = g->dptr[nd.in[1]];
          h_ptrs[G.ptr_off + 3 * k + 1] = nullptr;
          h_ptrs[G.ptr_off + 3 * k + 2] = g->dptr[nd.in[0]];
          h_ptrs[G.ptr_off + 3 * G.ids.size() + k] = g->dptr[G.ids[k]];
          break;
        case SPF_OP_NOT:
        case SPF_OP_MUL_XN:
          h_ptrs[G.ptr_off + 2 * k] = g->dptr[nd.in[0]];
          if (G.op == SPF_OP_MUL_XN) h_u32[G.u32_off + k] = nd.arg;
          break;
        case SPF_OP_GLWE_ADD:
          h_ptrs[G.ptr_off + 2 * k] = g->dptr[nd.in[0]];
          h_ptrs[G.ptr_off + 2 * k + 1] = g->dptr[nd.in[1]];
          break;
        default:
          if (oi.n_in == 1 && !(G.op >= SPF_OP_OUTPUT_LWE0 && G.op <= SPF_OP_OUTPUT_GLEV1)) {
            h_ptrs[G.ptr_off + k] = g->dptr[nd.in[0]];
            if (G.op == SPF_OP_SAMPLE_EXTRACT) h_u32[G.u32_off + k] = nd.arg;
          }
      }
    }
  }
  CU(cudaMemcpy(g->d_ptrs, h_ptrs.data(), h_ptrs.size() * sizeof(void*), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(g->d_u32, h_u32.data(), h_u32.size() * 4, cudaMemcpyHostToDevice));
  {  // gather tables for the outputs
    std::vector<void*> src;
    std::vector<unsigned long long> off16;
    std::vector<unsigned> n16;
    size_t total = 0;
    g->gather_off.assign(g->outputs.size(), (size_t)-1);
    for (size_t k = 0; k < g->outputs.size(); k++) {
      const int from = g->nodes[g->outputs[k]].in[0];
      if (g->type[from] == T_GGSW1) continue;
      const size_t bytes = ct_bytes(p, g->type[from]);
      g->gather_off[k] = total;
      src.push_back(g->dptr[from]);
      off16.push_back(total / 8);
      n16.push_back((unsigned)(bytes / 8));
      total += bytes;
    }
    g->gather_items = src.size();
    if (g->gather_items) {
      const size_t n_it = g->gather_items;
      CU(cudaMalloc(&g->d_gather, total));
      CU(cudaMalloc(&g->d_gather_tab, n_it * (sizeof(void*) + sizeof(unsigned long long) + sizeof(unsigned))));
      char* t = static_cast<char*>(g->d_gather_tab);
      CU(cudaMemcpy(t, src.data(), n_it * sizeof(void*), cudaMemcpyHostToDevice));
      CU(cudaMemcpy(t + n_it * sizeof(void*), off16.data(), n_it * sizeof(unsigned long long), cudaMemcpyHostToDevice));
      CU(cudaMemcpy(t + n_it * (sizeof(void*) + sizeof(unsigned long long)), n16.data(), n_it * sizeof(unsigned), cudaMemcpyHostToDevice));
    }
  }
  if (build_timing)
    fprintf(stderr, "[spf_b200 graph build] %zu nodes: plan %.1f ms, constants %.1f, layout %.1f, cudaMalloc of %.2f GB (%zu recycled CMux slots) %.1f, addresses + page-locking %zu io buffers %.1f, tables %.1f\n",
            n, t_plan - t_start, t_consts - t_plan, t_layout - t_consts, g->arena_bytes / 1e9, g->pool_slots, t_malloc - t_layout, g->inputs.size() + g->outputs.size(),
            t_pin - t_malloc, now_ms() - t_pin);
  *out = g.release();
  return 0;
}

int spf_b200_graph_build(spf_b200_ctx* ctx, const spf_node* nodes, size_t n, spf_b200_graph** out) {
  return spf_b200_graph_build_sharded(ctx, nodes, n, 1, out);
}

}  // extern "C"

namespace {

// offset of node id's ciphertext in the page-locked staging slab (kind-1 io: pageable host memory), growing the slab
int stage_slot(spf_b200_graph* g, int id, size_t bytes, char** out) {
  spf_b200_ctx* ctx = g->ctx;
  if (g->stage_off[id] == (size_t)-1) {
    size_t total = 0;
    for (size_t v = 0; v < g->nodes.size(); v++)
      if (g->io_kind[v] == 1 || (int)v == id) {
        const uint32_t op = g->nodes[v].op;
        const CtType t = op <= SPF_OP_INPUT_GLEV1 ? g->type[v] : g->type[g->nodes[v].in[0]];
        g->stage_off[v] = total;
        total += (ct_host_bytes(&ctx->p, t) + 255) & ~(size_t)255;
      }
    if (total > g->h_stage_bytes) {
      CU(cudaStreamSynchronize(g->stream));
      if (g->h_stage) CU(cudaFreeHost(g->h_stage));
      g->h_stage = nullptr;
      CU(cudaHostAlloc(reinterpret_cast<void**>(&g->h_stage), total, cudaHostAllocDefault));
      g->h_stage_bytes = total;
    }
  }
  (void)bytes;
  *out = g->h_stage + g->stage_off[id];
  return 0;
}

// Whether `rank` writes Output* node `id` into its io buffer: outputs of a MUX tree live on the tree's owner.
bool writes_output(const spf_b200_graph* g, size_t id, int rank) {
  const int r = spf_b200_graph_output_rank(g, id);
  return r == rank || (r < 0 && (g->replicated_writer < 0 || g->replicated_writer == rank));
}

// The parts of one run that are ENQUEUED on stream s (enqueue_run: inputs, every group in order, outputs).  Each
// returns the first error (message in ctx->err); work already enqueued keeps running -- the caller drains the stream.
// Input copies (and, in peer mode, the start-of-run barrier).
int enqueue_inputs(spf_b200_graph* g, bool peer_mode, cudaStream_t s) {
  spf_b200_ctx* ctx = g->ctx;
  const spf_params* p = &ctx->p;
  // every rank has finished its previous run before anyone stores into its arena again
  if (peer_mode) if (int rc = peer_barrier(g, s)) return rc;
  // inputs whose host buffers AND device buffers are consecutive (rows of one host slab, in node order) go up as one copy
  for (size_t i = 0; i < g->inputs.size();) {
    const int id0 = g->inputs[i];
    const int kind = g->io_kind[id0];
    size_t bytes = ct_host_bytes(p, g->type[id0]), j = i + 1;
    if (kind == 3) {  // box ciphertext handle: box.cuh copies it
      i = j;
      continue;
    }
    if (kind == 1) {  // pageable host buffer: through the page-locked slab
      char* st = nullptr;
      if (int rc = stage_slot(g, id0, bytes, &st)) return rc;
      memcpy(st, g->nodes[id0].io, bytes);
      CU(cudaMemcpyAsync(g->dptr[id0], st, bytes, cudaMemcpyHostToDevice, s));
      i = j;
      continue;
    }
    while (j < g->inputs.size() && g->io_kind[g->inputs[j]] == kind && g->io_alloc[id0] != 0 && g->io_alloc[g->inputs[j]] == g->io_alloc[id0] &&
           g->dptr[g->inputs[j]] == g->dptr[id0] + bytes &&
           static_cast<char*>(g->nodes[g->inputs[j]].io) == static_cast<char*>(g->nodes[id0].io) + bytes) {
      bytes += ct_host_bytes(p, g->type[g->inputs[j]]);
      j++;
    }
    CU(cudaMemcpyAsync(g->dptr[id0], g->nodes[id0].io, bytes, kind == 2 ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
    i = j;
  }
  for (int id : g->inputs) {
    const CtType t = g->type[id];
    if (t == T_GGSW1 && g->io_kind[id] < 2)  // device and box handles carry GGSWs in the device scale already
      if (int rc = launch_scale(ctx, reinterpret_cast<C2*>(g->dptr[id]), reinterpret_cast<const C2*>(g->dptr[id]),
                                spf_b200_len_ggsw_l1(p), 1.0 / 1024.0, s))
        return rc;
  }
  return 0;
}

// One group of this rank, then its exchange (circuit-bootstrap outputs (GGSW) and keyswitch outputs (L0 LWE)).
int enqueue_group(spf_b200_graph* g, const Group& G, int rank, int world, spf_exchange_fn exchange, void* user, cudaStream_t s,
                  cudaEvent_t after_group) {
  spf_b200_ctx* ctx = g->ctx;
  const bool peer_mode = world > 1 && !exchange;
  // peer mode: the scheme-switch kernel stores its GGSWs into every rank's arena while it computes them
  if (int rc = run_group(g, G, s, rank, peer_mode && G.op == SPF_OP_CIRCUIT_BOOTSTRAP ? &g->peers : nullptr)) return rc;
  if (after_group) cudaEventRecord(after_group, s);
  if (world > 1 && G.gather_chunk > 0) {
    const size_t item_bytes = ct_bytes(&ctx->p, op_info(G.op).out);
    if (!peer_mode) {
      if (int rc = exchange(user, G.out_base, G.gather_chunk * item_bytes, world, s))
        return fail(ctx, SPF_E_GRAPH, "exchange callback failed with status " + std::to_string(rc));
    } else {
      if (G.op == SPF_OP_KEYSWITCH_L1_TO_L0 && G.r_cnt[rank] > 0) {
        const size_t n16 = G.r_cnt[rank] * item_bytes / 16;
        peer_bcast_kernel<<<(unsigned)std::min<size_t>((n16 + 255) / 256, 4 * (size_t)ctx->sm_count), 256, 0, s>>>(
            reinterpret_cast<const uint4*>(G.out_base + G.r_start[rank] * item_bytes), n16, g->peers);
        if (int rc = check_launch(ctx, "peer_bcast_kernel")) return rc;
      }
      if (int rc = peer_barrier(g, s)) return rc;
    }
  }
  return 0;
}

int enqueue_outputs(spf_b200_graph* g, int rank, cudaStream_t s);

int enqueue_run(spf_b200_graph* g, int rank, int world, spf_exchange_fn exchange, void* user, cudaStream_t s,
                std::vector<cudaEvent_t>* timing_events) {
  if (int rc = enqueue_inputs(g, world > 1 && !exchange, s)) return rc;
  if (timing_events) cudaEventRecord((*timing_events)[0], s);
  size_t gi = 0;
  for (const Group& G : g->groups)
    if (int rc = enqueue_group(g, G, rank, world, exchange, user, s, timing_events ? (*timing_events)[++gi] : nullptr)) return rc;
  return enqueue_outputs(g, rank, s);
}

// Gathered and GGSW output copies of this rank.
int enqueue_outputs(spf_b200_graph* g, int rank, cudaStream_t s) {
  spf_b200_ctx* ctx = g->ctx;
  const spf_params* p = &ctx->p;
  if (g->gather_items) {
    const size_t n_it = g->gather_items;
    const char* t = static_cast<const char*>(g->d_gather_tab);
    gather_outputs_kernel<<<dim3(4, (unsigned)n_it), 256, 0, s>>>(
        reinterpret_cast<unsigned long long*>(g->d_gather), reinterpret_cast<const void* const*>(t),
        reinterpret_cast<const unsigned long long*>(t + n_it * sizeof(void*)),
        reinterpret_cast<const unsigned*>(t + n_it * (sizeof(void*) + sizeof(unsigned long long))));
    if (int rc = check_launch(ctx, "gather_outputs_kernel")) return rc;
  }
  auto mine = [&](size_t k) { return writes_output(g, (size_t)g->outputs[k], rank); };
  size_t stage = 0;
  for (size_t k = 0; k < g->outputs.size();) {
    const int id = g->outputs[k];
    const int src = g->nodes[id].in[0];
    const CtType t = g->type[src];
    const int kind = g->io_kind[id];
    if (kind == 3) {  // box ciphertext handle: box.cuh copies it
      k++;
      continue;
    }
    char* dst = static_cast<char*>(g->nodes[id].io);
    if (kind == 1 && mine(k))
      if (int rc = stage_slot(g, id, ct_host_bytes(p, t), &dst)) return rc;
    if (t == T_GGSW1) {
      char* tmp = g->d_out_stage + stage;
      stage += ct_bytes(p, T_GGSW1);
      if (mine(k)) {
        if (kind == 2) {  // device handle: the GGSW stays in HBM in the device scale
          CU(cudaMemcpyAsync(dst, g->dptr[src], ct_bytes(p, t), cudaMemcpyDeviceToDevice, s));
        } else {
          if (int rc = launch_scale(ctx, reinterpret_cast<C2*>(tmp), reinterpret_cast<const C2*>(g->dptr[src]), spf_b200_len_ggsw_l1(p), 1024.0, s))
            return rc;
          CU(cudaMemcpyAsync(dst, tmp, ct_host_bytes(p, t), cudaMemcpyDeviceToHost, s));
        }
      }
      k++;
      continue;
    }
    if (!mine(k)) { k++; continue; }
    // consecutive outputs whose host buffers are consecutive too leave in one copy
    size_t bytes = ct_host_bytes(p, t), j = k + 1;
    while (kind != 1 && j < g->outputs.size() && g->io_kind[g->outputs[j]] == kind && g->io_alloc[id] != 0 &&
           g->io_alloc[g->outputs[j]] == g->io_alloc[id] && g->gather_off[j] == g->gather_off[k] + bytes && mine(j) &&
           static_cast<char*>(g->nodes[g->outputs[j]].io) == static_cast<char*>(g->nodes[id].io) + bytes) {
      bytes += ct_host_bytes(p, g->type[g->nodes[g->outputs[j]].in[0]]);
      j++;
    }
    CU(cudaMemcpyAsync(dst, g->d_gather + g->gather_off[k], bytes, kind == 2 ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
    k = j;
  }
  return 0;
}

// After the stream has drained: staged (pageable) outputs go to their buffers.  Pure host work (also runs inside the
// stream's host-function callback of a spawned run).
void copy_out_staged(spf_b200_graph* g, int rank) {
  const spf_params* p = &g->ctx->p;
  for (size_t k = 0; k < g->outputs.size(); k++) {
    const int id = g->outputs[k];
    if (g->io_kind[id] != 1 || g->stage_off[id] == (size_t)-1) continue;
    if (!writes_output(g, (size_t)id, rank)) continue;
    memcpy(g->nodes[id].io, g->h_stage + g->stage_off[id], ct_host_bytes(p, g->type[g->nodes[id].in[0]]));
  }
}

void CUDART_CB spawn_done(void* arg) {
  SpawnRecord* rec = static_cast<SpawnRecord*>(arg);
  spf_b200_graph* g = rec->g;
  if (rec->status == 0) copy_out_staged(g, 0);
  spf_b200_ctx* ctx = g->ctx;
  {
    std::lock_guard<std::mutex> lk(ctx->fc_mu);
    ctx->in_flight--;
  }
  ctx->fc_cv.notify_all();
  if (rec->cb) rec->cb(rec->user, rec->status, rec->status ? rec->msg.c_str() : nullptr);
  delete rec;
}

}  // namespace

extern "C" {

// Executes the graph once: copies every Input* ciphertext from its io pointer, runs the levels,
// copies every Output* ciphertext to its io pointer, and returns when the outputs are valid
// (CircuitProcessor::run_graph_blocking, circuit_processor/mod.rs:641-655).
// Sharded over `world` ranks (one process per GPU, every rank runs the same graph on the same
// inputs): each CircuitBootstrap group -- the only expensive ops -- is split into `world` equal
// chunks, rank r bootstraps chunk r, then `exchange` (an all-gather over NVLink, see
// spf_b200/multi.py) or the peer-memory stores complete the group's GGSWs on every rank; MUX trees run on their
// owner ranks.  A failure after the first enqueue drains the stream before returning (the caller's io buffers are
// not touched afterwards); in peer mode it also leaves the ranks' barrier epochs out of step, so the graph is
// marked poisoned and must be rebuilt.
int spf_b200_graph_run_sharded(spf_b200_graph* g, int rank, int world, spf_exchange_fn exchange, void* user) {
  if (!g) return SPF_E_INVALID;
  spf_b200_ctx* ctx = g->ctx;
  if (world != g->world || rank < 0 || rank >= world)
    return fail(ctx, SPF_E_INVALID, "rank/world do not match the graph's sharded layout");
  const bool peer_mode = world > 1 && !exchange;
  if (peer_mode && (!g->peers_set || g->peer_rank != rank))
    return fail(ctx, SPF_E_INVALID, "a sharded run needs an exchange callback or opened peer arenas (spf_b200_graph_open_peers)");
  if (g->poisoned)
    return fail(ctx, SPF_E_GRAPH, "an earlier peer-memory run of this graph failed: the ranks' barrier epochs disagree, rebuild the graphs");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t s = g->stream;
  const uint64_t l0 = ctx->launches.load();
  // SPF_B200_GRAPH_TIMING=1: CUDA events around every group, per-op totals on stderr (diagnostics only;
  // the events serialise nothing but do defeat the programmatic overlap between CMUX levels)
  static const bool timing = getenv("SPF_B200_GRAPH_TIMING") != nullptr;
  std::vector<cudaEvent_t> ev;
  if (timing) {
    ev.resize(g->groups.size() + 1);
    for (auto& e : ev) cudaEventCreate(&e);
  }
  int rc = enqueue_run(g, rank, world, exchange, user, s, timing ? &ev : nullptr);
  const std::string msg = rc ? ctx->err : std::string();
  const cudaError_t se = cudaStreamSynchronize(s);  // also on failure: nothing of this run is in flight afterwards
  cudaEventRecord(g->done, s);
  if (rc == 0 && se != cudaSuccess) rc = fail(ctx, SPF_E_CUDA, std::string("graph run: ") + cudaGetErrorString(se));
  else if (rc) ctx->err = msg;
  if (rc == 0) copy_out_staged(g, rank);
  if (rc == 0 && peer_mode) {
    int err = 0;
    if (cudaMemcpy(&err, g->arena + 2048, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) err = 1;
    if (err) {
      cudaMemset(g->arena + 2048, 0, sizeof(int));
      rc = fail(ctx, SPF_E_GRAPH, "peer barrier timed out: a rank of the sharded run did not arrive");
    }
  }
  if (rc && peer_mode) g->poisoned = true;
  if (timing && rc == 0) {
    std::map<uint32_t, std::pair<double, size_t>> per_op;
    std::map<uint32_t, size_t> groups_of;
    for (size_t k = 0; k < g->groups.size(); k++) {
      float ms = 0;
      cudaEventElapsedTime(&ms, ev[k], ev[k + 1]);
      per_op[g->groups[k].op].first += ms;
      per_op[g->groups[k].op].second += g->groups[k].ids.size();
      groups_of[g->groups[k].op]++;
    }
    for (auto& kv : per_op)
      fprintf(stderr, "[spf_b200 graph] %-18s %6zu groups %8zu nodes %9.3f ms\n", kOpNames[kv.first], groups_of[kv.first], kv.second.second, kv.second.first);
  }
  for (auto& e : ev) cudaEventDestroy(e);
  g->status.store(rc);
  g->launches_per_run = ctx->launches.load() - l0;
  return rc;
}

// ---- asynchronous execution: CircuitProcessor::spawn_graph + CompletionHandler + flow control -------------------------
// (circuit_processor/mod.rs:130-253,573-623; completion_handler.rs:14-56).  The whole run is enqueued on the graph's own
// stream and the call returns; `on_complete(user, status, message)` fires exactly once when every op has retired, with
// the FIRST error of the run (0 = none).  A run whose dependency failed retires as a no-op with that error, as tasks
// do after CompletionHandler::error is set.  At most spf_b200_set_max_in_flight graphs are between dispatch and
// completion: further spawns block in the caller, as dispatch() blocks on the flow-control channel.  `after`: graphs
// whose LAST spawned run must complete first (stream-ordered on the device, no host wait) -- with device handles as
// io buffers (see spf_b200_graph_set_io) graph k + 1 consumes graph k's outputs without leaving HBM.
// The callback runs on a CUDA-internal thread: it must not call CUDA or spf_b200 functions.
int spf_b200_graph_spawn(spf_b200_graph* g, spf_b200_graph* const* after, size_t n_after, spf_completion_fn on_complete, void* user) {
  if (!g) return SPF_E_INVALID;
  spf_b200_ctx* ctx = g->ctx;
  if (g->world != 1) return fail(ctx, SPF_E_INVALID, "spawn: sharded graphs run through spf_b200_graph_run_sharded");
  if (n_after && !after) return fail(ctx, SPF_E_INVALID, "spawn: NULL dependency list");
  CU(cudaSetDevice(ctx->device));
  {
    std::unique_lock<std::mutex> lk(ctx->fc_mu);
    ctx->fc_cv.wait(lk, [&] { return ctx->in_flight < ctx->max_in_flight; });
    ctx->in_flight++;
  }
  // the staging slab of pageable io buffers is reused by the next run: wait for the previous one
  bool staged = false;
  for (char k : g->io_kind) staged |= k == 1;
  if (staged) cudaEventSynchronize(g->done);
  SpawnRecord* rec = new SpawnRecord{g, on_complete, user, 0, std::string()};
  for (size_t i = 0; i < n_after && rec->status == 0; i++) {
    spf_b200_graph* d = after[i];
    if (!d || d == g) continue;
    if (const int ds = d->status.load()) {
      rec->status = ds;
      rec->msg = "a dependency of this graph failed: " + d->status_msg;
    } else if (cudaStreamWaitEvent(g->stream, d->done, 0) != cudaSuccess) {
      rec->status = SPF_E_CUDA;
      rec->msg = "cudaStreamWaitEvent on a dependency failed";
    }
  }
  if (rec->status == 0) {
    if (const int rc = enqueue_run(g, 0, 1, nullptr, nullptr, g->stream, nullptr)) {
      rec->status = rc;
      rec->msg = ctx->err;
    }
  }
  g->status.store(rec->status);
  g->status_msg = rec->msg;
  const cudaError_t e = cudaLaunchHostFunc(g->stream, spawn_done, rec);
  cudaEventRecord(g->done, g->stream);
  if (e != cudaSuccess) {  // could not even enqueue the completion: deliver it here
    cudaStreamSynchronize(g->stream);
    rec->status = rec->status ? rec->status : SPF_E_CUDA;
    if (rec->msg.empty()) rec->msg = std::string("cudaLaunchHostFunc: ") + cudaGetErrorString(e);
    spawn_done(rec);
  }
  return 0;
}

// Blocks until the last run of the graph (spawned or blocking) has completed, callback included; returns its status.
int spf_b200_graph_wait(spf_b200_graph* g) {
  if (!g) return SPF_E_INVALID;
  spf_b200_ctx* ctx = g->ctx;
  CU(cudaSetDevice(ctx->device));
  CU(cudaEventSynchronize(g->done));
  return g->status.load();
}

// message of the error latched by the graph's last spawned run ("" when it succeeded)
const char* spf_b200_graph_status_message(const spf_b200_graph* g) { return g ? g->status_msg.c_str() : ""; }

int spf_b200_set_max_in_flight(spf_b200_ctx* ctx, int n) {
  if (!ctx) return SPF_E_INVALID;
  if (n < 1) return fail(ctx, SPF_E_INVALID, "max_in_flight must be at least 1");
  {
    std::lock_guard<std::mutex> lk(ctx->fc_mu);
    ctx->max_in_flight = n;
  }
  ctx->fc_cv.notify_all();
  return 0;
}

void spf_b200_graph_destroy(spf_b200_graph* g) {
  if (!g) return;
  spf_b200_ctx* ctx = g->ctx;
  cudaSetDevice(ctx->device);
  if (g->stream) cudaStreamSynchronize(g->stream);  // a spawned run may still be in flight
  for (void* q : g->ipc_opened) cudaIpcCloseMemHandle(q);
  cudaFree(g->arena);
  cudaFree(g->d_ptrs);
  cudaFree(g->d_u32);
  cudaFree(g->d_out_stage);
  cudaFree(g->d_gather);
  cudaFree(g->d_gather_tab);
  cudaFree(g->ks_states.p);
  if (g->h_stage) cudaFreeHost(g->h_stage);
  for (void* q : g->pinned) cudaHostUnregister(q);
  if (g->done) cudaEventDestroy(g->done);
  if (g->stream) cudaStreamDestroy(g->stream);
  delete g;
  spf_b200_destroy(ctx);  // drops the graph's reference; frees the context if its owner is gone already
}

int spf_b200_graph_run(spf_b200_graph* g) {
  if (!g) return SPF_E_INVALID;
  if (g->world != 1) return fail(g->ctx, SPF_E_INVALID, "graph was built sharded: use spf_b200_graph_run_sharded");
  return spf_b200_graph_run_sharded(g, 0, 1, nullptr, nullptr);
}

// Re-points the io buffer of an Input*/Output* node, so that one built (validated, levelised, device-
// resident) graph serves every invocation of the same instruction shape: the reference rebuilds the
// MUX circuit and re-levelises on every instruction dispatch (fhe_circuit.rs:473-494, SURVEY.md 8(f).3).
// The buffer may be page-locked host memory (plain DMA), pageable host memory (copied through the graph's own
// page-locked slab: no cudaHostRegister per call) or DEVICE memory (a ciphertext handle: device-to-device copy, GGSWs
// in the device scale) -- detected with cudaPointerGetAttributes.
int spf_b200_graph_set_io(spf_b200_graph* g, size_t node, void* io) {
  if (!g) return SPF_E_INVALID;
  if (node >= g->nodes.size() || g->nodes[node].op > SPF_OP_OUTPUT_GLEV1)
    return fail(g->ctx, SPF_E_INVALID, "set_io: node " + std::to_string(node) + " is not an Input*/Output* node");
  if (!io) return fail(g->ctx, SPF_E_INVALID, "set_io: io pointer is NULL");
  if (is_box_handle(io))
    return fail(g->ctx, SPF_E_INVALID, "set_io: a box ciphertext handle is the io of box graphs only (spf_b200_box_graph_set_io)");
  void* old = g->nodes[node].io;
  if (old == io) return 0;
  cudaSetDevice(g->ctx->device);
  auto it = std::find(g->pinned.begin(), g->pinned.end(), old);
  if (it != g->pinned.end()) {
    bool shared = false;  // several nodes may read the same registered buffer
    for (size_t v = 0; v < g->nodes.size(); v++) shared |= v != node && g->nodes[v].op <= SPF_OP_OUTPUT_GLEV1 && g->nodes[v].io == old;
    if (!shared) { cudaStreamSynchronize(g->stream); cudaHostUnregister(old); g->pinned.erase(it); }
  }
  g->nodes[node].io = io;
  const uint32_t op = g->nodes[node].op;
  const CtType t = op <= SPF_OP_INPUT_GLEV1 ? g->type[node] : g->type[g->nodes[node].in[0]];
  g->io_kind[node] = (char)pin_io(g, io, ct_host_bytes(&g->ctx->p, t), /*may_register=*/false);
  g->io_alloc[node] = alloc_base_of(io);
  return 0;
}

// Rank on which a sharded run delivers the ciphertext of Output* node `node`: -1 = on every rank (the
// producer is replicated or all-gathered: inputs, constants, circuit bootstraps, keyswitches), else the rank
// that owns the producing MUX tree.  -2 for a bad argument.
int spf_b200_graph_output_rank(const spf_b200_graph* g, size_t node) {
  if (!g || node >= g->nodes.size()) return -2;
  const uint32_t op = g->nodes[node].op;
  if (op < SPF_OP_OUTPUT_LWE0 || op > SPF_OP_OUTPUT_GLEV1) return -2;
  const int src = g->nodes[node].in[0];
  return g->nodes[src].op == SPF_OP_KEYSWITCH_L1_TO_L0 ? -1 : g->owner[src];
}

// Page-locked host memory for ciphertext buffers (one slab for many ciphertexts): graph IO from such memory is a
// true DMA without per-buffer registration.  No context needed; errors through spf_b200_last_error(NULL).
int spf_b200_host_alloc(void** out, size_t bytes) {
  if (!out || !bytes) return fail(nullptr, SPF_E_INVALID, "host_alloc: NULL / empty");
  *out = nullptr;
  const cudaError_t e = cudaHostAlloc(out, bytes, cudaHostAllocPortable);
  if (e != cudaSuccess) return fail(nullptr, SPF_E_CUDA, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
  return 0;
}
int spf_b200_device_alloc(spf_b200_ctx* ctx, void** out, size_t bytes) {
  if (!ctx) return SPF_E_INVALID;
  if (!out || !bytes) return fail(ctx, SPF_E_INVALID, "device_alloc: NULL / empty");
  *out = nullptr;
  CU(cudaSetDevice(ctx->device));
  CU(cudaMalloc(out, bytes));
  return 0;
}
int spf_b200_device_free(spf_b200_ctx* ctx, void* p) {
  if (!ctx) return SPF_E_INVALID;
  if (!p) return 0;
  CU(cudaSetDevice(ctx->device));
  CU(cudaFree(p));
  return 0;
}
int spf_b200_host_free(void* p) {
  if (!p) return 0;
  const cudaError_t e = cudaFreeHost(p);
  return e == cudaSuccess ? 0 : fail(nullptr, SPF_E_CUDA, std::string("cudaFreeHost: ") + cudaGetErrorString(e));
}

// ---- peer-memory exchange: the arenas of all ranks mapped into every process (CUDA IPC over NVLink) ----
void* spf_b200_graph_arena(const spf_b200_graph* g) { return g ? g->arena : nullptr; }

int spf_b200_graph_ipc_handle(spf_b200_graph* g, uint8_t* handle_out) {
  if (!g) return SPF_E_INVALID;
  if (!handle_out) return fail(g->ctx, SPF_E_INVALID, "NULL argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  spf_b200_ctx* ctx = g->ctx;
  CU(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, g->arena));
  memcpy(handle_out, &h, 64);
  return 0;
}

// arenas[r] = rank r's arena as addressable from THIS process (arenas[rank] is ignored); all ranks must have built
// the same graph with the same `world`, so that a ciphertext sits at the same offset in every arena.
int spf_b200_graph_set_peers(spf_b200_graph* g, int rank, int world, void* const* arenas) {
  if (!g) return SPF_E_INVALID;
  if (!arenas || world != g->world || rank < 0 || rank >= world || world - 1 > kMaxPeers)
    return fail(g->ctx, SPF_E_INVALID, "set_peers: rank/world do not match the graph (at most 8 ranks)");
  g->peers.n = 0;
  for (int r = 0; r < world; r++) {
    if (r == rank) continue;
    if (!arenas[r]) return fail(g->ctx, SPF_E_INVALID, "set_peers: NULL arena");
    g->peers.rank_of[g->peers.n] = r;
    g->peers.off[g->peers.n] = (long long)(static_cast<char*>(arenas[r]) - g->arena);
    g->peers.n++;
  }
  g->peer_rank = rank;
  g->peers_set = true;
  return 0;
}

// handles: world x 64 bytes, handles[r] = spf_b200_graph_ipc_handle of rank r's graph (gathered by the host, e.g.
// with torch.distributed.all_gather_object); opens every peer arena with peer access enabled.
int spf_b200_graph_open_peers(spf_b200_graph* g, int rank, int world, const uint8_t* handles) {
  if (!g) return SPF_E_INVALID;
  if (!handles || world != g->world || rank < 0 || rank >= world || world - 1 > kMaxPeers)
    return fail(g->ctx, SPF_E_INVALID, "open_peers: rank/world do not match the graph (at most 8 ranks)");
  spf_b200_ctx* ctx = g->ctx;
  CU(cudaSetDevice(ctx->device));
  std::vector<void*> arenas(world, nullptr);
  for (int r = 0; r < world; r++) {
    if (r == rank) { arenas[r] = g->arena; continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + 64 * (size_t)r, 64);
    void* q = nullptr;
    CU(cudaIpcOpenMemHandle(&q, h, cudaIpcMemLazyEnablePeerAccess));
    g->ipc_opened.push_back(q);
    arenas[r] = q;
  }
  return spf_b200_graph_set_peers(g, rank, world, arenas.data());
}

// Host-only planning (no GPU, no context): the validation, levelisation and ownership partition of
// spf_b200_graph_build_sharded, for hosts that want to inspect or test a schedule.
static int graph_plan_impl(const spf_params* params, const spf_node* nodes, size_t n, int world, int32_t* level_out, int32_t* owner_out);
int spf_b200_graph_plan(const spf_params* params, const spf_node* nodes, size_t n, int world, int32_t* level_out, int32_t* owner_out) {
  try {
    return graph_plan_impl(params, nodes, n, world, level_out, owner_out);
  } catch (const std::exception& e) {
    return fail(nullptr, SPF_E_GRAPH, std::string("graph plan: ") + e.what());
  } catch (...) {
    return fail(nullptr, SPF_E_GRAPH, "graph plan: unknown exception");
  }
}
static int graph_plan_impl(const spf_params* params, const spf_node* nodes, size_t n, int world, int32_t* level_out, int32_t* owner_out) {
  if (!params || (!nodes && n)) return fail(nullptr, SPF_E_INVALID, "NULL argument");
  if (world < 1 || world > 1024) return fail(nullptr, SPF_E_INVALID, "world must be in 1..1024");
  spf_b200_graph g;
  g.world = world;
  g.nodes.assign(nodes, nodes + n);
  std::vector<int> stage;
  if (int rc = plan_graph(nullptr, params, &g, world, stage)) return rc;
  for (size_t i = 0; i < n; i++) {
    if (level_out) level_out[i] = g.level[i];
    if (owner_out) owner_out[i] = g.owner[i];
  }
  return 0;
}

int spf_b200_graph_levels(const spf_b200_graph* g) { return g ? g->n_levels : -1; }
uint64_t spf_b200_graph_launches(const spf_b200_graph* g) { return g ? g->launches_per_run : 0; }

int spf_b200_run_graph(spf_b200_ctx* ctx, const spf_node* nodes, size_t n) {
  spf_b200_graph* g = nullptr;
  if (int rc = spf_b200_graph_build(ctx, nodes, n, &g)) return rc;
  const int rc = spf_b200_graph_run(g);
  spf_b200_graph_destroy(g);
  return rc;
}

}  // extern "C"
