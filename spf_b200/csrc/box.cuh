// box.cuh -- the GPUs of one box behind one handle (include/spf_b200.h: spf_b200_box_*), included by capi.cu after
// graph.cuh.  One process, one dispatching thread: a rank is a context on its own device; the compute key is uploaded
// once and replicated device to device; host-pointer ops split the batch over the ranks and run them concurrently on
// one worker thread per rank; a box graph is a sharded graph per rank, wired to the other ranks' arenas in-process,
// and every rank's run is enqueued from the calling thread, level by level across the ranks.  A box graph runs on an
// ordered subset of the box's ranks, its MEMBERS (all ranks in order by default): member i runs shard i of the graph
// sharded over the members.  A box ciphertext handle holds one replica of a ciphertext per rank of the box, so that box
// graphs hand their outputs to the next graph in HBM, whichever ranks either graph runs on.
#include <array>
#include <functional>
#include <thread>

struct spf_b200_box {
  int n = 0;
  std::vector<int> device;
  std::vector<spf_b200_ctx*> ctx;
  std::string err;
  double replication_ms = 0;
  // lifetime: box graphs keep the box alive (its flow control and error slot), as graphs keep their context
  std::atomic<int> refs{1};
  FlowControl fc;  // of the spawned runs of this box's graphs
  // one worker thread per rank for the host-pointer ops: created with the box, joined by spf_b200_box_destroy
  std::vector<std::thread> workers;
  std::mutex w_mu;
  std::condition_variable w_job, w_done;
  std::vector<std::function<int()>> jobs;
  std::vector<int> job_rc;
  int pending = 0;
  bool stop = false;
};

// One ciphertext kept in HBM, one replica per rank on that rank's device (a device that appears twice gets two).
// GGSWs are stored in the device scale (2^-10).  Reference-counted: the caller's reference and one per box graph node
// bound to it; the handle holds a reference on its box.
struct spf_b200_box_ciphertext {
  spf_b200_box* box = nullptr;
  uint32_t kind = 0;  // the Input* op code of the ciphertext type
  size_t bytes = 0;
  std::vector<char*> rep;  // rank r's replica
  std::atomic<int> refs{1};
};

struct spf_b200_box_graph {
  spf_b200_box* box = nullptr;
  std::vector<int> rank;           // member i's box rank
  std::vector<spf_b200_graph*> g;  // member i's sharded graph (shard i of rank.size()), on box rank rank[i]'s context
  std::vector<spf_b200_box_ciphertext*> bound;  // per node: the box ciphertext handle bound to it (a reference), or NULL
  std::vector<void*> pinned;       // host io buffers page-locked (portable: every device DMAs them) by this box graph
  int* h_err = nullptr;            // page-locked copy of every member's barrier error word, read by the completion
  RunState run;
};

namespace {

int box_fail(spf_b200_box* b, int code, const std::string& msg) {
  if (b) b->err = msg;
  else g_create_err = msg;
  return code;
}

#define BCU(b, call)                                                                      \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess) return box_fail(b, SPF_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

// The contiguous split of multi.shard: the first batch % n ranks get one extra item.
void box_shard(size_t batch, int n, int rank, size_t* start, size_t* count) {
  const size_t base = batch / (size_t)n, extra = batch % (size_t)n;
  *start = (size_t)rank * base + std::min((size_t)rank, extra);
  *count = base + ((size_t)rank < extra ? 1 : 0);
}

void box_worker(spf_b200_box* b, int r) {
  std::unique_lock<std::mutex> lk(b->w_mu);
  for (;;) {
    b->w_job.wait(lk, [&] { return b->stop || b->jobs[r]; });
    if (b->stop) return;
    std::function<int()> job = std::move(b->jobs[r]);
    b->jobs[r] = nullptr;
    lk.unlock();
    const int rc = job();
    lk.lock();
    b->job_rc[r] = rc;
    if (--b->pending == 0) b->w_done.notify_all();
  }
}

// Runs op(ctx, start, count) for every rank's slice of the batch, all ranks at once on their worker threads; returns
// when every rank is done, with the first failing rank's error.
int box_each(spf_b200_box* b, size_t batch, const std::function<int(spf_b200_ctx*, size_t, size_t)>& op) {
  {
    std::lock_guard<std::mutex> lk(b->w_mu);
    for (int r = 0; r < b->n; r++) {
      size_t start, count;
      box_shard(batch, b->n, r, &start, &count);
      b->job_rc[r] = 0;
      if (count == 0) continue;
      spf_b200_ctx* c = b->ctx[r];
      b->jobs[r] = [c, start, count, &op] { return op(c, start, count); };
      b->pending++;
    }
  }
  b->w_job.notify_all();
  std::unique_lock<std::mutex> lk(b->w_mu);
  b->w_done.wait(lk, [&] { return b->pending == 0; });
  for (int r = 0; r < b->n; r++)
    if (b->job_rc[r]) return box_fail(b, b->job_rc[r], "rank " + std::to_string(r) + ": " + spf_b200_last_error(b->ctx[r]));
  return 0;
}

void box_release(spf_b200_box* b) {
  if (b->refs.fetch_sub(1) == 1) delete b;
}

void box_ciphertext_delete(spf_b200_box_ciphertext* h) {
  for (size_t r = 0; r < h->rep.size(); r++) {
    if (!h->rep[r]) continue;
    cudaSetDevice(h->box->device[r]);
    cudaFree(h->rep[r]);
  }
  box_release(h->box);
  delete h;
}

// Drops one reference; the last one unregisters the handle and frees its replicas.  A spawned run of a graph that was
// rebound to another buffer may still read or write a replica (owners write the replicas of every rank), so every
// device of the box finishes its work first.
void box_ciphertext_release(spf_b200_box_ciphertext* h) {
  if (!h || h->refs.fetch_sub(1) != 1) return;
  {
    std::lock_guard<std::mutex> lk(g_box_handles_mu);
    g_box_handles.erase(h);
  }
  std::vector<int> devs = h->box->device;
  std::sort(devs.begin(), devs.end());
  devs.erase(std::unique(devs.begin(), devs.end()), devs.end());
  for (int d : devs) {
    cudaSetDevice(d);
    cudaDeviceSynchronize();
  }
  box_ciphertext_delete(h);
}

// A box ciphertext handle named by io node `node` (op `op`) of a box graph on box b: SPF_E_INVALID unless it belongs to
// b, the node is an Input* / Output* node and the handle holds the node's ciphertext type.
int check_box_handle(spf_b200_box* b, const spf_b200_box_ciphertext* h, size_t node, uint32_t op) {
  const std::string at = "box graph: node " + std::to_string(node);
  if (op > SPF_OP_OUTPUT_GLEV1)
    return box_fail(b, SPF_E_INVALID, at + " (" + (op <= SPF_OP_MUL_XN ? kOpNames[op] : "unknown op") +
                                          ") takes no io; box ciphertext handles bind Input* and Output* nodes");
  if (h->box != b) return box_fail(b, SPF_E_INVALID, at + ": the box ciphertext handle belongs to another box");
  if (op % 5 != h->kind)
    return box_fail(b, SPF_E_INVALID, at + " (" + kOpNames[op] + "): the box ciphertext handle holds a " +
                                          (kOpNames[h->kind] + 5) + " ciphertext, a kind mismatch");
  return 0;
}

// One or more box_copy_kernel launches over `items` (at most kBoxCopyLarge per launch).
template <int N>
int launch_box_copy_chunk(spf_b200_ctx* ctx, const BoxCopyItem* items, size_t cnt, cudaStream_t s) {
  BoxCopyTable<N> t{};
  unsigned widest = 0;
  for (size_t i = 0; i < cnt; i++) {
    t.item[i] = items[i];
    widest = std::max(widest, items[i].n8);
  }
  const unsigned gx = std::min(32u, std::max(1u, (widest / 2 + 255) / 256));
  box_copy_kernel<N><<<dim3(gx, (unsigned)cnt), 256, 0, s>>>(t);
  return check_launch(ctx, "box_copy_kernel");
}

int launch_box_copy(spf_b200_ctx* ctx, const std::vector<BoxCopyItem>& items, cudaStream_t s) {
  for (size_t i = 0; i < items.size(); i += kBoxCopyLarge) {
    const size_t cnt = std::min(items.size() - i, (size_t)kBoxCopyLarge);
    if (int rc = cnt <= (size_t)kBoxCopySmall ? launch_box_copy_chunk<kBoxCopySmall>(ctx, items.data() + i, cnt, s)
                                              : launch_box_copy_chunk<kBoxCopyLarge>(ctx, items.data() + i, cnt, s))
      return rc;
  }
  return 0;
}

// Member i's handle traffic of one run, enqueued on its stream: inputs copy the replica of the member's box rank into
// its arena.  Outputs reach the replicas of EVERY rank of the box, members or not: an output every member holds
// (output rank -1) goes from each member to its own replica, and from member 0 also to the replicas of the ranks
// outside the graph; an output of a MUX tree goes from its owner member to every replica.
int enqueue_handle_copies(spf_b200_box_graph* bg, int i, bool outputs) {
  spf_b200_graph* g = bg->g[i];
  const int n_box = bg->box->n;
  std::vector<char> member(n_box, 0);
  for (int r : bg->rank) member[r] = 1;
  std::vector<BoxCopyItem> items;
  for (int id : outputs ? g->outputs : g->inputs) {
    if (g->io_kind[id] != 3) continue;
    const spf_b200_box_ciphertext* h = static_cast<const spf_b200_box_ciphertext*>(g->nodes[id].io);
    BoxCopyItem it{};
    it.n8 = (unsigned)(h->bytes / 8);
    if (!outputs) {
      it.src = reinterpret_cast<const unsigned long long*>(h->rep[bg->rank[i]]);
      it.dst[it.n_dst++] = reinterpret_cast<unsigned long long*>(g->dptr[id]);
    } else {
      const int owner = spf_b200_graph_output_rank(g, id);
      if (owner >= 0 && owner != i) continue;
      it.src = reinterpret_cast<const unsigned long long*>(g->dptr[g->nodes[id].in[0]]);
      for (int q = 0; q < n_box; q++)
        if (owner >= 0 || q == bg->rank[i] || (i == 0 && !member[q]))
          it.dst[it.n_dst++] = reinterpret_cast<unsigned long long*>(h->rep[q]);
    }
    items.push_back(it);
  }
  if (items.empty()) return 0;
  return launch_box_copy(g->ctx, items, g->stream);
}

int box_create_impl(const spf_params* params, const double* bsk, size_t bsk_len, const uint64_t* ksk, size_t ksk_len,
                    const double* ssk, size_t ssk_len, const double* ak, size_t ak_len, const int* devices, int n,
                    spf_b200_box** out) {
  if (!out) return box_fail(nullptr, SPF_E_INVALID, "out is NULL");
  *out = nullptr;
  if (n < 1 || n > kMaxPeers + 1) return box_fail(nullptr, SPF_E_INVALID, "box: n must be in 1..8 (a rank has at most 7 peers)");
  if (!devices) return box_fail(nullptr, SPF_E_INVALID, "box: devices is NULL");
  if (int rc = validate_params(params)) return rc;
  if (!bsk || !ksk || !ssk || !ak) return box_fail(nullptr, SPF_E_INVALID, "NULL key array");
  if (bsk_len != spf_b200_len_bsk(params) || ksk_len != spf_b200_len_ksk(params) ||
      ssk_len != spf_b200_len_ssk(params) || ak_len != spf_b200_len_ak(params))
    return box_fail(nullptr, SPF_E_INVALID, "key length does not match params (ComputeKey::check_is_valid, keys.rs:190-206)");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return box_fail(nullptr, SPF_E_CUDA, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
  for (int r = 0; r < n; r++)
    if (devices[r] < 0 || devices[r] >= ndev) return box_fail(nullptr, SPF_E_INVALID, "box: device index out of range");
  // distinct devices exchange GGSWs and barrier flags through each other's memory: peer access both ways
  std::vector<int> uniq(devices, devices + n);
  std::sort(uniq.begin(), uniq.end());
  uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
  for (int a : uniq)
    for (int c : uniq) {
      if (a == c) continue;
      int ok = 0;
      BCU(nullptr, cudaDeviceCanAccessPeer(&ok, a, c));
      if (!ok)
        return box_fail(nullptr, SPF_E_UNSUPPORTED, "box: device " + std::to_string(a) + " cannot access device " + std::to_string(c) + " as a peer");
    }
  for (int a : uniq) {
    BCU(nullptr, cudaSetDevice(a));
    for (int c : uniq) {
      if (a == c) continue;
      const cudaError_t pe = cudaDeviceEnablePeerAccess(c, 0);
      if (pe == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
      else if (pe != cudaSuccess) return box_fail(nullptr, SPF_E_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(pe));
    }
  }
  // The compute key crosses PCIe once, to rank 0; rank r + s receives it from rank r in step s = 1, 2, 4, ... over
  // NVLink.  Each rank's context is then made from its replica exactly as spf_b200_create_from_device does.
  const size_t bytes[4] = {bsk_len * 16, ksk_len * 8, ssk_len * 16, ak_len * 16};
  const void* host[4] = {bsk, ksk, ssk, ak};
  std::vector<std::array<void*, 4>> rep(n, std::array<void*, 4>{nullptr, nullptr, nullptr, nullptr});
  std::vector<cudaStream_t> st(n, nullptr);
  std::unique_ptr<spf_b200_box> b(new spf_b200_box());
  b->n = n;
  b->device.assign(devices, devices + n);
  b->ctx.assign(n, nullptr);
  auto cleanup = [&] {
    for (int r = 0; r < n; r++) {
      cudaSetDevice(devices[r]);
      if (st[r]) { cudaStreamSynchronize(st[r]); cudaStreamDestroy(st[r]); st[r] = nullptr; }
      for (void*& q : rep[r]) { cudaFree(q); q = nullptr; }
    }
  };
  auto fail_all = [&](int rc, const std::string& msg) {
    cleanup();
    for (spf_b200_ctx* c : b->ctx) spf_b200_destroy(c);
    return box_fail(nullptr, rc, msg);
  };
#define BOX_CU(call)                                                                        \
  do {                                                                                      \
    cudaError_t e_ = (call);                                                                \
    if (e_ != cudaSuccess) return fail_all(SPF_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)
  for (int r = 0; r < n; r++) {
    BOX_CU(cudaSetDevice(devices[r]));
    BOX_CU(cudaStreamCreateWithFlags(&st[r], cudaStreamNonBlocking));
    for (int k = 0; k < 4; k++) BOX_CU(cudaMalloc(&rep[r][k], bytes[k]));
  }
  BOX_CU(cudaSetDevice(devices[0]));
  for (int k = 0; k < 4; k++) BOX_CU(cudaMemcpyAsync(rep[0][k], host[k], bytes[k], cudaMemcpyHostToDevice, st[0]));
  BOX_CU(cudaStreamSynchronize(st[0]));
  const auto t0 = std::chrono::steady_clock::now();
  for (int step = 1; step < n; step *= 2) {
    for (int r = step; r < std::min(2 * step, n); r++) {
      BOX_CU(cudaSetDevice(devices[r]));
      for (int k = 0; k < 4; k++)
        BOX_CU(cudaMemcpyPeerAsync(rep[r][k], devices[r], rep[r - step][k], devices[r - step], bytes[k], st[r]));
    }
    for (int r = step; r < std::min(2 * step, n); r++) {
      BOX_CU(cudaSetDevice(devices[r]));
      BOX_CU(cudaStreamSynchronize(st[r]));
    }
  }
  b->replication_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  for (int r = 0; r < n; r++) {
    if (int rc = spf_b200_create_from_device(params, (const double*)rep[r][0], bsk_len, (const uint64_t*)rep[r][1], ksk_len,
                                             (const double*)rep[r][2], ssk_len, (const double*)rep[r][3], ak_len, devices[r],
                                             &b->ctx[r]))
      return fail_all(rc, "rank " + std::to_string(r) + ": " + g_create_err);
  }
#undef BOX_CU
  cleanup();
  b->jobs.resize(n);
  b->job_rc.assign(n, 0);
  for (int r = 0; r < n; r++) b->workers.emplace_back(box_worker, b.get(), r);
  *out = b.release();
  return 0;
}

// A host io buffer that a rank copies by DMA must lie inside ONE portable page-locked allocation or registration: a
// copy from memory that is pageable for the rank's device (a buffer whose first and last pages happen to be locked by
// its neighbours' registrations, a registration made for another device) synchronises the stream first -- and the
// stream may be held at a peer barrier until a rank that has not been enqueued yet arrives.  Every other io buffer is
// staged through the rank graph's own page-locked slab (io kind 1); registrations the rank graph made itself (for its
// device only) are dropped.
void settle_io(spf_b200_graph* g, size_t node) {
  const uint32_t op = g->nodes[node].op;
  if (op > SPF_OP_OUTPUT_GLEV1 || !g->nodes[node].io || g->io_kind[node] != 0) return;
  void* io = g->nodes[node].io;
  const size_t bytes = ct_host_bytes(&g->ctx->p, (CtType)(T_LWE0 + op % 5));
  unsigned int flags = 0;
  size_t size = 0;
  const unsigned long long base = alloc_base_of(io, &size);
  const bool dma = cudaHostGetFlags(&flags, io) == cudaSuccess && (flags & cudaHostAllocPortable) && base &&
                   (uintptr_t)io + bytes <= base + size;
  cudaGetLastError();
  if (!dma) g->io_kind[node] = 1;
}

void settle_all_io(spf_b200_graph* g) {
  for (void* q : g->pinned) cudaHostUnregister(q);
  g->pinned.clear();
  for (size_t v = 0; v < g->nodes.size(); v++) settle_io(g, v);
}

// A run of a box graph: member i runs shard i on box rank rank[i]; errors go to the box's slot, prefixed with that rank.
Run box_run(spf_b200_box_graph* bg) {
  return Run{bg->g, 0, nullptr, nullptr, bg, &bg->rank, bg->h_err, &bg->run, &bg->box->fc, &bg->box->err};
}

}  // namespace

extern "C" {

int spf_b200_box_create(const spf_params* params, const double* bsk_fft, size_t bsk_len, const uint64_t* ksk,
                        size_t ksk_len, const double* ssk_fft, size_t ssk_len, const double* ak_fft, size_t ak_len,
                        const int* devices, int n, spf_b200_box** out) {
  try {
    return box_create_impl(params, bsk_fft, bsk_len, ksk, ksk_len, ssk_fft, ssk_len, ak_fft, ak_len, devices, n, out);
  } catch (const std::exception& e) {
    return box_fail(nullptr, SPF_E_CUDA, std::string("box create: ") + e.what());
  }
}

int spf_b200_box_create_from_serialized(const spf_params* params, const uint8_t* buf, size_t len, const int* devices,
                                        int n, spf_b200_box** out) {
  if (!out) return box_fail(nullptr, SPF_E_INVALID, "out is NULL");
  *out = nullptr;
  if (n < 1 || n > kMaxPeers + 1) return box_fail(nullptr, SPF_E_INVALID, "box: n must be in 1..8 (a rank has at most 7 peers)");
  if (!devices) return box_fail(nullptr, SPF_E_INVALID, "box: devices is NULL");
  size_t off[4];
  if (int rc = spf_b200_parse_compute_key(params, buf, len, off)) return rc;
  return spf_b200_box_create(params, (const double*)(buf + off[0]), spf_b200_len_bsk(params), (const uint64_t*)(buf + off[1]),
                             spf_b200_len_ksk(params), (const double*)(buf + off[2]), spf_b200_len_ssk(params),
                             (const double*)(buf + off[3]), spf_b200_len_ak(params), devices, n, out);
}

void spf_b200_box_destroy(spf_b200_box* b) {
  if (!b) return;
  {
    std::lock_guard<std::mutex> lk(b->w_mu);
    b->stop = true;
  }
  b->w_job.notify_all();
  for (std::thread& t : b->workers) t.join();
  b->workers.clear();
  for (spf_b200_ctx* c : b->ctx) spf_b200_destroy(c);  // box graphs hold their own references
  box_release(b);
}

const char* spf_b200_box_last_error(const spf_b200_box* b) { return b ? b->err.c_str() : g_create_err.c_str(); }
int spf_b200_box_size(const spf_b200_box* b) { return b ? b->n : 0; }
int spf_b200_box_device(const spf_b200_box* b, int rank) { return b && rank >= 0 && rank < b->n ? b->device[rank] : -1; }
spf_b200_ctx* spf_b200_box_context(spf_b200_box* b, int rank) { return b && rank >= 0 && rank < b->n ? b->ctx[rank] : nullptr; }
double spf_b200_box_key_replication_ms(const spf_b200_box* b) { return b ? b->replication_ms : 0.0; }

void spf_b200_box_shard(size_t batch, int n, int rank, size_t* start, size_t* count) {
  if (!start || !count) return;
  *start = *count = 0;
  if (n < 1 || rank < 0 || rank >= n) return;
  box_shard(batch, n, rank, start, count);
}

int spf_b200_box_key_slice(spf_b200_box* b, int rank, int which, size_t offset, size_t count, void* out) {
  if (!b) return SPF_E_INVALID;
  if (rank < 0 || rank >= b->n || which < 0 || which > 3 || (!out && count))
    return box_fail(b, SPF_E_INVALID, "key_slice: bad rank, array or buffer");
  spf_b200_ctx* c = b->ctx[rank];
  const size_t len[4] = {spf_b200_len_bsk(&c->p), spf_b200_len_ksk(&c->p), spf_b200_len_ssk(&c->p), spf_b200_len_ak(&c->p)};
  if (offset > len[which] || count > len[which] - offset) return box_fail(b, SPF_E_INVALID, "key_slice: range outside the array");
  if (count == 0) return 0;
  BCU(b, cudaSetDevice(c->device));
  if (which == 1) {
    BCU(b, cudaMemcpy(out, c->ksk + offset, count * 8, cudaMemcpyDeviceToHost));
    return 0;
  }
  const C2* src = which == 0 ? c->bsk : which == 2 ? c->ssk : c->ak;
  BCU(b, cudaMemcpy(out, src + offset, count * 16, cudaMemcpyDeviceToHost));
  double* d = static_cast<double*>(out);
  for (size_t i = 0; i < 2 * count; i++) d[i] *= 1024.0;  // FFT keys are resident in the device scale (exact)
  return 0;
}

int spf_b200_box_circuit_bootstrap(spf_b200_box* b, double* ggsw_out, const uint64_t* lwe0_in, size_t batch) {
  if (!b) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!ggsw_out || !lwe0_in) return box_fail(b, SPF_E_INVALID, "NULL buffer");
  const spf_params* p = &b->ctx[0]->p;
  const size_t lwe = spf_b200_len_lwe_l0(p), ggsw = 2 * spf_b200_len_ggsw_l1(p);
  return box_each(b, batch, [&](spf_b200_ctx* c, size_t s, size_t k) {
    return spf_b200_circuit_bootstrap(c, ggsw_out + s * ggsw, lwe0_in + s * lwe, k);
  });
}

int spf_b200_box_programmable_bootstrap(spf_b200_box* b, uint64_t* glwe_out, const uint64_t* lwe0_in,
                                        const uint64_t* lut_glwe, uint32_t log_chi, uint32_t log_v, size_t batch) {
  if (!b) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!glwe_out || !lwe0_in || !lut_glwe) return box_fail(b, SPF_E_INVALID, "NULL buffer");
  const spf_params* p = &b->ctx[0]->p;
  const size_t lwe = spf_b200_len_lwe_l0(p), glwe = spf_b200_len_glwe_l1(p);
  return box_each(b, batch, [&](spf_b200_ctx* c, size_t s, size_t k) {
    return spf_b200_programmable_bootstrap(c, glwe_out + s * glwe, lwe0_in + s * lwe, lut_glwe, log_chi, log_v, k);
  });
}

int spf_b200_box_keyswitch_lwe_l1_lwe_l0(spf_b200_box* b, uint64_t* lwe0_out, const uint64_t* lwe1_in, size_t batch) {
  if (!b) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!lwe0_out || !lwe1_in) return box_fail(b, SPF_E_INVALID, "NULL buffer");
  const spf_params* p = &b->ctx[0]->p;
  const size_t l1 = spf_b200_len_lwe_l1(p), l0 = spf_b200_len_lwe_l0(p);
  return box_each(b, batch, [&](spf_b200_ctx* c, size_t s, size_t k) {
    return spf_b200_keyswitch_lwe_l1_lwe_l0(c, lwe0_out + s * l0, lwe1_in + s * l1, k);
  });
}

int spf_b200_box_cmux(spf_b200_box* b, uint64_t* glwe_out, const double* sel_ggsw, const uint64_t* a, const uint64_t* bb,
                      size_t batch) {
  if (!b) return SPF_E_INVALID;
  if (batch == 0) return 0;
  if (!glwe_out || !sel_ggsw || !a || !bb) return box_fail(b, SPF_E_INVALID, "NULL buffer");
  const spf_params* p = &b->ctx[0]->p;
  const size_t glwe = spf_b200_len_glwe_l1(p), ggsw = 2 * spf_b200_len_ggsw_l1(p);
  return box_each(b, batch, [&](spf_b200_ctx* c, size_t s, size_t k) {
    return spf_b200_cmux(c, glwe_out + s * glwe, sel_ggsw + s * ggsw, a + s * glwe, bb + s * glwe, k);
  });
}

int spf_b200_box_set_max_in_flight(spf_b200_box* b, int n) {
  if (!b) return SPF_E_INVALID;
  if (n < 1) return box_fail(b, SPF_E_INVALID, "max_in_flight must be at least 1");
  b->fc.set(n);
  return 0;
}

void spf_b200_box_graph_destroy(spf_b200_box_graph* bg) {
  if (!bg) return;
  // a spawned run may still be in flight: its completion uses bg until its last host function has returned
  for (spf_b200_graph* g : bg->g) {
    if (!g) continue;
    cudaSetDevice(g->ctx->device);
    cudaStreamSynchronize(g->stream);
  }
  for (spf_b200_graph* g : bg->g) spf_b200_graph_destroy(g);
  for (void* q : bg->pinned) cudaHostUnregister(q);
  if (bg->h_err) cudaFreeHost(bg->h_err);
  for (spf_b200_box_ciphertext* h : bg->bound) box_ciphertext_release(h);
  spf_b200_box* b = bg->box;
  delete bg;
  box_release(b);
}

int spf_b200_box_graph_build_on(spf_b200_box* b, const spf_node* nodes, size_t n_nodes, const int* ranks, int n_ranks,
                                spf_b200_box_graph** out) {
  if (!b) return SPF_E_INVALID;
  if (!out || (!nodes && n_nodes)) return box_fail(b, SPF_E_INVALID, "NULL argument");
  *out = nullptr;
  if (!ranks) return box_fail(b, SPF_E_INVALID, "box graph: ranks is NULL");
  if (n_ranks < 1 || n_ranks > b->n)
    return box_fail(b, SPF_E_INVALID, "box graph: n_ranks is " + std::to_string(n_ranks) + ", must be in 1.." + std::to_string(b->n) +
                                          " (the box size)");
  std::vector<char> seen(b->n, 0);
  for (int i = 0; i < n_ranks; i++) {
    if (ranks[i] < 0 || ranks[i] >= b->n)
      return box_fail(b, SPF_E_INVALID, "box graph: ranks[" + std::to_string(i) + "] = " + std::to_string(ranks[i]) +
                                            " is not a rank of the box (0.." + std::to_string(b->n - 1) + ")");
    if (seen[ranks[i]]++)
      return box_fail(b, SPF_E_INVALID, "box graph: rank " + std::to_string(ranks[i]) + " is named twice in ranks");
  }
  const spf_params* p = &b->ctx[0]->p;
  BCU(b, cudaSetDevice(b->device[0]));
  // io buffers: box ciphertext handles or host memory.  Unpinned host buffers are page-locked here as PORTABLE memory,
  // so that every rank's device copies them by DMA (a plain registration is page-locked for one device only).
  std::unique_ptr<spf_b200_box_graph, void (*)(spf_b200_box_graph*)> bg(new spf_b200_box_graph(), spf_b200_box_graph_destroy);
  bg->box = b;
  b->refs.fetch_add(1);
  bg->bound.assign(n_nodes, nullptr);
  for (size_t i = 0; i < n_nodes; i++) {
    if (!is_box_handle(nodes[i].io)) continue;
    spf_b200_box_ciphertext* h = static_cast<spf_b200_box_ciphertext*>(nodes[i].io);
    if (int rc = check_box_handle(b, h, i, nodes[i].op)) return rc;
    h->refs.fetch_add(1);
    bg->bound[i] = h;
  }
  for (size_t i = 0; i < n_nodes; i++) {
    const uint32_t op = nodes[i].op;
    if (op > SPF_OP_OUTPUT_GLEV1 || !nodes[i].io || bg->bound[i]) continue;
    const size_t bytes = ct_host_bytes(p, (CtType)(T_LWE0 + op % 5));
    cudaPointerAttributes a0, a1;
    if (cudaPointerGetAttributes(&a0, nodes[i].io) == cudaSuccess &&
        cudaPointerGetAttributes(&a1, static_cast<char*>(nodes[i].io) + bytes - 1) == cudaSuccess) {
      if (a0.type == cudaMemoryTypeDevice || a0.type == cudaMemoryTypeManaged)
        return box_fail(b, SPF_E_INVALID, "box graph: node " + std::to_string(i) +
                                              " has a device-memory io buffer; box graphs take host buffers or box "
                                              "ciphertext handles (spf_b200_box_ciphertext_alloc)");
      if (a0.type == cudaMemoryTypeHost && a1.type == cudaMemoryTypeHost) continue;
    }
    cudaGetLastError();
    if (cudaHostRegister(nodes[i].io, bytes, cudaHostRegisterPortable) == cudaSuccess) bg->pinned.push_back(nodes[i].io);
    else cudaGetLastError();  // left pageable: the rank graphs stage it through their page-locked slabs
  }
  // member i runs shard i of the graph sharded over the members; member 0 writes the outputs every member holds
  const int n = n_ranks;
  bg->rank.assign(ranks, ranks + n);
  bg->g.assign(n, nullptr);
  for (int i = 0; i < n; i++) {
    spf_b200_ctx* c = b->ctx[bg->rank[i]];
    if (int rc = graph_build_checked(c, nodes, n_nodes, n, &bg->g[i], true))
      return box_fail(b, rc, (bg->rank[i] ? "rank " + std::to_string(bg->rank[i]) + ": " : std::string()) + c->err);
    bg->g[i]->replicated_writer = 0;
    settle_all_io(bg->g[i]);
  }
  if (n > 1) {
    std::vector<void*> arenas(n);
    for (int i = 0; i < n; i++) arenas[i] = bg->g[i]->arena;
    for (int i = 0; i < n; i++)
      if (int rc = spf_b200_graph_set_peers(bg->g[i], i, n, arenas.data())) return box_fail(b, rc, bg->g[i]->ctx->err);
  }
  BCU(b, cudaHostAlloc(reinterpret_cast<void**>(&bg->h_err), sizeof(int) * n, cudaHostAllocPortable));
  memset(bg->h_err, 0, sizeof(int) * n);
  *out = bg.release();
  return 0;
}

int spf_b200_box_graph_build(spf_b200_box* b, const spf_node* nodes, size_t n_nodes, spf_b200_box_graph** out) {
  if (!b) return SPF_E_INVALID;
  std::vector<int> all(b->n);
  for (int r = 0; r < b->n; r++) all[r] = r;
  return spf_b200_box_graph_build_on(b, nodes, n_nodes, all.data(), b->n, out);
}

int spf_b200_box_graph_ranks(const spf_b200_box_graph* bg, int* ranks_out) {
  if (!bg) return SPF_E_INVALID;
  if (ranks_out) std::copy(bg->rank.begin(), bg->rank.end(), ranks_out);
  return (int)bg->rank.size();
}

int spf_b200_box_graph_run(spf_b200_box_graph* bg) { return bg ? run_blocking(box_run(bg)) : SPF_E_INVALID; }

int spf_b200_box_graph_spawn(spf_b200_box_graph* bg, spf_b200_box_graph* const* after, size_t n_after,
                             spf_completion_fn on_complete, void* user) {
  if (!bg) return SPF_E_INVALID;
  spf_b200_box* b = bg->box;
  if (n_after && !after) return box_fail(b, SPF_E_INVALID, "spawn: NULL dependency list");
  const Run run = box_run(bg);
  spawn_begin(run);
  int status = 0;
  std::string msg;
  if (poisoned(run)) {
    status = SPF_E_GRAPH;
    msg = kPoisoned;
  }
  std::vector<std::vector<spf_b200_graph*>> deps;
  for (size_t i = 0; i < n_after && status == 0; i++) {
    spf_b200_box_graph* d = after[i];
    if (!d || d == bg) continue;
    if (d->box != b) {
      status = SPF_E_INVALID;
      msg = "spawn: a dependency belongs to another box";
    } else if (const int ds = d->run.status.load()) {
      status = ds;
      msg = "a dependency of this graph failed: " + d->run.msg;
    } else {
      deps.push_back(d->g);
    }
  }
  return spawn(run, deps, status, msg, on_complete, user);
}

int spf_b200_box_graph_wait(spf_b200_box_graph* bg) { return bg ? wait_run(box_run(bg)) : SPF_E_INVALID; }

const char* spf_b200_box_graph_status_message(const spf_b200_box_graph* bg) { return bg ? bg->run.msg.c_str() : ""; }

int spf_b200_box_graph_set_io(spf_b200_box_graph* bg, size_t node, void* io) {
  if (!bg) return SPF_E_INVALID;
  spf_b200_box* b = bg->box;
  if (!io) return box_fail(b, SPF_E_INVALID, "set_io: io pointer is NULL");
  if (node >= bg->bound.size())
    return box_fail(b, SPF_E_INVALID, "set_io: node " + std::to_string(node) + " is not an Input*/Output* node");
  spf_b200_box_ciphertext* const old = bg->bound[node];
  if (is_box_handle(io)) {
    spf_b200_box_ciphertext* h = static_cast<spf_b200_box_ciphertext*>(io);
    if (int rc = check_box_handle(b, h, node, bg->g[0]->nodes[node].op)) return rc;
    h->refs.fetch_add(1);
    for (spf_b200_graph* g : bg->g) {
      g->nodes[node].io = h;
      g->io_kind[node] = 3;
      g->io_alloc[node] = 0;
    }
    bg->bound[node] = h;
    box_ciphertext_release(old);
    return 0;
  }
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, io) == cudaSuccess && (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged))
    return box_fail(b, SPF_E_INVALID, "box graph: device-memory io buffers are not supported; box graphs take host buffers "
                                      "or box ciphertext handles (spf_b200_box_ciphertext_alloc)");
  cudaGetLastError();
  for (size_t r = 0; r < bg->g.size(); r++) {
    if (int rc = spf_b200_graph_set_io(bg->g[r], node, io)) return box_fail(b, rc, bg->g[r]->ctx->err);
    settle_io(bg->g[r], node);
  }
  bg->bound[node] = nullptr;
  box_ciphertext_release(old);
  return 0;
}

int spf_b200_box_ciphertext_alloc(spf_b200_box* b, uint32_t kind, spf_b200_box_ciphertext** out) {
  if (out) *out = nullptr;
  if (kind > SPF_OP_INPUT_GLEV1)
    return box_fail(b, SPF_E_INVALID, "box ciphertext: unknown kind " + std::to_string(kind) +
                                          " (the Input* op code of the ciphertext type: SPF_OP_INPUT_LWE0 .. SPF_OP_INPUT_GLEV1)");
  if (!b) return box_fail(nullptr, SPF_E_INVALID, "box ciphertext: box is NULL");
  if (!out) return box_fail(b, SPF_E_INVALID, "box ciphertext: out is NULL");
  spf_b200_box_ciphertext* h = new spf_b200_box_ciphertext();
  h->box = b;
  b->refs.fetch_add(1);
  h->kind = kind;
  h->bytes = ct_bytes(&b->ctx[0]->p, (CtType)(T_LWE0 + kind));
  h->rep.assign(b->n, nullptr);
  // zero-filled, as the reference's enc.allocate_* (the legacy stream orders the fill before any later copy)
  for (int r = 0; r < b->n; r++) {
    cudaError_t e = cudaSetDevice(b->device[r]);
    if (e == cudaSuccess) e = cudaMalloc(&h->rep[r], h->bytes);
    if (e == cudaSuccess) e = cudaMemsetAsync(h->rep[r], 0, h->bytes, 0);
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);
    if (e != cudaSuccess) {
      box_ciphertext_delete(h);
      return box_fail(b, SPF_E_CUDA, std::string("box ciphertext alloc: ") + cudaGetErrorString(e));
    }
  }
  {
    std::lock_guard<std::mutex> lk(g_box_handles_mu);
    g_box_handles.insert(h);
  }
  *out = h;
  return 0;
}

void spf_b200_box_ciphertext_free(spf_b200_box_ciphertext* h) {
  if (is_box_handle(h)) box_ciphertext_release(h);
}

int spf_b200_box_ciphertext_write(spf_b200_box_ciphertext* h, const void* host_src) {
  if (!is_box_handle(h)) return box_fail(nullptr, SPF_E_INVALID, "box ciphertext: not a live handle");
  spf_b200_box* b = h->box;
  if (!host_src) return box_fail(b, SPF_E_INVALID, "box ciphertext write: NULL buffer");
  const void* src = host_src;
  std::vector<double> scaled;
  if (h->kind == SPF_OP_INPUT_GGSW1) {  // reference scale -> device scale (exact: a power of two)
    const double* d = static_cast<const double*>(host_src);
    scaled.assign(d, d + h->bytes / 8);
    for (double& x : scaled) x *= 1.0 / 1024.0;
    src = scaled.data();
  }
  for (size_t r = 0; r < h->rep.size(); r++) {
    BCU(b, cudaSetDevice(b->device[r]));
    BCU(b, cudaMemcpyAsync(h->rep[r], src, h->bytes, cudaMemcpyHostToDevice, 0));
    BCU(b, cudaStreamSynchronize(0));
  }
  return 0;
}

int spf_b200_box_ciphertext_read(spf_b200_box_ciphertext* h, int rank, void* host_dst) {
  if (!is_box_handle(h)) return box_fail(nullptr, SPF_E_INVALID, "box ciphertext: not a live handle");
  spf_b200_box* b = h->box;
  if (rank < 0 || rank >= (int)h->rep.size()) return box_fail(b, SPF_E_INVALID, "box ciphertext read: rank out of range");
  if (!host_dst) return box_fail(b, SPF_E_INVALID, "box ciphertext read: NULL buffer");
  BCU(b, cudaSetDevice(b->device[rank]));
  BCU(b, cudaMemcpyAsync(host_dst, h->rep[rank], h->bytes, cudaMemcpyDeviceToHost, 0));
  BCU(b, cudaStreamSynchronize(0));
  if (h->kind == SPF_OP_INPUT_GGSW1) {  // device scale -> reference scale
    double* d = static_cast<double*>(host_dst);
    for (size_t i = 0; i < h->bytes / 8; i++) d[i] *= 1024.0;
  }
  return 0;
}

int spf_b200_box_graph_levels(const spf_b200_box_graph* bg) { return bg && !bg->g.empty() ? bg->g[0]->n_levels : -1; }
uint64_t spf_b200_box_graph_launches(const spf_b200_box_graph* bg) { return bg ? bg->run.launches : 0; }

}  // extern "C"
