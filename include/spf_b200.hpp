// spf_b200.hpp -- C++17 host side above the C ABI (include/spf_b200.h), header-only.
//
// The reference's host language is Rust; its toolchain is absent from this image, so next to the Rust
// `extern "C"` shim shown in INTEGRATION.md this header mirrors the reference's interface for the hot path in
// C++, with the reference's names, argument meaning and error behaviour:
//   spf::Evaluation        parasol_runtime/src/crypto/evaluation.rs:125-255 (Evaluation / KeylessEvaluation)
//   spf::FheCircuit        parasol_runtime/src/fhe_circuit.rs:205-398 (add_node / add_edge collapsed into add())
//   spf::CircuitProcessor  parasol_runtime/src/circuit_processor/mod.rs:62-655 (run_graph_blocking, compiled graphs)
//   spf::MuxCircuit        mux_circuits/src/lib.rs:153-341 and the generators of mux_circuits/src/*.rs
// Errors: the tfhe layer of the reference panics on wrong sizes and the runtime returns RuntimeError(String); here
// every failing call throws spf::Error carrying the C ABI's status code and message.  Outputs are caller-allocated
// (std::vector sized with the len_* helpers), inputs are const, batched calls take a leading batch dimension.
#pragma once

#include <cstdint>
#include <initializer_list>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "spf_b200.h"

namespace spf {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& what) : std::runtime_error(what), code(c) {}
};

inline void check(int rc, const spf_b200_ctx* ctx = nullptr) {
  if (rc == SPF_OK) return;
  const char* msg = spf_b200_last_error(ctx);
  throw Error(rc, msg && *msg ? msg : "spf_b200 error " + std::to_string(rc));
}

// DEFAULT_128 (parasol_runtime/src/params.rs:107-134)
inline spf_params default_128() {
  spf_params p;
  spf_b200_default_128(&p);
  return p;
}

using Torus = std::uint64_t;
using Complex = double;  // FFT-domain entities are (re, im) pairs: 2 doubles per element

class Evaluation {
 public:
  // Evaluation::new (evaluation.rs:161-197): the four arrays of ComputeKey, element counts must equal len_*.
  Evaluation(const spf_params& params, const std::vector<Complex>& bsk_fft, const std::vector<Torus>& ksk,
             const std::vector<Complex>& ssk_fft, const std::vector<Complex>& ak_fft, int device = 0)
      : p_(params) {
    check(spf_b200_create(&p_, bsk_fft.data(), bsk_fft.size() / 2, ksk.data(), ksk.size(), ssk_fft.data(), ssk_fft.size() / 2,
                          ak_fft.data(), ak_fft.size() / 2, device, &ctx_));
  }
  // safe_bincode::deserialize::<ComputeKey> + Evaluation::new (safe_bincode.rs:16-27)
  static Evaluation from_serialized(const spf_params& params, const std::uint8_t* buf, std::size_t len, int device = 0) {
    Evaluation e(params);
    check(spf_b200_create_from_serialized(&e.p_, buf, len, device, &e.ctx_));
    return e;
  }
  Evaluation(Evaluation&& o) noexcept : p_(o.p_), ctx_(std::exchange(o.ctx_, nullptr)) {}
  Evaluation& operator=(Evaluation&& o) noexcept {
    if (this != &o) { reset(); p_ = o.p_; ctx_ = std::exchange(o.ctx_, nullptr); }
    return *this;
  }
  Evaluation(const Evaluation&) = delete;
  Evaluation& operator=(const Evaluation&) = delete;
  ~Evaluation() { reset(); }

  const spf_params& params() const { return p_; }
  spf_b200_ctx* handle() const { return ctx_; }
  std::size_t len_lwe_l0() const { return spf_b200_len_lwe_l0(&p_); }
  std::size_t len_lwe_l1() const { return spf_b200_len_lwe_l1(&p_); }
  std::size_t len_glwe_l1() const { return spf_b200_len_glwe_l1(&p_); }
  std::size_t len_glev_l1() const { return spf_b200_len_glev_l1(&p_); }
  std::size_t len_ggsw_l1() const { return spf_b200_len_ggsw_l1(&p_); }  // complex elements
  std::uint64_t kernel_launches() const { return spf_b200_kernel_launches(ctx_); }

  // Evaluation::circuit_bootstrap (evaluation.rs:211-225), `batch` independent L0 LWE inputs
  void circuit_bootstrap(std::vector<Complex>& ggsw_out, const std::vector<Torus>& lwe0_in) const {
    const std::size_t batch = batch_of(lwe0_in.size(), len_lwe_l0(), "circuit_bootstrap");
    ggsw_out.resize(batch * len_ggsw_l1() * 2);
    check(spf_b200_circuit_bootstrap(ctx_, ggsw_out.data(), lwe0_in.data(), batch), ctx_);
  }
  // generalized_programmable_bootstrap (programmable_bootstrapping.rs:342-410); one LUT for the batch
  void programmable_bootstrap(std::vector<Torus>& glwe_out, const std::vector<Torus>& lwe0_in, const std::vector<Torus>& lut_glwe,
                              std::uint32_t log_chi, std::uint32_t log_v) const {
    const std::size_t batch = batch_of(lwe0_in.size(), len_lwe_l0(), "programmable_bootstrap");
    if (lut_glwe.size() != len_glwe_l1()) throw Error(SPF_E_INVALID, "programmable_bootstrap: LUT has the wrong length");
    glwe_out.resize(batch * len_glwe_l1());
    check(spf_b200_programmable_bootstrap(ctx_, glwe_out.data(), lwe0_in.data(), lut_glwe.data(), log_chi, log_v, batch), ctx_);
  }
  // KeylessEvaluation::cmux (evaluation.rs:68-83): out = sel ? b : a
  void cmux(std::vector<Torus>& out, const std::vector<Complex>& sel, const std::vector<Torus>& a, const std::vector<Torus>& b) const {
    const std::size_t batch = batch_of(a.size(), len_glwe_l1(), "cmux");
    if (b.size() != a.size() || sel.size() != batch * len_ggsw_l1() * 2) throw Error(SPF_E_INVALID, "cmux: operand sizes differ");
    out.resize(a.size());
    check(spf_b200_cmux(ctx_, out.data(), sel.data(), a.data(), b.data(), batch), ctx_);
  }
  // KeylessEvaluation::glev_cmux (evaluation.rs:86-101)
  void glev_cmux(std::vector<Torus>& out, const std::vector<Complex>& sel, const std::vector<Torus>& a, const std::vector<Torus>& b) const {
    const std::size_t batch = batch_of(a.size(), len_glev_l1(), "glev_cmux");
    if (b.size() != a.size() || sel.size() != batch * len_ggsw_l1() * 2) throw Error(SPF_E_INVALID, "glev_cmux: operand sizes differ");
    out.resize(a.size());
    check(spf_b200_glev_cmux(ctx_, out.data(), sel.data(), a.data(), b.data(), batch), ctx_);
  }
  // KeylessEvaluation::multiply_glwe_ggsw (evaluation.rs:104-123)
  void multiply_glwe_ggsw(std::vector<Torus>& out, const std::vector<Torus>& glwe, const std::vector<Complex>& ggsw) const {
    const std::size_t batch = batch_of(glwe.size(), len_glwe_l1(), "multiply_glwe_ggsw");
    if (ggsw.size() != batch * len_ggsw_l1() * 2) throw Error(SPF_E_INVALID, "multiply_glwe_ggsw: operand sizes differ");
    out.resize(glwe.size());
    check(spf_b200_multiply_glwe_ggsw(ctx_, out.data(), glwe.data(), ggsw.data(), batch), ctx_);
  }
  // Evaluation::keyswitch_lwe_l1_lwe_l0 (evaluation.rs:243-252)
  void keyswitch_lwe_l1_lwe_l0(std::vector<Torus>& lwe0_out, const std::vector<Torus>& lwe1_in) const {
    const std::size_t batch = batch_of(lwe1_in.size(), len_lwe_l1(), "keyswitch_lwe_l1_lwe_l0");
    lwe0_out.resize(batch * len_lwe_l0());
    check(spf_b200_keyswitch_lwe_l1_lwe_l0(ctx_, lwe0_out.data(), lwe1_in.data(), batch), ctx_);
  }
  // Evaluation::scheme_switch (evaluation.rs:231-240)
  void scheme_switch(std::vector<Complex>& ggsw_out, const std::vector<Torus>& glev_in) const {
    const std::size_t batch = batch_of(glev_in.size(), len_glev_l1(), "scheme_switch");
    ggsw_out.resize(batch * len_ggsw_l1() * 2);
    check(spf_b200_scheme_switch(ctx_, ggsw_out.data(), glev_in.data(), batch), ctx_);
  }
  // KeylessEvaluation::sample_extract_l1 (evaluation.rs:126-133), the same index for the whole batch
  void sample_extract_l1(std::vector<Torus>& lwe1_out, const std::vector<Torus>& glwe_in, std::uint32_t idx) const {
    const std::size_t batch = batch_of(glwe_in.size(), len_glwe_l1(), "sample_extract_l1");
    lwe1_out.resize(batch * len_lwe_l1());
    check(spf_b200_sample_extract_l1(ctx_, lwe1_out.data(), glwe_in.data(), nullptr, idx, batch), ctx_);
  }
  // KeylessEvaluation::{not, xor, mul_xn} (evaluation.rs:48-65)
  void not_(std::vector<Torus>& out, const std::vector<Torus>& in) const {
    out.resize(in.size());
    check(spf_b200_not(ctx_, out.data(), in.data(), batch_of(in.size(), len_glwe_l1(), "not")), ctx_);
  }
  void xor_(std::vector<Torus>& out, const std::vector<Torus>& a, const std::vector<Torus>& b) const {
    if (a.size() != b.size()) throw Error(SPF_E_INVALID, "xor: operand sizes differ");
    out.resize(a.size());
    check(spf_b200_xor(ctx_, out.data(), a.data(), b.data(), batch_of(a.size(), len_glwe_l1(), "xor")), ctx_);
  }
  void mul_xn(std::vector<Torus>& out, const std::vector<Torus>& in, std::uint32_t n) const {
    out.resize(in.size());
    check(spf_b200_mul_xn(ctx_, out.data(), in.data(), n, batch_of(in.size(), len_glwe_l1(), "mul_xn")), ctx_);
  }

  // Encryption::encrypt_rlwe_l1 / rlwe_encrypt_public (encryption.rs:205-215, rlwe_encryption.rs:108-160), randomness given
  void rlwe_encrypt_public(std::vector<Torus>& out, const std::vector<Torus>& public_key, const std::vector<Torus>& encoded_msg,
                           const std::vector<Torus>& u, const std::vector<Torus>& e0, const std::vector<Torus>& e1) const {
    const std::size_t n = len_glwe_l1() / 2, batch = batch_of(encoded_msg.size(), n, "rlwe_encrypt_public");
    if (public_key.size() != 2 * n || u.size() != batch * n || e0.size() != batch * n || e1.size() != batch * n)
      throw Error(SPF_E_INVALID, "rlwe_encrypt_public: operand sizes differ");
    out.resize(batch * 2 * n);
    check(spf_b200_rlwe_encrypt_public(ctx_, out.data(), public_key.data(), encoded_msg.data(), u.data(), e0.data(), e1.data(), batch), ctx_);
  }

 private:
  explicit Evaluation(const spf_params& params) : p_(params) {}
  void reset() {
    if (ctx_) spf_b200_destroy(ctx_);
    ctx_ = nullptr;
  }
  static std::size_t batch_of(std::size_t len, std::size_t item, const char* what) {
    if (item == 0 || len % item) throw Error(SPF_E_INVALID, std::string(what) + ": length is not a whole number of ciphertexts");
    return len / item;
  }
  spf_params p_;
  spf_b200_ctx* ctx_ = nullptr;
};

// FheCircuit (fhe_circuit.rs:205-208): a DAG of FheOp nodes; edges are given when the consumer is added, in the
// order of the reference's FheEdge names (Unary | Left, Right | Sel, Low, High | Glwe, Ggsw).
class FheCircuit {
 public:
  int add(spf_op op, int in0 = -1, int in1 = -1, int in2 = -1, std::uint32_t arg = 0, void* io = nullptr) {
    spf_node n{};
    n.op = static_cast<std::uint32_t>(op);
    n.arg = arg;
    n.in[0] = in0; n.in[1] = in1; n.in[2] = in2;
    n.io = io;
    nodes_.push_back(n);
    return static_cast<int>(nodes_.size()) - 1;
  }
  int input(spf_op op, void* io) { return add(op, -1, -1, -1, 0, io); }
  int output(spf_op op, int src, void* io) { return add(op, src, -1, -1, 0, io); }
  const std::vector<spf_node>& nodes() const { return nodes_; }
  std::size_t size() const { return nodes_.size(); }

  // Host-only schedule (spf_b200_graph_plan): dependency level and owning rank of every node; throws Error(SPF_E_GRAPH)
  // for malformed graphs as run_graph_blocking returns Err(RuntimeError).
  std::pair<std::vector<std::int32_t>, std::vector<std::int32_t>> plan(const spf_params& p, int world = 1) const {
    std::vector<std::int32_t> level(nodes_.size()), owner(nodes_.size());
    check(spf_b200_graph_plan(&p, nodes_.data(), nodes_.size(), world, level.data(), owner.data()));
    return {std::move(level), std::move(owner)};
  }

 private:
  std::vector<spf_node> nodes_;
};

// A levelised graph resident on one GPU; reusable across invocations (set_io re-binds host buffers).
class CompiledGraph {
 public:
  CompiledGraph(const Evaluation& ev, const FheCircuit& c, int world = 1) : ctx_(ev.handle()) {
    check(spf_b200_graph_build_sharded(ctx_, c.nodes().data(), c.size(), world, &g_), ctx_);
  }
  CompiledGraph(CompiledGraph&& o) noexcept : ctx_(o.ctx_), g_(std::exchange(o.g_, nullptr)) {}
  CompiledGraph(const CompiledGraph&) = delete;
  CompiledGraph& operator=(const CompiledGraph&) = delete;
  ~CompiledGraph() { if (g_) spf_b200_graph_destroy(g_); }
  void run() { check(spf_b200_graph_run(g_), ctx_); }
  void run_sharded(int rank, int world, spf_exchange_fn exchange = nullptr, void* user = nullptr) {
    check(spf_b200_graph_run_sharded(g_, rank, world, exchange, user), ctx_);
  }
  void set_io(std::size_t node, void* io) { check(spf_b200_graph_set_io(g_, node, io), ctx_); }
  int output_rank(std::size_t node) const { return spf_b200_graph_output_rank(g_, node); }
  int levels() const { return spf_b200_graph_levels(g_); }
  std::uint64_t launches() const { return spf_b200_graph_launches(g_); }
  spf_b200_graph* handle() const { return g_; }

 private:
  spf_b200_ctx* ctx_;
  spf_b200_graph* g_ = nullptr;
};

// CircuitProcessor (circuit_processor/mod.rs:62-655) for one GPU.
class CircuitProcessor {
 public:
  explicit CircuitProcessor(const Evaluation& ev) : ev_(ev) {}
  CompiledGraph compile(const FheCircuit& c, int world = 1) const { return CompiledGraph(ev_, c, world); }
  // run_graph_blocking (mod.rs:641-655)
  void run_graph_blocking(const FheCircuit& c) const { check(spf_b200_run_graph(ev_.handle(), c.nodes().data(), c.size()), ev_.handle()); }

 private:
  const Evaluation& ev_;
};

inline void check_box(int rc, const spf_b200_box* box) {
  if (rc == SPF_OK) return;
  const char* msg = spf_b200_box_last_error(box);
  throw Error(rc, msg && *msg ? msg : "spf_b200 error " + std::to_string(rc));
}

// Evaluation over several GPUs of one box, from one thread (spf_b200_box_*): rank r is a context on devices[r]; the
// compute key crosses PCIe once and is replicated device to device.  Batched ops split the batch over the ranks.
class BoxEvaluation {
 public:
  BoxEvaluation(const spf_params& params, const std::vector<Complex>& bsk_fft, const std::vector<Torus>& ksk,
                const std::vector<Complex>& ssk_fft, const std::vector<Complex>& ak_fft, const std::vector<int>& devices)
      : p_(params) {
    check_box(spf_b200_box_create(&p_, bsk_fft.data(), bsk_fft.size() / 2, ksk.data(), ksk.size(), ssk_fft.data(), ssk_fft.size() / 2,
                                  ak_fft.data(), ak_fft.size() / 2, devices.data(), static_cast<int>(devices.size()), &box_),
              nullptr);
  }
  static BoxEvaluation from_serialized(const spf_params& params, const std::uint8_t* buf, std::size_t len, const std::vector<int>& devices) {
    BoxEvaluation e(params);
    check_box(spf_b200_box_create_from_serialized(&e.p_, buf, len, devices.data(), static_cast<int>(devices.size()), &e.box_), nullptr);
    return e;
  }
  BoxEvaluation(BoxEvaluation&& o) noexcept : p_(o.p_), box_(std::exchange(o.box_, nullptr)) {}
  BoxEvaluation(const BoxEvaluation&) = delete;
  BoxEvaluation& operator=(const BoxEvaluation&) = delete;
  ~BoxEvaluation() { if (box_) spf_b200_box_destroy(box_); }

  const spf_params& params() const { return p_; }
  spf_b200_box* handle() const { return box_; }
  int size() const { return spf_b200_box_size(box_); }
  spf_b200_ctx* context(int rank) const { return spf_b200_box_context(box_, rank); }
  double key_replication_ms() const { return spf_b200_box_key_replication_ms(box_); }

  void circuit_bootstrap(std::vector<Complex>& ggsw_out, const std::vector<Torus>& lwe0_in) const {
    const std::size_t batch = batch_of(lwe0_in.size(), spf_b200_len_lwe_l0(&p_), "circuit_bootstrap");
    ggsw_out.resize(batch * spf_b200_len_ggsw_l1(&p_) * 2);
    check_box(spf_b200_box_circuit_bootstrap(box_, ggsw_out.data(), lwe0_in.data(), batch), box_);
  }
  void programmable_bootstrap(std::vector<Torus>& glwe_out, const std::vector<Torus>& lwe0_in, const std::vector<Torus>& lut_glwe,
                              std::uint32_t log_chi, std::uint32_t log_v) const {
    const std::size_t batch = batch_of(lwe0_in.size(), spf_b200_len_lwe_l0(&p_), "programmable_bootstrap");
    if (lut_glwe.size() != spf_b200_len_glwe_l1(&p_)) throw Error(SPF_E_INVALID, "programmable_bootstrap: LUT has the wrong length");
    glwe_out.resize(batch * spf_b200_len_glwe_l1(&p_));
    check_box(spf_b200_box_programmable_bootstrap(box_, glwe_out.data(), lwe0_in.data(), lut_glwe.data(), log_chi, log_v, batch), box_);
  }
  void keyswitch_lwe_l1_lwe_l0(std::vector<Torus>& lwe0_out, const std::vector<Torus>& lwe1_in) const {
    const std::size_t batch = batch_of(lwe1_in.size(), spf_b200_len_lwe_l1(&p_), "keyswitch_lwe_l1_lwe_l0");
    lwe0_out.resize(batch * spf_b200_len_lwe_l0(&p_));
    check_box(spf_b200_box_keyswitch_lwe_l1_lwe_l0(box_, lwe0_out.data(), lwe1_in.data(), batch), box_);
  }
  void cmux(std::vector<Torus>& out, const std::vector<Complex>& sel, const std::vector<Torus>& a, const std::vector<Torus>& b) const {
    const std::size_t batch = batch_of(a.size(), spf_b200_len_glwe_l1(&p_), "cmux");
    if (b.size() != a.size() || sel.size() != batch * spf_b200_len_ggsw_l1(&p_) * 2) throw Error(SPF_E_INVALID, "cmux: operand sizes differ");
    out.resize(a.size());
    check_box(spf_b200_box_cmux(box_, out.data(), sel.data(), a.data(), b.data(), batch), box_);
  }
  void set_max_in_flight(int n) const { check_box(spf_b200_box_set_max_in_flight(box_, n), box_); }

 private:
  explicit BoxEvaluation(const spf_params& params) : p_(params) {}
  static std::size_t batch_of(std::size_t len, std::size_t item, const char* what) {
    if (item == 0 || len % item) throw Error(SPF_E_INVALID, std::string(what) + ": length is not a whole number of ciphertexts");
    return len / item;
  }
  spf_params p_;
  spf_b200_box* box_ = nullptr;
};

// A box ciphertext handle (spf_b200_box_ciphertext_*): one ciphertext in HBM, one replica per rank.  Bind handle()
// as the io of box graph Input* / Output* nodes; box graphs hold their own references, so the handle may go out of
// scope while a graph still binds it.  kind: SPF_OP_INPUT_LWE0 .. SPF_OP_INPUT_GLEV1.
class BoxCiphertext {
 public:
  BoxCiphertext(const BoxEvaluation& ev, spf_op kind) : box_(ev.handle()) {
    check_box(spf_b200_box_ciphertext_alloc(box_, static_cast<std::uint32_t>(kind), &h_), box_);
  }
  BoxCiphertext(BoxCiphertext&& o) noexcept : box_(o.box_), h_(std::exchange(o.h_, nullptr)) {}
  BoxCiphertext(const BoxCiphertext&) = delete;
  BoxCiphertext& operator=(const BoxCiphertext&) = delete;
  ~BoxCiphertext() { spf_b200_box_ciphertext_free(h_); }
  // host -> every replica (reference layout and scale); host_src holds one whole ciphertext
  void write(const void* host_src) { check_box(spf_b200_box_ciphertext_write(h_, host_src), box_); }
  // rank's replica -> host (reference layout and scale)
  void read(void* host_dst, int rank = 0) const { check_box(spf_b200_box_ciphertext_read(h_, rank, host_dst), box_); }
  spf_b200_box_ciphertext* handle() const { return h_; }

 private:
  spf_b200_box* box_;
  spf_b200_box_ciphertext* h_ = nullptr;
};

// A levelised graph over every rank of a box, or over the ranks named in `ranks` (member i runs on box rank ranks[i]);
// io buffers are host memory or BoxCiphertext handles.
class BoxGraph {
 public:
  BoxGraph(const BoxEvaluation& ev, const FheCircuit& c) : box_(ev.handle()) {
    check_box(spf_b200_box_graph_build(box_, c.nodes().data(), c.size(), &g_), box_);
  }
  BoxGraph(const BoxEvaluation& ev, const FheCircuit& c, const std::vector<int>& ranks) : box_(ev.handle()) {
    check_box(spf_b200_box_graph_build_on(box_, c.nodes().data(), c.size(), ranks.data(), static_cast<int>(ranks.size()), &g_),
              box_);
  }
  // the box ranks the graph runs on, in member order
  std::vector<int> ranks() const {
    const int n = spf_b200_box_graph_ranks(g_, nullptr);
    std::vector<int> r(static_cast<std::size_t>(n > 0 ? n : 0));
    if (n > 0) spf_b200_box_graph_ranks(g_, r.data());
    return r;
  }
  BoxGraph(BoxGraph&& o) noexcept : box_(o.box_), g_(std::exchange(o.g_, nullptr)) {}
  BoxGraph(const BoxGraph&) = delete;
  BoxGraph& operator=(const BoxGraph&) = delete;
  ~BoxGraph() { if (g_) spf_b200_box_graph_destroy(g_); }
  void run() { check_box(spf_b200_box_graph_run(g_), box_); }
  // spawn_graph: on_complete(user, status, message) fires once, after every rank has retired, on a CUDA thread
  void spawn(const std::vector<const BoxGraph*>& after, spf_completion_fn on_complete, void* user) {
    std::vector<spf_b200_box_graph*> deps;
    for (const BoxGraph* d : after) deps.push_back(d->g_);
    check_box(spf_b200_box_graph_spawn(g_, deps.data(), deps.size(), on_complete, user), box_);
  }
  void wait() {
    const int rc = spf_b200_box_graph_wait(g_);
    if (rc != SPF_OK) throw Error(rc, spf_b200_box_graph_status_message(g_));
  }
  void set_io(std::size_t node, void* io) { check_box(spf_b200_box_graph_set_io(g_, node, io), box_); }
  int levels() const { return spf_b200_box_graph_levels(g_); }
  std::uint64_t launches() const { return spf_b200_box_graph_launches(g_); }
  spf_b200_box_graph* handle() const { return g_; }

 private:
  spf_b200_box* box_;
  spf_b200_box_graph* g_ = nullptr;
};

// CircuitProcessor (circuit_processor/mod.rs:62-655) over every GPU of a box.
class BoxCircuitProcessor {
 public:
  explicit BoxCircuitProcessor(const BoxEvaluation& ev) : ev_(ev) {}
  BoxGraph compile(const FheCircuit& c) const { return BoxGraph(ev_, c); }
  BoxGraph compile(const FheCircuit& c, const std::vector<int>& ranks) const { return BoxGraph(ev_, c, ranks); }
  void run_graph_blocking(const FheCircuit& c) const { compile(c).run(); }

 private:
  const BoxEvaluation& ev_;
};

// MuxCircuit (mux_circuits/src/lib.rs:153-163) as the C ABI's flat, topologically ordered node list.
class MuxCircuit {
 public:
  static MuxCircuit generate(spf_mux_kind kind, std::uint32_t n, std::uint32_t m = 0, std::uint32_t flags = 0) {
    spf_mux_node* p = nullptr;
    std::size_t count = 0;
    check(spf_b200_mux_circuit(kind, n, m, flags, &p, &count));
    MuxCircuit c;
    c.nodes_.assign(p, p + count);
    spf_b200_mux_free(p);
    for (std::size_t i = 0; i < count; i++) {
      if (c.nodes_[i].op == SPF_MUX_VARIABLE) c.inputs_.push_back(static_cast<int>(i));   // emitted in index order
      if (c.nodes_[i].op == SPF_MUX_OUTPUT) c.outputs_.push_back(static_cast<int>(i));
    }
    return c;
  }
  // mux_circuits::{add::ripple_carry_adder, mul::unsigned_multiplier, comparisons::compare_or_maybe_equal, ...}
  static MuxCircuit ripple_carry_adder(std::uint32_t n, std::uint32_t m, bool cin = false) { return generate(SPF_MUX_RIPPLE_CARRY_ADDER, n, m, cin); }
  static MuxCircuit unsigned_multiplier(std::uint32_t n, std::uint32_t m) { return generate(SPF_MUX_UNSIGNED_MULTIPLIER, n, m); }
  static MuxCircuit gradeschool_reduce(std::uint32_t n, std::uint32_t m) { return generate(SPF_MUX_GRADESCHOOL_REDUCE, n, m); }
  static MuxCircuit compare_or_maybe_equal(std::uint32_t n, bool greater, bool or_equal) {
    return generate(SPF_MUX_COMPARE, n, 0, (greater ? 1u : 0u) | (or_equal ? 2u : 0u));
  }
  const std::vector<spf_mux_node>& nodes() const { return nodes_; }
  const std::vector<int>& inputs() const { return inputs_; }
  const std::vector<int>& outputs() const { return outputs_; }
  std::size_t mux_gates() const {
    std::size_t g = 0;
    for (const auto& n : nodes_) g += n.op == SPF_MUX_MUX;
    return g;
  }
  // plaintext evaluation (the reference's test_mux_circuit, lib.rs:470-540)
  std::vector<int> evaluate(const std::vector<int>& bits) const {
    if (bits.size() != inputs_.size()) throw Error(SPF_E_INVALID, "MuxCircuit::evaluate: wrong number of input bits");
    std::vector<int> v(nodes_.size(), 0), out;
    for (std::size_t i = 0; i < nodes_.size(); i++) {
      const spf_mux_node& n = nodes_[i];
      switch (n.op) {
        case SPF_MUX_ONE: v[i] = 1; break;
        case SPF_MUX_VARIABLE: v[i] = bits[n.arg]; break;
        case SPF_MUX_MUX: v[i] = v[n.sel] ? v[n.high] : v[n.low]; break;
        case SPF_MUX_OUTPUT: v[i] = v[n.low]; break;
        default: break;
      }
    }
    for (int o : outputs_) out.push_back(v[o]);
    return out;
  }

 private:
  std::vector<spf_mux_node> nodes_;
  std::vector<int> inputs_, outputs_;
};

// FheCircuit::insert_mux_circuit (fhe_circuit.rs:274-398), MuxMode::Glwe: Mux -> CMux, One/Zero -> OneGlwe1/ZeroGlwe1,
// Variable(i) -> nodes_to_inputs[i] (GGSW producers); returns the node behind every Output(i).
inline std::vector<int> insert_mux_circuit(FheCircuit& c, const MuxCircuit& mux, const std::vector<int>& nodes_to_inputs) {
  if (nodes_to_inputs.size() != mux.inputs().size()) throw Error(SPF_E_INVALID, "insert_mux_circuit: wrong number of inputs");
  std::vector<int> ren(mux.nodes().size(), -1), outs;
  for (std::size_t i = 0; i < mux.nodes().size(); i++) {
    const spf_mux_node& n = mux.nodes()[i];
    switch (n.op) {
      case SPF_MUX_ZERO: ren[i] = c.add(SPF_OP_ZERO_GLWE1); break;
      case SPF_MUX_ONE: ren[i] = c.add(SPF_OP_ONE_GLWE1); break;
      case SPF_MUX_VARIABLE: ren[i] = nodes_to_inputs[n.arg]; break;
      case SPF_MUX_MUX: ren[i] = c.add(SPF_OP_CMUX, ren[n.sel], ren[n.low], ren[n.high]); break;
      case SPF_MUX_OUTPUT: outs.push_back(ren[n.low]); break;
      default: break;
    }
  }
  return outs;
}

// insert_ciphertext_conversion(L1Glwe -> L1Ggsw) (fhe_circuit.rs:562-619): SampleExtract(0) -> KeyswitchL1toL0 -> CircuitBootstrap
inline int glwe_to_ggsw(FheCircuit& c, int node) {
  return c.add(SPF_OP_CIRCUIT_BOOTSTRAP, c.add(SPF_OP_KEYSWITCH_L1_TO_L0, c.add(SPF_OP_SAMPLE_EXTRACT, node)));
}

// mux_circuits::mul::partition_integer (mul.rs:263-273), CIRCUIT_CUTOFF = 16: (low, high) word widths
inline std::pair<std::size_t, std::size_t> partition_integer(std::size_t n) {
  return n <= 16 ? std::make_pair(n, std::size_t{0}) : std::make_pair(n - n / 2, n / 2);
}

// circuits/mul.rs:91-199 (mul_impl): recursive grade-school multiplication of GGSW-encrypted operands (LSB first):
// blocks of at most 16 x 16 bits from the multiplier MUX circuit, then -- behind one bootstrap level -- the 4-way
// reduction circuit fed in the order of encode_gradeschool_reduction (mul.rs:289-387).  Returns the GLWE nodes of the
// len(a) + len(b) product bits.
inline std::vector<int> append_uint_multiply(FheCircuit& c, std::vector<int> a, std::vector<int> b) {
  if (a.size() < b.size()) std::swap(a, b);
  const auto [a_lo, a_hi] = partition_integer(a.size());
  const auto [b_lo, b_hi] = partition_integer(b.size());
  const std::vector<int> al(a.begin(), a.begin() + a_lo), ah(a.begin() + a_lo, a.end());
  const std::vector<int> bl(b.begin(), b.begin() + b_lo), bh(b.begin() + b_lo, b.end());
  if (a_hi == 0 && b_hi == 0) {
    std::vector<int> in = a;
    in.insert(in.end(), b.begin(), b.end());
    return insert_mux_circuit(c, MuxCircuit::unsigned_multiplier((std::uint32_t)a.size(), (std::uint32_t)b.size()), in);
  }
  if (b_hi == 0) {  // a_lo * b + ((a_hi * b) << a_lo): the low word passes through, the rest goes through an adder
    const std::vector<int> ll = append_uint_multiply(c, al, bl), hl = append_uint_multiply(c, ah, bl);
    std::vector<int> in;
    for (std::size_t i = 0; i < b_lo; i++) { in.push_back(glwe_to_ggsw(c, ll[a_lo + i])); in.push_back(glwe_to_ggsw(c, hl[i])); }
    for (std::size_t i = b_lo; i < hl.size(); i++) in.push_back(glwe_to_ggsw(c, hl[i]));
    const std::vector<int> sum = insert_mux_circuit(c, MuxCircuit::ripple_carry_adder((std::uint32_t)b_lo, (std::uint32_t)(a_hi + b_lo)), in);
    std::vector<int> out(ll.begin(), ll.begin() + a_lo);
    out.insert(out.end(), sum.begin(), sum.end());
    return out;
  }
  const std::vector<int> ll = append_uint_multiply(c, al, bl), lh = append_uint_multiply(c, al, bh);
  const std::vector<int> hl = append_uint_multiply(c, ah, bl), hh = append_uint_multiply(c, ah, bh);
  const std::vector<int>* src[4] = {&ll, &hl, &lh, &hh};
  std::size_t pos[4] = {0, 0, 0, 0};
  std::vector<int> bits;
  auto take = [&](std::initializer_list<int> which, std::size_t run) {
    for (std::size_t i = 0; i < run; i++)
      for (int w : which) bits.push_back((*src[w])[pos[w] + i]);
    for (int w : which) pos[w] += run;
  };
  take({0}, b_lo); take({0, 2}, a_lo - b_lo); take({0, 1, 2}, b_lo); take({1, 2, 3}, b_hi); take({1, 3}, a_hi - b_hi); take({3}, b_hi);
  std::vector<int> sel;
  for (int n : bits) sel.push_back(glwe_to_ggsw(c, n));
  return insert_mux_circuit(c, MuxCircuit::gradeschool_reduce((std::uint32_t)a.size(), (std::uint32_t)b.size()), sel);
}

}  // namespace spf
