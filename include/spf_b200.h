/*
 * spf_b200.h -- C ABI of libspf_b200.so, the B200-native TFHE bootstrapping engine that slots in
 * under parasol_runtime's Evaluation / CircuitProcessor::exec_op.
 *
 * The reference (Sunscreen-tech/spf v0.9.0) has no FFI of its own: the seam is a set of plain
 * Rust calls on `Evaluation` (parasol_runtime/src/crypto/evaluation.rs) dispatched one task at
 * a time from CircuitProcessor::exec_op (parasol_runtime/src/circuit_processor/mod.rs:255-546).
 * Each entry point below names the reference method it replaces.  Differences that are
 * deliberate: every op is BATCHED (`batch` independent inputs, contiguous), because the GPU is
 * fed from the runtime's ready-queue rather than one rayon task at a time.
 *
 * Conventions
 *  - All buffers are caller-owned, contiguous, in the reference's own flat layouts
 *    (sunscreen_tfhe/src/entities/, OverlaySize::size): element = u64 torus value or
 *    Complex<f64> = (re, im) pair of doubles.  FFT-domain data (GGSW, keys) is in the
 *    reference's natural bin order and scale (unnormalised forward DFT).
 *  - Functions return 0 on success, a negative spf_status otherwise; they never throw or abort.
 *    The reference panics on wrong sizes (dst.rs:520-523) -- here that is SPF_E_INVALID.
 *    spf_b200_last_error() returns the message of the last failing call on that context (or of
 *    the last failing spf_b200_create when ctx is NULL).
 *  - `spf_b200_*`    : host pointers; the call copies in, computes on the GPU, copies out, and
 *                      returns when the outputs are valid (what Evaluation's methods do).
 *    `spf_b200_dev_*`: device pointers, asynchronous on `stream` (a cudaStream_t passed as
 *                      void*, NULL = the context's own stream).  Device-resident FFT-domain
 *                      ciphertexts (GGSW) carry a 2^-10 scale factor (see DESIGN.md); they only
 *                      ever travel between spf_b200_dev_* calls.
 *  - Device-pointer ops of one context share grow-only device scratch (PBS outputs, keyswitch digit
 *    states): issue them on ONE stream at a time, or serialise streams with events; independent
 *    pipelines use independent contexts.
 *  - A context is bound to one CUDA device and may be used from one thread at a time (the
 *    reference allows only one dispatching thread as well: CircuitProcessor methods take
 *    &mut self, circuit_processor/mod.rs:125-130).
 *  - There is no CPU fallback: without a usable CUDA device spf_b200_create fails.
 */
#ifndef SPF_B200_H
#define SPF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  SPF_OK = 0,
  SPF_E_INVALID = -1,     /* bad argument / size mismatch (reference: panic in assert_is_valid) */
  SPF_E_UNSUPPORTED = -2, /* parameter set the sm_100a kernels are not specialised for */
  SPF_E_CUDA = -3,        /* CUDA runtime error; message in spf_b200_last_error */
  SPF_E_GRAPH = -4        /* malformed graph (reference: RuntimeError, runtime_error.rs:8) */
} spf_status;

/* RadixDecomposition (sunscreen_tfhe/src/params.rs) */
typedef struct { uint32_t radix_log; uint32_t count; } spf_radix;

/* Params (parasol_runtime/src/params.rs:59-91), flattened.  spf_b200_default_128 fills in
 * DEFAULT_128 (params.rs:107-134). */
typedef struct {
  uint32_t lwe_n;    /* l0_params.dim                        637     */
  double   lwe_std;  /* l0_params.std                        7.25e-5 */
  uint32_t glwe_k;   /* l1_params.dim.size                   1       */
  uint32_t glwe_n;   /* l1_params.dim.polynomial_degree      2048    */
  double   glwe_std; /* l1_params.std                        7e-16   */
  spf_radix cbs, pbs, ks, pfks, ss, tr;
} spf_params;

typedef struct spf_b200_ctx spf_b200_ctx;

void spf_b200_default_128(spf_params *p);

/* Entity sizes in elements (u64 or complex) for the given params; the OverlaySize::size
 * functions of sunscreen_tfhe/src/entities (SURVEY.md section 8). */
size_t spf_b200_len_lwe_l0(const spf_params *p);   /* n+1                       638   */
size_t spf_b200_len_lwe_l1(const spf_params *p);   /* kN+1                      2049  */
size_t spf_b200_len_glwe_l1(const spf_params *p);  /* (k+1)N                    4096  */
size_t spf_b200_len_glev_l1(const spf_params *p);  /* l_cbs (k+1) N             16384 */
size_t spf_b200_len_ggsw_l1(const spf_params *p);  /* (k+1) l_cbs (k+1) N/2 c64 16384 */
size_t spf_b200_len_bsk(const spf_params *p);      /* BootstrapKeyFft   (bootstrap_key.rs:122-124) */
size_t spf_b200_len_ksk(const spf_params *p);      /* LweKeyswitchKey   (lwe_keyswitch_key.rs:27-36) */
size_t spf_b200_len_ssk(const spf_params *p);      /* SchemeSwitchKeyFft */
size_t spf_b200_len_ak(const spf_params *p);       /* AutomorphismKeyFft (automorphism_key_fft.rs:25-27) */

/* Evaluation::new(Arc<ComputeKey>, &Params, &Encryption) (evaluation.rs:161-197): uploads the
 * four arrays of ComputeKey {bs_key, ks_key, ss_key, auto_key} (crypto/keys.rs:306-318) to
 * `device`.  Lengths are element counts and must equal spf_b200_len_*.  FFT keys are complex
 * (re, im) pairs exactly as ComputeKey serialises them. */
int spf_b200_create(const spf_params *params, const double *bsk_fft, size_t bsk_len, const uint64_t *ksk,
                    size_t ksk_len, const double *ssk_fft, size_t ssk_len, const double *ak_fft, size_t ak_len,
                    int device, spf_b200_ctx **out);
/* Same, with the key arrays already resident on `device` in the reference layout (used after a
 * one-time NCCL / peer broadcast of the compute key to every GPU of a box). */
int spf_b200_create_from_device(const spf_params *params, const double *d_bsk_fft, size_t bsk_len,
                                const uint64_t *d_ksk, size_t ksk_len, const double *d_ssk_fft, size_t ssk_len,
                                const double *d_ak_fft, size_t ak_len, int device, spf_b200_ctx **out);
void spf_b200_destroy(spf_b200_ctx *ctx);
const char *spf_b200_last_error(const spf_b200_ctx *ctx);
/* Number of CUDA kernels this context has launched so far (bench.py's gpu_launches). */
uint64_t spf_b200_kernel_launches(const spf_b200_ctx *ctx);
int spf_b200_device(const spf_b200_ctx *ctx);
int spf_b200_synchronize(spf_b200_ctx *ctx);

/* ---- host-pointer ops: one call == `batch` calls of the reference method ---------------- */

/* Evaluation::circuit_bootstrap (evaluation.rs:211-225) ->
 * circuit_bootstrap_via_trace_and_scheme_switch (circuit_bootstrapping.rs:342-384).
 * lwe0_in [batch][n+1] u64 -> ggsw_out [batch][len_ggsw_l1] complex. */
int spf_b200_circuit_bootstrap(spf_b200_ctx *ctx, double *ggsw_out, const uint64_t *lwe0_in, size_t batch);

/* generalized_programmable_bootstrap (programmable_bootstrapping.rs:342-410).
 * lut_glwe: one trivial-GLWE LUT [len_glwe_l1] shared by the batch. glwe_out [batch][len_glwe_l1]. */
int spf_b200_programmable_bootstrap(spf_b200_ctx *ctx, uint64_t *glwe_out, const uint64_t *lwe0_in,
                                    const uint64_t *lut_glwe, uint32_t log_chi, uint32_t log_v, size_t batch);

/* KeylessEvaluation::cmux (evaluation.rs:68-83): out = sel ? b : a.  sel [batch][len_ggsw_l1]. */
int spf_b200_cmux(spf_b200_ctx *ctx, uint64_t *glwe_out, const double *sel_ggsw, const uint64_t *a,
                  const uint64_t *b, size_t batch);
/* KeylessEvaluation::glev_cmux (evaluation.rs:86-101); a, b, out are GLEVs [batch][len_glev_l1]. */
int spf_b200_glev_cmux(spf_b200_ctx *ctx, uint64_t *glev_out, const double *sel_ggsw, const uint64_t *a,
                       const uint64_t *b, size_t batch);
/* KeylessEvaluation::multiply_glwe_ggsw (evaluation.rs:104-123). */
int spf_b200_multiply_glwe_ggsw(spf_b200_ctx *ctx, uint64_t *glwe_out, const uint64_t *glwe, const double *ggsw,
                                size_t batch);
/* Evaluation::keyswitch_lwe_l1_lwe_l0 (evaluation.rs:243-252). [batch][kN+1] -> [batch][n+1]. */
int spf_b200_keyswitch_lwe_l1_lwe_l0(spf_b200_ctx *ctx, uint64_t *lwe0_out, const uint64_t *lwe1_in, size_t batch);
/* KeylessEvaluation::sample_extract_l1 (evaluation.rs:126-133); idx[batch] or NULL with idx_all. */
int spf_b200_sample_extract_l1(spf_b200_ctx *ctx, uint64_t *lwe1_out, const uint64_t *glwe_in, const uint32_t *idx,
                               uint32_t idx_all, size_t batch);
/* Evaluation::scheme_switch (evaluation.rs:231-240): GLEV [batch][len_glev_l1] -> GGSW-FFT. */
int spf_b200_scheme_switch(spf_b200_ctx *ctx, double *ggsw_out, const uint64_t *glev_in, size_t batch);
/* sunscreen_tfhe::ops::automorphisms::trace (automorphisms/mod.rs:53-85). */
int spf_b200_trace(spf_b200_ctx *ctx, uint64_t *glwe_out, const uint64_t *glwe_in, size_t batch);
/* KeylessEvaluation::{not,xor,mul_xn} (evaluation.rs:48-65). */
int spf_b200_not(spf_b200_ctx *ctx, uint64_t *glwe_out, const uint64_t *glwe_in, size_t batch);
int spf_b200_xor(spf_b200_ctx *ctx, uint64_t *glwe_out, const uint64_t *a, const uint64_t *b, size_t batch);
int spf_b200_mul_xn(spf_b200_ctx *ctx, uint64_t *glwe_out, const uint64_t *glwe_in, uint32_t n, size_t batch);
/* Encryption::encrypt_rlwe_l1 / encrypt_rlev_l1 (parasol_runtime/src/crypto/encryption.rs:205-249) =
 * rlwe_encrypt_public (sunscreen_tfhe/src/ops/encryption/rlwe_encryption.rs:108-160), batched, with the randomness
 * the reference draws inside (binary u, Gaussian e0 / e1; returned there as RlwePublicEncryptionRandomness) supplied
 * by the caller, who owns the cryptographic RNG:  glwe_out[b] = (p0 * u[b] + e0[b], p1 * u[b] + e1[b] + encoded_msg[b])
 * over Z_2^64[X]/(X^N + 1), exact integer arithmetic (polynomial_external_mad), for any u64 multiplier u.
 * public_key: RlwePublicKey [2][N] (an encryption of zero, shared by the batch); encoded_msg, u, e0, e1: [batch][N];
 * an RLEV encryption is cbs.count batch items with encoded_msg * q / B^(j+1).  k = 1, N = 2048 only. */
int spf_b200_rlwe_encrypt_public(spf_b200_ctx *ctx, uint64_t *glwe_out, const uint64_t *public_key,
                                 const uint64_t *encoded_msg, const uint64_t *u, const uint64_t *e0, const uint64_t *e1,
                                 size_t batch);

/* ---- device-pointer ops (asynchronous on `stream`) --------------------------------------- */

/* scratch_glwe: device scratch of batch*len_glwe_l1 u64 for the PBS output (may be NULL: the
 * context's own grow-only scratch is used).  ggsw_out is device-scale (2^-10) unless
 * reference_scale != 0. */
int spf_b200_dev_circuit_bootstrap(spf_b200_ctx *ctx, double *d_ggsw_out, const uint64_t *d_lwe0_in, size_t batch,
                                   int reference_scale, void *stream);
int spf_b200_dev_programmable_bootstrap(spf_b200_ctx *ctx, uint64_t *d_glwe_out, const uint64_t *d_lwe0_in,
                                        const uint64_t *d_lut_glwe, uint32_t log_chi, uint32_t log_v, size_t batch,
                                        void *stream);
/* d_sel_ggsw is device-scale.  ggsw_stride: elements between consecutive selectors (0 = one
 * selector shared by the whole batch). */
int spf_b200_dev_cmux(spf_b200_ctx *ctx, uint64_t *d_glwe_out, const double *d_sel_ggsw, size_t ggsw_stride,
                      const uint64_t *d_a, const uint64_t *d_b, size_t batch, void *stream);
int spf_b200_dev_keyswitch_lwe_l1_lwe_l0(spf_b200_ctx *ctx, uint64_t *d_lwe0_out, const uint64_t *d_lwe1_in,
                                         size_t batch, void *stream);
int spf_b200_dev_sample_extract_l1(spf_b200_ctx *ctx, uint64_t *d_lwe1_out, const uint64_t *d_glwe_in,
                                   const uint32_t *d_idx, uint32_t idx_all, size_t batch, void *stream);
int spf_b200_dev_rlwe_encrypt_public(spf_b200_ctx *ctx, uint64_t *d_glwe_out, const uint64_t *d_public_key,
                                     const uint64_t *d_encoded_msg, const uint64_t *d_u, const uint64_t *d_e0,
                                     const uint64_t *d_e1, size_t batch, void *stream);
/* dst = src * 2^-10 (to_device != 0) or * 2^10: converts GGSW-FFT data between the reference
 * scale and the device scale; n complex elements. */
int spf_b200_dev_fft_rescale(spf_b200_ctx *ctx, double *d_dst, const double *d_src, size_t n, int to_device,
                             void *stream);

/* ---- graph execution: CircuitProcessor::{spawn_graph, run_graph_blocking} --------------------
 * (parasol_runtime/src/circuit_processor/mod.rs:573-655), level-synchronous and batched: all
 * nodes of one (dependency level, op) group run as ONE kernel launch; intermediates stay in HBM. */

/* FheOp (parasol_runtime/src/fhe_circuit.rs:34-127), same order. */
typedef enum {
  SPF_OP_INPUT_LWE0 = 0, SPF_OP_INPUT_LWE1, SPF_OP_INPUT_GLWE1, SPF_OP_INPUT_GGSW1, SPF_OP_INPUT_GLEV1,
  SPF_OP_OUTPUT_LWE0, SPF_OP_OUTPUT_LWE1, SPF_OP_OUTPUT_GLWE1, SPF_OP_OUTPUT_GGSW1, SPF_OP_OUTPUT_GLEV1,
  SPF_OP_SAMPLE_EXTRACT, SPF_OP_KEYSWITCH_L1_TO_L0, SPF_OP_NOT, SPF_OP_GLWE_ADD, SPF_OP_CMUX, SPF_OP_GLEV_CMUX,
  SPF_OP_MULTIPLY_GGSW_GLWE, SPF_OP_CIRCUIT_BOOTSTRAP, SPF_OP_SCHEME_SWITCH,
  SPF_OP_ZERO_LWE0, SPF_OP_ONE_LWE0, SPF_OP_ZERO_GLWE1, SPF_OP_ONE_GLWE1, SPF_OP_ZERO_GGSW1, SPF_OP_ONE_GGSW1,
  SPF_OP_ZERO_GLEV1, SPF_OP_ONE_GLEV1, SPF_OP_RETIRE, SPF_OP_NOP, SPF_OP_MUL_XN
} spf_op;

/* One graph node.  `in` holds producer node indices by FheEdge (fhe_circuit.rs:174-198), -1 = none:
 *   unary ops: in[0] = Unary;  GlweAdd: in[0] = Left, in[1] = Right;
 *   CMux / GlevCMux: in[0] = Sel, in[1] = Low (selected when sel = 0), in[2] = High;
 *   MultiplyGgswGlwe: in[0] = Glwe, in[1] = Ggsw.
 * `arg` is SampleExtract's index / MulXN's exponent.  `io` is the host ciphertext buffer of an
 * Input* node (read at every run) or Output* node (written at every run), reference layouts. */
typedef struct {
  uint32_t op;
  uint32_t arg;
  int32_t in[3];
  void *io;
} spf_node;

typedef struct spf_b200_graph spf_b200_graph;

/* Validates (Task::validate, circuit_processor/task.rs:24-179: wrong ciphertext kind, missing
 * input, illegal sample-extract index, plus cycles -> SPF_E_GRAPH), levelises, allocates the
 * device arena and uploads the per-group pointer tables.  Nodes may come in any order. */
int spf_b200_graph_build(spf_b200_ctx *ctx, const spf_node *nodes, size_t n_nodes, spf_b200_graph **out);
/* One blocking execution (run_graph_blocking): inputs H2D, all levels, outputs D2H. */
int spf_b200_graph_run(spf_b200_graph *graph);
void spf_b200_graph_destroy(spf_b200_graph *graph);
int spf_b200_graph_levels(const spf_b200_graph *graph);
uint64_t spf_b200_graph_launches(const spf_b200_graph *graph); /* kernel launches of the last run */
/* Re-points the io buffer of an Input* / Output* node of a built graph: one validated, levelised,
 * device-resident graph then serves every invocation of the same instruction shape (the reference
 * rebuilds and re-levelises the MUX circuit per instruction dispatch, fhe_circuit.rs:473-494).
 *
 * CIPHERTEXT HANDLES.  An io pointer (here and in spf_node.io) may be
 *   - page-locked host memory (spf_b200_host_alloc, cudaHostAlloc, a caller's cudaHostRegister): plain DMA;
 *   - pageable host memory: page-locked by spf_b200_graph_build, staged through the graph's own page-locked slab when it
 *     arrives through spf_b200_graph_set_io (no per-call registration);
 *   - DEVICE memory (cudaMalloc / a torch tensor / spf_b200_device_alloc): a ciphertext that never leaves HBM -- the
 *     role of the reference's Arc<AtomicRefCell<Option<Ciphertext>>> task outputs shared between graphs
 *     (circuit_processor/task.rs:10-16): the Output* node of graph k and the Input* node of graph k + 1 name the same
 *     device buffer, the copies are device-to-device, GGSWs keep the device scale (2^-10) and, like the reference's
 *     L1GgswCiphertext (encryption.rs:94-98), never reach the host.
 * The kind is detected with cudaPointerGetAttributes. */
int spf_b200_graph_set_io(spf_b200_graph *graph, size_t node, void *io);
/* Device memory for ciphertext handles (cudaMalloc / cudaFree on the context's device). */
int spf_b200_device_alloc(spf_b200_ctx *ctx, void **out, size_t bytes);
int spf_b200_device_free(spf_b200_ctx *ctx, void *p);

/* ---- asynchronous execution: CircuitProcessor::spawn_graph, CompletionHandler, flow control --------------------
 * (parasol_runtime/src/circuit_processor/mod.rs:130-253,573-623; completion_handler.rs:14-56).
 * spf_b200_graph_spawn enqueues one whole run of `graph` on the graph's own CUDA stream and returns; on_complete(user,
 * status, message) fires exactly once when every op of the run has retired, with the FIRST error of the run (0 and
 * NULL = none) -- CompletionHandler's callback with Option<RuntimeError>.  Outputs must not be read before it fires.
 * `after`: graphs whose last spawned run must complete first (ordered on the device by events, the host does not wait);
 * a run whose dependency failed retires as a no-op with the dependency's error, as tasks do once
 * CompletionHandler::error is set.  At most spf_b200_set_max_in_flight (default 4) spawned runs are between dispatch and
 * completion per context: further spawns block in the caller, as dispatch() blocks on the flow-control channel.
 * The callback runs on a CUDA-internal thread and must not call CUDA or spf_b200 functions.  Sharded graphs
 * (world > 1) are not spawned.  spf_b200_graph_wait blocks until the graph's last run (callback included) is over
 * and returns its status. */
typedef void (*spf_completion_fn)(void *user, int status, const char *message);
int spf_b200_graph_spawn(spf_b200_graph *graph, spf_b200_graph *const *after, size_t n_after,
                         spf_completion_fn on_complete, void *user);
int spf_b200_graph_wait(spf_b200_graph *graph);
const char *spf_b200_graph_status_message(const spf_b200_graph *graph); /* error of the last run (spawned or blocking), "" if none */
int spf_b200_set_max_in_flight(spf_b200_ctx *ctx, int n);
/* Page-locked host memory for ciphertext buffers.  Input and Output node buffers that are already page-locked (this
 * allocator, cudaHostAlloc, a cudaHostRegister done by the caller) are used as they are; any other buffer is registered
 * by the graph on first use, which is slow when there are hundreds of them (allocate ONE slab and slice it). */
int spf_b200_host_alloc(void **out, size_t bytes);
int spf_b200_host_free(void *p);
/* build + run + destroy */
int spf_b200_run_graph(spf_b200_ctx *ctx, const spf_node *nodes, size_t n_nodes);

/* ---- the same graph sharded over the GPUs of one box (SURVEY.md 8(e)) ---------------------------
 * One process per GPU; every rank builds the same graph over the same inputs and a replica of the
 * compute key.  Work is split two ways:
 *  - each CircuitBootstrap group (a dependency level's ready batch) is laid out as `world` equal
 *    chunks; rank r bootstraps chunk r;
 *  - the ops between two bootstrap levels (CMux / Not / GlweAdd / MulXN trees and the SampleExtract ->
 *    KeyswitchL1toL0 chains behind them) are partitioned by connected component of their data edges:
 *    one instruction's MUX tree runs on ONE rank, trees are spread over the ranks by size.
 * After every CircuitBootstrap group (GGSWs, 256 KiB each) and every KeyswitchL1toL0 group (L0 LWEs,
 * 5 KB each) the run calls `exchange`, which must complete the buffer on every rank (an in-place
 * all-gather: on entry chunk r of d_buf[world][chunk_bytes] is valid on rank r, on return -- in stream
 * order -- all chunks are valid everywhere).  spf_b200/multi.py provides the NCCL implementation.
 * Output* nodes fed by a MUX tree are written on the owning rank only (spf_b200_graph_output_rank);
 * everything else is written on every rank.
 * Returns nonzero from `exchange` abort the run with SPF_E_GRAPH. */
typedef int (*spf_exchange_fn)(void *user, void *d_buf, size_t chunk_bytes, int world, void *stream);
int spf_b200_graph_build_sharded(spf_b200_ctx *ctx, const spf_node *nodes, size_t n_nodes, int world,
                                 spf_b200_graph **out);
int spf_b200_graph_run_sharded(spf_b200_graph *graph, int rank, int world, spf_exchange_fn exchange, void *user);
/* ---- peer-memory exchange for sharded runs (no NCCL on the data path) --------------------------------
 * With the arenas of all ranks mapped into every process, spf_b200_graph_run_sharded(graph, rank, world, NULL, NULL)
 * replaces the exchange callback by direct P2P traffic over NVLink: the scheme-switch kernel stores every GGSW it
 * produces at the same offset into the arena of every rank while it computes the next one (the all-gather is fused
 * into the kernel that produces the data), keyswitch outputs are broadcast by a small copy kernel, and dependency
 * levels are separated by a flag barrier through peer memory (a rank that never arrives makes the run fail with
 * SPF_E_GRAPH after a 5 s device-side timeout instead of hanging; the epochs of the ranks then disagree, so the
 * graphs must be rebuilt before another sharded run).  Every rank must build the same graph with the
 * same `world`.  One process per GPU: export with spf_b200_graph_ipc_handle (a 64-byte cudaIpcMemHandle_t), gather
 * the handles on the host, import with spf_b200_graph_open_peers.  Several ranks inside one process (tests):
 * spf_b200_graph_set_peers with the arena addresses. */
void *spf_b200_graph_arena(const spf_b200_graph *graph);
int spf_b200_graph_ipc_handle(spf_b200_graph *graph, uint8_t *handle_out /* 64 bytes */);
int spf_b200_graph_open_peers(spf_b200_graph *graph, int rank, int world, const uint8_t *handles /* world x 64 */);
int spf_b200_graph_set_peers(spf_b200_graph *graph, int rank, int world, void *const *arenas);

/* Host-only planning (no GPU, no context): validates the graph exactly as spf_b200_graph_build does and returns,
 * per node, its dependency level (after bootstrap-stage alignment) and the rank that computes it in a run sharded
 * over `world` ranks (-1 = every rank).  level_out / owner_out may be NULL.  Malformed graphs: SPF_E_GRAPH with
 * the message in spf_b200_last_error(NULL). */
int spf_b200_graph_plan(const spf_params *params, const spf_node *nodes, size_t n_nodes, int world,
                        int32_t *level_out, int32_t *owner_out);
/* Rank that writes Output* node `node` in a sharded run; -1 = every rank; -2 = not an Output* node. */
int spf_b200_graph_output_rank(const spf_b200_graph *graph, size_t node);

/* ---- one process, every GPU of a box: spf_b200_box ---------------------------------------------------
 * A box is N ranks (1 <= N <= 8), each a context on its own device, owned by ONE handle and driven from ONE thread --
 * the shape of parasol_runtime's CircuitProcessor (one dispatching thread, &mut self).  The same device may appear
 * more than once (several ranks on one GPU).  Distinct devices must reach each other as peers (cudaDeviceCanAccessPeer
 * both ways, else SPF_E_UNSUPPORTED); peer access is enabled for every pair.  The compute key is uploaded once, to
 * rank 0's device, and replicated device to device over NVLink in a fan-out tree (0 -> 1, {0,1} -> {2,3}, ...); each
 * rank's context is then made as spf_b200_create_from_device makes it.  Errors of box calls: spf_b200_box_last_error
 * (box NULL: the last failing spf_b200_box_create* of this thread). */
typedef struct spf_b200_box spf_b200_box;
typedef struct spf_b200_box_graph spf_b200_box_graph;
int spf_b200_box_create(const spf_params *params, const double *bsk_fft, size_t bsk_len, const uint64_t *ksk,
                        size_t ksk_len, const double *ssk_fft, size_t ssk_len, const double *ak_fft, size_t ak_len,
                        const int *devices, int n, spf_b200_box **out);
int spf_b200_box_create_from_serialized(const spf_params *params, const uint8_t *buf, size_t len, const int *devices,
                                        int n, spf_b200_box **out);
/* Joins the box's worker threads and drops its contexts; box graphs still alive keep what they use. */
void spf_b200_box_destroy(spf_b200_box *box);
const char *spf_b200_box_last_error(const spf_b200_box *box);
int spf_b200_box_size(const spf_b200_box *box);
int spf_b200_box_device(const spf_b200_box *box, int rank);
/* Rank `rank`'s context, for spf_b200_dev_* calls on that rank's device.  Owned by the box: do not destroy it. */
spf_b200_ctx *spf_b200_box_context(spf_b200_box *box, int rank);
/* Wall time of the device-to-device replication of the compute key at creation, milliseconds. */
double spf_b200_box_key_replication_ms(const spf_b200_box *box);
/* Elements [offset, offset + count) of key array `which` (0 bs_key, 1 ks_key, 2 ss_key, 3 auto_key) as resident on
 * rank `rank`'s device, copied to `out` in the reference layout and scale (to check a replica against the host key). */
int spf_b200_box_key_slice(spf_b200_box *box, int rank, int which, size_t offset, size_t count, void *out);
/* The split of a batch over n ranks used by the box ops: contiguous ranges, the first batch % n ranks get one extra
 * item (spf_b200/multi.py shard).  Host only. */
void spf_b200_box_shard(size_t batch, int n, int rank, size_t *start, size_t *count);

/* Host-pointer ops over the box: the batch is split by spf_b200_box_shard, every rank runs its slice of the
 * single-context op at the same time (one worker thread per rank, created with the box), the call returns when every
 * output is valid.  Outputs are bit-identical to the single-context op on the same slices. */
int spf_b200_box_circuit_bootstrap(spf_b200_box *box, double *ggsw_out, const uint64_t *lwe0_in, size_t batch);
int spf_b200_box_programmable_bootstrap(spf_b200_box *box, uint64_t *glwe_out, const uint64_t *lwe0_in,
                                        const uint64_t *lut_glwe, uint32_t log_chi, uint32_t log_v, size_t batch);
int spf_b200_box_keyswitch_lwe_l1_lwe_l0(spf_b200_box *box, uint64_t *lwe0_out, const uint64_t *lwe1_in, size_t batch);
int spf_b200_box_cmux(spf_b200_box *box, uint64_t *glwe_out, const double *sel_ggsw, const uint64_t *a,
                      const uint64_t *b, size_t batch);

/* Graphs over the box: spf_b200_graph_build_sharded on every rank with world = N, wired to each other's arenas in
 * this process (the peer-memory exchange of spf_b200_graph_run_sharded: fused GGSW stores, keyswitch broadcast, flag
 * barriers between levels).  Every rank's run is enqueued from the calling thread, level-interleaved across the ranks;
 * everything that could make the host wait on a device is done before the first enqueue, so no rank waits at a barrier
 * for a rank that has not been enqueued.
 * io buffers are host memory or BOX CIPHERTEXT HANDLES (below); one graph may mix both.  Raw device pointers are
 * refused with SPF_E_INVALID (a box needs one copy per rank, and which rank computes an output is known only after
 * sharding).  Output* nodes with a host buffer are written by their owner rank (spf_b200_graph_output_rank; rank 0 for
 * nodes every rank holds).  A handle-bound Output* node is written into every rank's replica: by each rank itself when
 * every rank holds the ciphertext, by the owner over NVLink when one rank computes it (after a barrier that every rank
 * reaches once it has read its handle inputs).  A handle-bound Input* node is read by each rank from its own replica.
 * All handle copies of a rank go through one table-driven copy kernel for the inputs and one for the outputs.
 * Spawn semantics are those of spf_b200_graph_spawn: on_complete fires exactly once per run, after every rank has
 * retired, with the first error of any rank; `after` orders on the device (every rank behind every rank of the
 * dependency); a run whose dependency failed
 * retires as a no-op with that error; at most spf_b200_box_set_max_in_flight (default 4) runs per box are in flight,
 * further spawns block the caller.  A failed run with N > 1 poisons the box graph (rebuild it).  Destroying a box
 * graph waits for its run in flight.
 * PLACEMENT: spf_b200_box_graph_build_on runs the graph on an ordered subset of the box's ranks, its members:
 * ranks[i] is the box rank that runs member i, and the graph is sharded over the n_ranks members exactly as a box graph
 * over a box of n_ranks ranks would be ("rank" above then means member; member 0 writes the host outputs every member
 * holds).  spf_b200_box_graph_build is build_on with ranks 0 .. N - 1.  Independent graphs placed on different ranks
 * run at the same time.  A one-member graph has no peer barriers and runs as a one-rank box does (a failed run does
 * not poison it).  Handle-bound inputs are read from the members' own replicas; handle-bound outputs are written into
 * the replicas of EVERY rank of the box, members or not (a MUX-tree output by its owner member, an output every member
 * holds by each member into its own replica and by member 0 into the replicas of the other ranks), so the next graph
 * reads it wherever it is placed.  `after` may name graphs placed on other ranks: every member waits for every member
 * of the dependency.  Errors (SPF_E_INVALID, the box stays usable): ranks NULL, n_ranks outside 1 .. N, a rank outside
 * 0 .. N - 1, a rank named twice.  spf_b200_box_graph_ranks returns the member count and, if ranks_out is not NULL,
 * stores the members' box ranks in it.
 * HAZARD RULE: a run writes a handle-bound output into every replica, on every rank.  So a graph that writes a handle
 * which another graph reads -- on any rank -- must be spawned with that reader in `after` (and a graph that reads a
 * handle with its writer in `after`), as for DeviceCiphertext handles on one context. */
int spf_b200_box_graph_build(spf_b200_box *box, const spf_node *nodes, size_t n_nodes, spf_b200_box_graph **out);
int spf_b200_box_graph_build_on(spf_b200_box *box, const spf_node *nodes, size_t n_nodes, const int *ranks, int n_ranks,
                                spf_b200_box_graph **out);
int spf_b200_box_graph_ranks(const spf_b200_box_graph *graph, int *ranks_out);
int spf_b200_box_graph_run(spf_b200_box_graph *graph);
int spf_b200_box_graph_spawn(spf_b200_box_graph *graph, spf_b200_box_graph *const *after, size_t n_after,
                             spf_completion_fn on_complete, void *user);
int spf_b200_box_graph_wait(spf_b200_box_graph *graph);
const char *spf_b200_box_graph_status_message(const spf_b200_box_graph *graph);
int spf_b200_box_graph_set_io(spf_b200_box_graph *graph, size_t node, void *io);
void spf_b200_box_graph_destroy(spf_b200_box_graph *graph);
int spf_b200_box_graph_levels(const spf_b200_box_graph *graph);
uint64_t spf_b200_box_graph_launches(const spf_b200_box_graph *graph); /* kernel launches of the last run, all ranks */
int spf_b200_box_set_max_in_flight(spf_b200_box *box, int n);

/* Box ciphertext handles: one ciphertext kept in HBM between box graphs -- the box's DeviceCiphertext.  A handle holds
 * one replica per rank of the box, on that rank's device (a device that appears twice in the box gets two), whatever
 * ranks the graphs that use it are placed on (see PLACEMENT and the HAZARD RULE above).  Pass the handle
 * pointer itself as spf_node.io or to spf_b200_box_graph_set_io: graph k's Output* node and graph k + 1's Input* node
 * name the same handle, nothing crosses PCIe, and `after` orders the two graphs on the devices.  Errors
 * (SPF_E_INVALID): a handle of another box, a handle whose kind is not the node's ciphertext type, a handle on a node
 * that is not Input* / Output*; single-context graphs (spf_b200_graph_build*, spf_b200_graph_set_io) refuse handles.
 * `kind` is the Input* op code of the ciphertext type (SPF_OP_INPUT_LWE0 .. SPF_OP_INPUT_GLEV1).  alloc zero-fills.
 * GGSWs stay in the device scale (x 2^-10) in every replica: write takes and read returns the reference scale.
 * Handles are reference-counted: a box graph holds a reference for every node bound to the handle (dropped on rebind
 * and destroy), free drops the caller's; the memory goes with the last reference.  A handle keeps its box alive.
 * write and read are synchronous; order them against spawned runs with spf_b200_box_graph_wait. */
typedef struct spf_b200_box_ciphertext spf_b200_box_ciphertext;
int spf_b200_box_ciphertext_alloc(spf_b200_box *box, uint32_t kind, spf_b200_box_ciphertext **out);
void spf_b200_box_ciphertext_free(spf_b200_box_ciphertext *h);
/* host -> every replica */
int spf_b200_box_ciphertext_write(spf_b200_box_ciphertext *h, const void *host_src);
/* rank `rank`'s replica -> host */
int spf_b200_box_ciphertext_read(spf_b200_box_ciphertext *h, int rank, void *host_dst);

/* ---- serialized keys and ciphertexts (SURVEY.md 8(f).1) ------------------------------------------
 * The reference serialises with bincode 1.3.3 (Cargo.lock:244-245), fixed-width little-endian
 * integers: every sunscreen_tfhe entity is one sequence `u64 length || elements`
 * (sunscreen_tfhe/src/dst.rs:31-33; Torus<u64> is a transparent u64, math/torus.rs:217-220;
 * Complex<f64> is re, im).  ComputeKey = bs_key || ks_key || ss_key || auto_key
 * (parasol_runtime/src/crypto/keys.rs:306-318).  Parsing follows safe_bincode::deserialize
 * (parasol_runtime/src/safe_bincode.rs:16-27): reads are limited to GetSize::get_size(params)
 * bytes, trailing bytes are allowed, every length must equal the entity's OverlaySize::size
 * (check_is_valid, dst.rs:510-516); violations return SPF_E_INVALID (the reference returns Err).
 * These functions need no GPU and no context; errors are reported through
 * spf_b200_last_error(NULL). */
typedef enum { SPF_CT_LWE0 = 0, SPF_CT_LWE1 = 1, SPF_CT_GLWE1 = 2, SPF_CT_GLEV1 = 3 } spf_ct_kind;

/* exact byte count of bincode::serialize(&ComputeKey) */
size_t spf_b200_serialized_size_compute_key(const spf_params *p);
/* ComputeKey::get_size (keys.rs:326-349), the deserialisation byte limit (>= the exact size) */
size_t spf_b200_serialized_limit_compute_key(const spf_params *p);
/* offsets[i] = byte offset inside buf of the first element of {bs_key, ks_key, ss_key, auto_key};
 * element counts are spf_b200_len_{bsk,ksk,ssk,ak}.  Zero-copy: nothing is allocated. */
int spf_b200_parse_compute_key(const spf_params *params, const uint8_t *buf, size_t len, size_t offsets[4]);
int spf_b200_write_compute_key(const spf_params *params, uint8_t *out, size_t cap, const double *bsk_fft,
                               const uint64_t *ksk, const double *ssk_fft, const double *ak_fft, size_t *written);
/* safe_bincode::deserialize::<ComputeKey> + Evaluation::new in one call: a key file written by the
 * reference loads unmodified. */
int spf_b200_create_from_serialized(const spf_params *params, const uint8_t *buf, size_t len, int device,
                                    spf_b200_ctx **out);
/* L0LweCiphertext / L1LweCiphertext / L1GlweCiphertext / L1GlevCiphertext (encryption.rs:22-116,
 * GetSize at :454-519).  L1GgswCiphertext is deliberately not serialisable (encryption.rs:94-98). */
size_t spf_b200_serialized_size_ciphertext(const spf_params *p, int kind);
int spf_b200_parse_ciphertext(const spf_params *params, int kind, const uint8_t *buf, size_t len, size_t *offset);
int spf_b200_write_ciphertext(const spf_params *params, int kind, const uint64_t *data, uint8_t *out, size_t cap,
                              size_t *written);

/* ---- MUX-circuit generation (SURVEY.md 8(f).3: the step before the path) -------------------------
 * A Parasol instruction becomes a FheCircuit by expanding a multiplexer circuit derived from reduced
 * ordered BDDs (mux_circuits/src/{add,sub,neg,comparisons,and,or,mul}.rs; MuxCircuit::from(&[Bdd]),
 * mux_circuits/src/lib.rs:355-451).  spf_b200_mux_circuit builds the same Boolean functions over the
 * same input order with its own shared-ROBDD manager (host code, no GPU, no context) and returns a
 * flat node list in topological order: node 0 = Zero, node 1 = One, nodes 2..2+inputs = Variable(i),
 * then Mux nodes (sel = a Variable node; output = low when the selector is 0, high when 1,
 * lib.rs:66-76), then one Output(i) node per result bit whose `low` is the node it forwards.
 * Tags equal MuxOp's bincode variant indices (lib.rs:54-94). */
typedef enum { SPF_MUX_ONE = 0, SPF_MUX_ZERO = 1, SPF_MUX_MUX = 2, SPF_MUX_VARIABLE = 3, SPF_MUX_OUTPUT = 4 } spf_mux_op;
typedef struct {
  uint32_t op;  /* spf_mux_op */
  uint32_t arg; /* Variable / Output index */
  int32_t sel, low, high; /* producer node indices, -1 = none */
} spf_mux_node;
typedef enum {
  SPF_MUX_RIPPLE_CARRY_ADDER = 0, /* add.rs:13-56; n, m operand widths; flags bit0 = carry-in first */
  SPF_MUX_FULL_SUBTRACTOR = 1,    /* sub.rs:12-49; flags bit0 = borrow-in first */
  SPF_MUX_NEGATOR = 2,            /* neg.rs:7-27 */
  SPF_MUX_COMPARE = 3,            /* comparisons.rs:127-181; flags bit0 = greater (else less), bit1 = or-equal */
  SPF_MUX_COMPARE_SIGNED = 4,     /* comparisons.rs:79-117; same flags */
  SPF_MUX_COMPARE_EQUAL = 5,      /* comparisons.rs:19-72; flags bit0 = not-equal */
  SPF_MUX_BITWISE = 6,            /* and.rs / or.rs; flags bit0 = or (else and) */
  SPF_MUX_UNSIGNED_MULTIPLIER = 7,/* mul.rs:30-141, n x m -> n + m bits; inputs a[0..n) then b[0..m) */
  SPF_MUX_GRADESCHOOL_REDUCE = 8, /* mul.rs:428-586; inputs ordered by encode_gradeschool_reduction */
  SPF_MUX_BITSHIFT = 9,           /* bitshift.rs:49-157; n value bits + m shift bits, both big-endian; flags bit0 = right,
                                     bits1-2 = mode (0 logical, 1 rotation, 2 arithmetic) */
  SPF_MUX_CONST_MULTIPLIER = 10   /* low n bits of x * flags (the plaintext constant), n <= 32, m = 0; inputs x[0..n)
                                     least significant first, in natural order: depth <= n */
} spf_mux_kind;
/* *out is malloc'ed; release with spf_b200_mux_free.  SPF_E_INVALID for bad sizes. */
int spf_b200_mux_circuit(uint32_t kind, uint32_t n, uint32_t m, uint32_t flags, spf_mux_node **out, size_t *count);
void spf_b200_mux_free(spf_mux_node *nodes);

/* FP64 peak probe used by bench.py for the roofline denominator: runs a dependent-free DFMA
 * loop on every SM and returns achieved TFLOP/s (2 flops per DFMA). */
int spf_b200_fp64_peak(spf_b200_ctx *ctx, double *tflops_out);

#ifdef __cplusplus
}
#endif
#endif
