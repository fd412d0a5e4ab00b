//! Safe Rust layer over `libspf_b200.so`.
//!
//! * [`Evaluation`] has the method names and argument order of `parasol_runtime::crypto::Evaluation`
//!   (`parasol_runtime/src/crypto/evaluation.rs:48-255`), batched: every call takes `batch` ciphertexts laid out
//!   back to back in the reference's flat layouts (`sunscreen_tfhe/src/dst.rs:31-33`; `Torus<u64>` is
//!   `repr(transparent)` over `u64`, `Complex<f64>` is `(re, im)`), so `ct.0.as_slice()` of a reference ciphertext is
//!   exactly what these functions take.
//! * [`Graph`] is `CircuitProcessor::{spawn_graph, run_graph_blocking}` for a whole `FheCircuit`
//!   (`circuit_processor/mod.rs:573-655`): [`Graph::spawn`] returns at once and calls the completion handler with the
//!   first error (`completion_handler.rs:14-56`); [`DeviceCiphertext`] handles keep task outputs in HBM between graphs
//!   (`circuit_processor/task.rs:10-16`).
//! * [`BoxEvaluation`] / [`BoxGraph`]: the same over every GPU of a box, from one thread (one handle, one key upload),
//!   or over chosen ranks of it ([`BoxGraph::build_on`]); [`BoxCiphertext`] handles keep task outputs in HBM between
//!   box graphs, one replica per rank.
//! * module [`parasol`] (feature `parasol`): the glue a maintainer pastes into `parasol_runtime` so that
//!   `CircuitProcessor::exec_op` (`circuit_processor/mod.rs:255-546`) dispatches to the GPU.
//!
//! This crate cannot be compiled in the image the library is developed in (no Rust toolchain); `tests/test_rust_ffi.py`
//! keeps the declarations it relies on in step with the C header.
use spf_b200_sys as sys;
use std::ffi::{c_void, CStr};
use std::os::raw::{c_char, c_int};
use std::ptr::{self, NonNull};
use std::sync::Arc;

use spf_b200_sys::{spf_b200_box as RawBox, spf_b200_box_ciphertext as RawBoxCiphertext, spf_b200_box_graph as RawBoxGraph};
pub use sys::{spf_node, spf_params, spf_radix};

/// `RuntimeError` of the GPU path: the library's status code and message.
#[derive(Debug, Clone)]
pub struct Error {
    pub code: i32,
    pub message: String,
}
impl std::fmt::Display for Error {
    fn fmt(&self, f: &mut std::fmt::Formatter<'_>) -> std::fmt::Result {
        write!(f, "spf_b200 error {}: {}", self.code, self.message)
    }
}
impl std::error::Error for Error {}
pub type Result<T> = std::result::Result<T, Error>;

/// `DEFAULT_128` (`parasol_runtime/src/params.rs:107-134`).
pub fn default_128() -> spf_params {
    let mut p = spf_params::default();
    unsafe { sys::spf_b200_default_128(&mut p) };
    p
}

struct Ctx(NonNull<sys::spf_b200_ctx>);
unsafe impl Send for Ctx {}
unsafe impl Sync for Ctx {} // the library serialises per call; graphs carry their own streams
impl Drop for Ctx {
    fn drop(&mut self) {
        unsafe { sys::spf_b200_destroy(self.0.as_ptr()) }
    }
}

fn last_error(ctx: *const sys::spf_b200_ctx) -> String {
    let p = unsafe { sys::spf_b200_last_error(ctx) };
    if p.is_null() { String::new() } else { unsafe { CStr::from_ptr(p) }.to_string_lossy().into_owned() }
}

/// `Evaluation` (`evaluation.rs:141-255`) on one B200.  Cloning shares the context.
#[derive(Clone)]
pub struct Evaluation {
    ctx: Arc<Ctx>,
    pub params: spf_params,
}

macro_rules! check {
    ($self:expr, $rc:expr) => {{
        let rc = $rc;
        if rc == 0 { Ok(()) } else { Err(Error { code: rc, message: last_error($self.raw()) }) }
    }};
}

impl Evaluation {
    /// `Evaluation::new(compute_key, params, enc)` (`evaluation.rs:161-197`): the four arrays of `ComputeKey`
    /// (`crypto/keys.rs:306-318`), FFT keys as `(re, im)` pairs.
    pub fn new(params: &spf_params, bs_key: &[f64], ks_key: &[u64], ss_key: &[f64], auto_key: &[f64], device: i32) -> Result<Self> {
        let mut raw = ptr::null_mut();
        let rc = unsafe {
            sys::spf_b200_create(params, bs_key.as_ptr(), bs_key.len() / 2, ks_key.as_ptr(), ks_key.len(), ss_key.as_ptr(),
                                 ss_key.len() / 2, auto_key.as_ptr(), auto_key.len() / 2, device as c_int, &mut raw)
        };
        match NonNull::new(raw) {
            Some(p) if rc == 0 => Ok(Self { ctx: Arc::new(Ctx(p)), params: *params }),
            _ => Err(Error { code: rc, message: last_error(ptr::null()) }),
        }
    }
    /// `safe_bincode::deserialize::<ComputeKey>` + `Evaluation::new` (`safe_bincode.rs:16-27`).
    pub fn from_serialized(params: &spf_params, compute_key_bincode: &[u8], device: i32) -> Result<Self> {
        let mut raw = ptr::null_mut();
        let rc = unsafe { sys::spf_b200_create_from_serialized(params, compute_key_bincode.as_ptr(), compute_key_bincode.len(), device as c_int, &mut raw) };
        match NonNull::new(raw) {
            Some(p) if rc == 0 => Ok(Self { ctx: Arc::new(Ctx(p)), params: *params }),
            _ => Err(Error { code: rc, message: last_error(ptr::null()) }),
        }
    }
    fn raw(&self) -> *mut sys::spf_b200_ctx {
        self.ctx.0.as_ptr()
    }
    fn len(&self, f: unsafe extern "C" fn(*const spf_params) -> usize) -> usize {
        unsafe { f(&self.params) }
    }
    fn expect(&self, what: &str, got: usize, want: usize) -> Result<()> {
        if got == want { Ok(()) } else { Err(Error { code: sys::SPF_E_INVALID, message: format!("{what}: {got} elements, expected {want}") }) }
    }

    /// `Evaluation::circuit_bootstrap` (`evaluation.rs:211-225`): `[batch][n+1]` L0 LWE -> `[batch][len_ggsw_l1]` GGSW-FFT.
    pub fn circuit_bootstrap(&self, output: &mut [f64], input: &[u64]) -> Result<()> {
        let batch = input.len() / self.len(sys::spf_b200_len_lwe_l0);
        self.expect("circuit_bootstrap output", output.len(), 2 * batch * self.len(sys::spf_b200_len_ggsw_l1))?;
        check!(self, unsafe { sys::spf_b200_circuit_bootstrap(self.raw(), output.as_mut_ptr(), input.as_ptr(), batch) })
    }
    /// `generalized_programmable_bootstrap` (`programmable_bootstrapping.rs:342-410`).
    pub fn programmable_bootstrap(&self, output: &mut [u64], input: &[u64], lut: &[u64], log_chi: u32, log_v: u32) -> Result<()> {
        let batch = input.len() / self.len(sys::spf_b200_len_lwe_l0);
        self.expect("programmable_bootstrap output", output.len(), batch * self.len(sys::spf_b200_len_glwe_l1))?;
        check!(self, unsafe { sys::spf_b200_programmable_bootstrap(self.raw(), output.as_mut_ptr(), input.as_ptr(), lut.as_ptr(), log_chi, log_v, batch) })
    }
    /// `KeylessEvaluation::cmux` (`evaluation.rs:68-83`): `output = sel ? b : a`.
    pub fn cmux(&self, output: &mut [u64], sel: &[f64], a: &[u64], b: &[u64]) -> Result<()> {
        let batch = a.len() / self.len(sys::spf_b200_len_glwe_l1);
        self.expect("cmux output", output.len(), a.len())?;
        check!(self, unsafe { sys::spf_b200_cmux(self.raw(), output.as_mut_ptr(), sel.as_ptr(), a.as_ptr(), b.as_ptr(), batch) })
    }
    /// `KeylessEvaluation::glev_cmux` (`evaluation.rs:86-101`).
    pub fn glev_cmux(&self, output: &mut [u64], sel: &[f64], a: &[u64], b: &[u64]) -> Result<()> {
        let batch = a.len() / self.len(sys::spf_b200_len_glev_l1);
        self.expect("glev_cmux output", output.len(), a.len())?;
        check!(self, unsafe { sys::spf_b200_glev_cmux(self.raw(), output.as_mut_ptr(), sel.as_ptr(), a.as_ptr(), b.as_ptr(), batch) })
    }
    /// `KeylessEvaluation::multiply_glwe_ggsw` (`evaluation.rs:104-123`).
    pub fn multiply_glwe_ggsw(&self, output: &mut [u64], glwe: &[u64], ggsw: &[f64]) -> Result<()> {
        let batch = glwe.len() / self.len(sys::spf_b200_len_glwe_l1);
        self.expect("multiply_glwe_ggsw output", output.len(), glwe.len())?;
        check!(self, unsafe { sys::spf_b200_multiply_glwe_ggsw(self.raw(), output.as_mut_ptr(), glwe.as_ptr(), ggsw.as_ptr(), batch) })
    }
    /// `Evaluation::keyswitch_lwe_l1_lwe_l0` (`evaluation.rs:243-252`).
    pub fn keyswitch_lwe_l1_lwe_l0(&self, output: &mut [u64], input: &[u64]) -> Result<()> {
        let batch = input.len() / self.len(sys::spf_b200_len_lwe_l1);
        self.expect("keyswitch output", output.len(), batch * self.len(sys::spf_b200_len_lwe_l0))?;
        check!(self, unsafe { sys::spf_b200_keyswitch_lwe_l1_lwe_l0(self.raw(), output.as_mut_ptr(), input.as_ptr(), batch) })
    }
    /// `KeylessEvaluation::sample_extract_l1` (`evaluation.rs:126-133`), one index for the whole batch.
    pub fn sample_extract_l1(&self, output: &mut [u64], input: &[u64], idx: usize) -> Result<()> {
        let batch = input.len() / self.len(sys::spf_b200_len_glwe_l1);
        self.expect("sample_extract output", output.len(), batch * self.len(sys::spf_b200_len_lwe_l1))?;
        check!(self, unsafe { sys::spf_b200_sample_extract_l1(self.raw(), output.as_mut_ptr(), input.as_ptr(), ptr::null(), idx as u32, batch) })
    }
    /// `Evaluation::scheme_switch` (`evaluation.rs:231-240`).
    pub fn scheme_switch(&self, output: &mut [f64], input: &[u64]) -> Result<()> {
        let batch = input.len() / self.len(sys::spf_b200_len_glev_l1);
        self.expect("scheme_switch output", output.len(), 2 * batch * self.len(sys::spf_b200_len_ggsw_l1))?;
        check!(self, unsafe { sys::spf_b200_scheme_switch(self.raw(), output.as_mut_ptr(), input.as_ptr(), batch) })
    }
    /// `sunscreen_tfhe::ops::automorphisms::trace` (`automorphisms/mod.rs:53-85`).
    pub fn trace(&self, output: &mut [u64], input: &[u64]) -> Result<()> {
        let batch = input.len() / self.len(sys::spf_b200_len_glwe_l1);
        self.expect("trace output", output.len(), input.len())?;
        check!(self, unsafe { sys::spf_b200_trace(self.raw(), output.as_mut_ptr(), input.as_ptr(), batch) })
    }
    /// `KeylessEvaluation::not` (`evaluation.rs:48-50`).
    pub fn not(&self, output: &mut [u64], input: &[u64]) -> Result<()> {
        let batch = input.len() / self.len(sys::spf_b200_len_glwe_l1);
        self.expect("not output", output.len(), input.len())?;
        check!(self, unsafe { sys::spf_b200_not(self.raw(), output.as_mut_ptr(), input.as_ptr(), batch) })
    }
    /// `KeylessEvaluation::xor` (`evaluation.rs:53-55`).
    pub fn xor(&self, output: &mut [u64], a: &[u64], b: &[u64]) -> Result<()> {
        let batch = a.len() / self.len(sys::spf_b200_len_glwe_l1);
        self.expect("xor output", output.len(), a.len())?;
        check!(self, unsafe { sys::spf_b200_xor(self.raw(), output.as_mut_ptr(), a.as_ptr(), b.as_ptr(), batch) })
    }
    /// `KeylessEvaluation::mul_xn` (`evaluation.rs:58-65`).
    pub fn mul_xn(&self, output: &mut [u64], input: &[u64], n: usize) -> Result<()> {
        let batch = input.len() / self.len(sys::spf_b200_len_glwe_l1);
        self.expect("mul_xn output", output.len(), input.len())?;
        check!(self, unsafe { sys::spf_b200_mul_xn(self.raw(), output.as_mut_ptr(), input.as_ptr(), n as u32, batch) })
    }
    /// `rlwe_encrypt_public` (`ops/encryption/rlwe_encryption.rs:108-160`) for a batch, randomness supplied by the caller
    /// (the `RlwePublicEncryptionRandomness` the reference returns): `(p0 u + e0, p1 u + e1 + m)`, exact u64 arithmetic.
    #[allow(clippy::too_many_arguments)]
    pub fn rlwe_encrypt_public(&self, output: &mut [u64], public_key: &[u64], encoded_msg: &[u64], u: &[u64], e0: &[u64], e1: &[u64]) -> Result<()> {
        let glwe = self.len(sys::spf_b200_len_glwe_l1);
        let batch = output.len() / glwe;
        self.expect("rlwe_encrypt_public public_key", public_key.len(), glwe)?;
        for (name, x) in [("encoded_msg", encoded_msg), ("u", u), ("e0", e0), ("e1", e1)] {
            self.expect(name, x.len(), batch * glwe / 2)?;
        }
        check!(self, unsafe {
            sys::spf_b200_rlwe_encrypt_public(self.raw(), output.as_mut_ptr(), public_key.as_ptr(), encoded_msg.as_ptr(), u.as_ptr(), e0.as_ptr(), e1.as_ptr(), batch)
        })
    }
    /// Flow control of the asynchronous executor: the bound of `CircuitProcessor::new`'s channel (`mod.rs:95-123`).
    pub fn set_max_in_flight(&self, n: usize) -> Result<()> {
        check!(self, unsafe { sys::spf_b200_set_max_in_flight(self.raw(), n as c_int) })
    }
    /// A ciphertext that lives in HBM: the GPU's `Arc<AtomicRefCell<Option<Ciphertext>>>` (`task.rs:10-16`).
    pub fn alloc_device(&self, bytes: usize) -> Result<DeviceCiphertext> {
        let mut p = ptr::null_mut();
        check!(self, unsafe { sys::spf_b200_device_alloc(self.raw(), &mut p, bytes) })?;
        Ok(DeviceCiphertext { ptr: p, bytes, ev: self.clone() })
    }
}

/// Device memory holding one ciphertext; pass `as_io()` as the `io` of an `Output*` node of one graph and of an
/// `Input*` node of the next.
pub struct DeviceCiphertext {
    ptr: *mut c_void,
    pub bytes: usize,
    ev: Evaluation,
}
unsafe impl Send for DeviceCiphertext {}
impl DeviceCiphertext {
    pub fn as_io(&self) -> *mut c_void {
        self.ptr
    }
}
impl Drop for DeviceCiphertext {
    fn drop(&mut self) {
        unsafe { sys::spf_b200_device_free(self.ev.raw(), self.ptr) };
    }
}

/// A validated, levelised `FheCircuit` resident on the GPU (`spf_b200_graph_build`).
pub struct Graph {
    raw: NonNull<sys::spf_b200_graph>,
    ev: Evaluation,
}
unsafe impl Send for Graph {}

/// `CompletionHandler` (`completion_handler.rs:14-56`): called once, with `None` or the first error.
type Handler = Box<dyn FnOnce(Option<Error>) + Send + 'static>;

unsafe extern "C" fn completion_trampoline(user: *mut c_void, status: c_int, message: *const c_char) {
    let handler: Box<Handler> = Box::from_raw(user as *mut Handler);
    let err = if status == 0 {
        None
    } else {
        let message = if message.is_null() { String::new() } else { CStr::from_ptr(message).to_string_lossy().into_owned() };
        Some(Error { code: status, message })
    };
    // never unwind into C
    let _ = std::panic::catch_unwind(std::panic::AssertUnwindSafe(move || (*handler)(err)));
}

impl Graph {
    /// Validation errors are `Task::validate`'s (`circuit_processor/task.rs:24-179`) plus cycles and stray `Retire`s.
    pub fn build(ev: &Evaluation, nodes: &[spf_node]) -> Result<Self> {
        let mut raw = ptr::null_mut();
        let rc = unsafe { sys::spf_b200_graph_build(ev.raw(), nodes.as_ptr(), nodes.len(), &mut raw) };
        match NonNull::new(raw) {
            Some(p) if rc == 0 => Ok(Self { raw: p, ev: ev.clone() }),
            _ => Err(Error { code: rc, message: last_error(ev.raw()) }),
        }
    }
    /// `CircuitProcessor::run_graph_blocking` (`mod.rs:641-655`).
    pub fn run_blocking(&mut self) -> Result<()> {
        let rc = unsafe { sys::spf_b200_graph_run(self.raw.as_ptr()) };
        if rc == 0 { Ok(()) } else { Err(Error { code: rc, message: last_error(self.ev.raw()) }) }
    }
    /// `CircuitProcessor::spawn_graph` (`mod.rs:573-623`): returns once the run is enqueued (or blocks on flow control);
    /// `on_completion` fires on a CUDA callback thread and must not call back into this crate.  `after`: graphs whose
    /// last spawned run must finish first (device-side ordering).
    pub fn spawn<F: FnOnce(Option<Error>) + Send + 'static>(&mut self, after: &[&Graph], on_completion: F) -> Result<()> {
        let deps: Vec<*mut sys::spf_b200_graph> = after.iter().map(|g| g.raw.as_ptr()).collect();
        let handler: Box<Handler> = Box::new(Box::new(on_completion));
        let user = Box::into_raw(handler) as *mut c_void;
        let rc = unsafe { sys::spf_b200_graph_spawn(self.raw.as_ptr(), deps.as_ptr(), deps.len(), Some(completion_trampoline), user) };
        if rc == 0 {
            Ok(())
        } else {
            drop(unsafe { Box::from_raw(user as *mut Handler) }); // the library did not take the handler
            Err(Error { code: rc, message: last_error(self.ev.raw()) })
        }
    }
    /// Blocks until the last run (callback included) is over and returns its status.
    pub fn wait(&self) -> Result<()> {
        let rc = unsafe { sys::spf_b200_graph_wait(self.raw.as_ptr()) };
        if rc == 0 {
            Ok(())
        } else {
            let m = unsafe { CStr::from_ptr(sys::spf_b200_graph_status_message(self.raw.as_ptr())) }.to_string_lossy().into_owned();
            Err(Error { code: rc, message: m })
        }
    }
    /// Re-point an `Input*` / `Output*` node (host buffer or [`DeviceCiphertext::as_io`]).
    ///
    /// # Safety
    /// `io` must stay valid, and large enough for the node's ciphertext, until the graph has run.
    pub unsafe fn set_io(&mut self, node: usize, io: *mut c_void) -> Result<()> {
        let rc = sys::spf_b200_graph_set_io(self.raw.as_ptr(), node, io);
        if rc == 0 { Ok(()) } else { Err(Error { code: rc, message: last_error(self.ev.raw()) }) }
    }
}
impl Drop for Graph {
    fn drop(&mut self) {
        unsafe { sys::spf_b200_graph_destroy(self.raw.as_ptr()) }
    }
}

/// `Evaluation` over several GPUs of one box, driven from one thread (`spf_b200_box_*`): rank `r` is a context on
/// `devices[r]`; the compute key crosses PCIe once and is replicated device to device.  The batched ops split the batch
/// contiguously over the ranks and run them concurrently; [`BoxGraph`] runs a whole `FheCircuit` over every rank.
#[derive(Clone)]
pub struct BoxEvaluation {
    boxed: Arc<BoxHandle>,
    pub params: spf_params,
}

struct BoxHandle(NonNull<RawBox>);
unsafe impl Send for BoxHandle {}
unsafe impl Sync for BoxHandle {} // one call at a time per box, as for a context
impl Drop for BoxHandle {
    fn drop(&mut self) {
        unsafe { sys::spf_b200_box_destroy(self.0.as_ptr()) }
    }
}

fn box_error(b: *const RawBox) -> String {
    let p = unsafe { sys::spf_b200_box_last_error(b) };
    if p.is_null() { String::new() } else { unsafe { CStr::from_ptr(p) }.to_string_lossy().into_owned() }
}

macro_rules! box_check {
    ($self:expr, $rc:expr) => {{
        let rc = $rc;
        if rc == 0 { Ok(()) } else { Err(Error { code: rc, message: box_error($self.raw()) }) }
    }};
}

impl BoxEvaluation {
    /// `Evaluation::new` for every rank of the box; `devices` may repeat a device (several ranks on one GPU).
    #[allow(clippy::too_many_arguments)]
    pub fn new(params: &spf_params, bs_key: &[f64], ks_key: &[u64], ss_key: &[f64], auto_key: &[f64], devices: &[i32]) -> Result<Self> {
        let devs: Vec<c_int> = devices.iter().map(|&d| d as c_int).collect();
        let mut raw = ptr::null_mut();
        let rc = unsafe {
            sys::spf_b200_box_create(params, bs_key.as_ptr(), bs_key.len() / 2, ks_key.as_ptr(), ks_key.len(), ss_key.as_ptr(),
                                     ss_key.len() / 2, auto_key.as_ptr(), auto_key.len() / 2, devs.as_ptr(), devs.len() as c_int, &mut raw)
        };
        match NonNull::new(raw) {
            Some(p) if rc == 0 => Ok(Self { boxed: Arc::new(BoxHandle(p)), params: *params }),
            _ => Err(Error { code: rc, message: box_error(ptr::null()) }),
        }
    }
    /// `safe_bincode::deserialize::<ComputeKey>` + [`BoxEvaluation::new`].
    pub fn from_serialized(params: &spf_params, compute_key_bincode: &[u8], devices: &[i32]) -> Result<Self> {
        let devs: Vec<c_int> = devices.iter().map(|&d| d as c_int).collect();
        let mut raw = ptr::null_mut();
        let rc = unsafe {
            sys::spf_b200_box_create_from_serialized(params, compute_key_bincode.as_ptr(), compute_key_bincode.len(), devs.as_ptr(),
                                                     devs.len() as c_int, &mut raw)
        };
        match NonNull::new(raw) {
            Some(p) if rc == 0 => Ok(Self { boxed: Arc::new(BoxHandle(p)), params: *params }),
            _ => Err(Error { code: rc, message: box_error(ptr::null()) }),
        }
    }
    fn raw(&self) -> *mut RawBox {
        self.boxed.0.as_ptr()
    }
    fn len(&self, f: unsafe extern "C" fn(*const spf_params) -> usize) -> usize {
        unsafe { f(&self.params) }
    }
    fn expect(&self, what: &str, got: usize, want: usize) -> Result<()> {
        if got == want { Ok(()) } else { Err(Error { code: sys::SPF_E_INVALID, message: format!("{what}: {got} elements, expected {want}") }) }
    }
    /// Number of ranks.
    pub fn size(&self) -> usize {
        unsafe { sys::spf_b200_box_size(self.raw()) as usize }
    }
    /// `Evaluation::circuit_bootstrap` over the box.
    pub fn circuit_bootstrap(&self, output: &mut [f64], input: &[u64]) -> Result<()> {
        let batch = input.len() / self.len(sys::spf_b200_len_lwe_l0);
        self.expect("circuit_bootstrap output", output.len(), 2 * batch * self.len(sys::spf_b200_len_ggsw_l1))?;
        box_check!(self, unsafe { sys::spf_b200_box_circuit_bootstrap(self.raw(), output.as_mut_ptr(), input.as_ptr(), batch) })
    }
    /// `generalized_programmable_bootstrap` over the box.
    pub fn programmable_bootstrap(&self, output: &mut [u64], input: &[u64], lut: &[u64], log_chi: u32, log_v: u32) -> Result<()> {
        let batch = input.len() / self.len(sys::spf_b200_len_lwe_l0);
        self.expect("programmable_bootstrap output", output.len(), batch * self.len(sys::spf_b200_len_glwe_l1))?;
        box_check!(self, unsafe { sys::spf_b200_box_programmable_bootstrap(self.raw(), output.as_mut_ptr(), input.as_ptr(), lut.as_ptr(), log_chi, log_v, batch) })
    }
    /// `Evaluation::keyswitch_lwe_l1_lwe_l0` over the box.
    pub fn keyswitch_lwe_l1_lwe_l0(&self, output: &mut [u64], input: &[u64]) -> Result<()> {
        let batch = input.len() / self.len(sys::spf_b200_len_lwe_l1);
        self.expect("keyswitch output", output.len(), batch * self.len(sys::spf_b200_len_lwe_l0))?;
        box_check!(self, unsafe { sys::spf_b200_box_keyswitch_lwe_l1_lwe_l0(self.raw(), output.as_mut_ptr(), input.as_ptr(), batch) })
    }
    /// `KeylessEvaluation::cmux` over the box: `output = sel ? b : a`.
    pub fn cmux(&self, output: &mut [u64], sel: &[f64], a: &[u64], b: &[u64]) -> Result<()> {
        let batch = a.len() / self.len(sys::spf_b200_len_glwe_l1);
        self.expect("cmux output", output.len(), a.len())?;
        box_check!(self, unsafe { sys::spf_b200_box_cmux(self.raw(), output.as_mut_ptr(), sel.as_ptr(), a.as_ptr(), b.as_ptr(), batch) })
    }
    /// Flow control of spawned box graphs (runs in flight per box).
    pub fn set_max_in_flight(&self, n: usize) -> Result<()> {
        box_check!(self, unsafe { sys::spf_b200_box_set_max_in_flight(self.raw(), n as c_int) })
    }
}

/// A ciphertext kept in HBM with one replica per rank of a box (`spf_b200_box_ciphertext_*`): the box's
/// [`DeviceCiphertext`].  Pass `as_io()` as the `io` of an `Output*` node of one box graph and of an `Input*` node of the
/// next.  Box graphs hold their own references, so the handle may be dropped while a graph still binds it.  GGSWs stay
/// in the device scale in the replicas; `write` takes and `read` returns the reference scale.
pub struct BoxCiphertext {
    raw: NonNull<RawBoxCiphertext>,
    ev: BoxEvaluation,
    pub bytes: usize,
}
unsafe impl Send for BoxCiphertext {}
impl BoxCiphertext {
    /// A zero-filled handle; `kind` is the `Input*` op code of the ciphertext type (`SPF_OP_INPUT_LWE0` ..
    /// `SPF_OP_INPUT_GLEV1`).
    pub fn alloc(ev: &BoxEvaluation, kind: u32) -> Result<Self> {
        let mut raw = ptr::null_mut();
        let rc = unsafe { sys::spf_b200_box_ciphertext_alloc(ev.raw(), kind, &mut raw) };
        let p = match NonNull::new(raw) {
            Some(p) if rc == 0 => p,
            _ => return Err(Error { code: rc, message: box_error(ev.raw()) }),
        };
        let bytes = match kind {
            sys::SPF_OP_INPUT_LWE0 => ev.len(sys::spf_b200_len_lwe_l0) * 8,
            sys::SPF_OP_INPUT_LWE1 => ev.len(sys::spf_b200_len_lwe_l1) * 8,
            sys::SPF_OP_INPUT_GLWE1 => ev.len(sys::spf_b200_len_glwe_l1) * 8,
            sys::SPF_OP_INPUT_GGSW1 => ev.len(sys::spf_b200_len_ggsw_l1) * 16,
            _ => ev.len(sys::spf_b200_len_glev_l1) * 8,
        };
        Ok(Self { raw: p, ev: ev.clone(), bytes })
    }
    pub fn as_io(&self) -> *mut c_void {
        self.raw.as_ptr() as *mut c_void
    }
    /// One host ciphertext (reference layout and scale) to every rank's replica.
    pub fn write<T: Copy>(&self, src: &[T]) -> Result<()> {
        self.ev.expect("BoxCiphertext::write bytes", std::mem::size_of_val(src), self.bytes)?;
        box_check!(self.ev, unsafe { sys::spf_b200_box_ciphertext_write(self.raw.as_ptr(), src.as_ptr() as *const c_void) })
    }
    /// Rank `rank`'s replica to the host (reference layout and scale).
    pub fn read<T: Copy>(&self, rank: usize, dst: &mut [T]) -> Result<()> {
        self.ev.expect("BoxCiphertext::read bytes", std::mem::size_of_val(dst), self.bytes)?;
        box_check!(self.ev, unsafe { sys::spf_b200_box_ciphertext_read(self.raw.as_ptr(), rank as c_int, dst.as_mut_ptr() as *mut c_void) })
    }
}
impl Drop for BoxCiphertext {
    fn drop(&mut self) {
        unsafe { sys::spf_b200_box_ciphertext_free(self.raw.as_ptr()) }
    }
}

/// A validated, levelised `FheCircuit` over every rank of a [`BoxEvaluation`] (`spf_b200_box_graph_build`), or over the
/// ranks chosen with [`BoxGraph::build_on`].  io buffers are host memory or [`BoxCiphertext::as_io`].
pub struct BoxGraph {
    raw: NonNull<RawBoxGraph>,
    ev: BoxEvaluation,
}
unsafe impl Send for BoxGraph {}

impl BoxGraph {
    pub fn build(ev: &BoxEvaluation, nodes: &[spf_node]) -> Result<Self> {
        let mut raw = ptr::null_mut();
        let rc = unsafe { sys::spf_b200_box_graph_build(ev.raw(), nodes.as_ptr(), nodes.len(), &mut raw) };
        match NonNull::new(raw) {
            Some(p) if rc == 0 => Ok(Self { raw: p, ev: ev.clone() }),
            _ => Err(Error { code: rc, message: box_error(ev.raw()) }),
        }
    }
    /// The graph on the box ranks `ranks` only (`spf_b200_box_graph_build_on`): member `i` runs on box rank `ranks[i]`,
    /// and the graph is sharded over the members as over a box of `ranks.len()` ranks.  Handle outputs still reach the
    /// replica of every rank.  A graph that writes a handle another graph reads, on any rank, must be named in that
    /// reader's `after`.
    pub fn build_on(ev: &BoxEvaluation, nodes: &[spf_node], ranks: &[i32]) -> Result<Self> {
        let mut raw = ptr::null_mut();
        let n = c_int::try_from(ranks.len()).unwrap_or(c_int::MAX);  // the library refuses more ranks than the box has
        let rc = unsafe { sys::spf_b200_box_graph_build_on(ev.raw(), nodes.as_ptr(), nodes.len(), ranks.as_ptr(), n, &mut raw) };
        match NonNull::new(raw) {
            Some(p) if rc == 0 => Ok(Self { raw: p, ev: ev.clone() }),
            _ => Err(Error { code: rc, message: box_error(ev.raw()) }),
        }
    }
    /// The box ranks the graph runs on, in member order.
    pub fn ranks(&self) -> Vec<i32> {
        let n = unsafe { sys::spf_b200_box_graph_ranks(self.raw.as_ptr(), ptr::null_mut()) };
        let mut out = vec![0; n.max(0) as usize];
        unsafe { sys::spf_b200_box_graph_ranks(self.raw.as_ptr(), out.as_mut_ptr()) };
        out
    }
    /// `CircuitProcessor::run_graph_blocking` over the box.
    pub fn run_blocking(&mut self) -> Result<()> {
        let rc = unsafe { sys::spf_b200_box_graph_run(self.raw.as_ptr()) };
        if rc == 0 { Ok(()) } else { Err(Error { code: rc, message: box_error(self.ev.raw()) }) }
    }
    /// `CircuitProcessor::spawn_graph` over the box: the handler fires once, after every rank has retired.
    pub fn spawn<F: FnOnce(Option<Error>) + Send + 'static>(&mut self, after: &[&BoxGraph], on_completion: F) -> Result<()> {
        let deps: Vec<*mut RawBoxGraph> = after.iter().map(|g| g.raw.as_ptr()).collect();
        let handler: Box<Handler> = Box::new(Box::new(on_completion));
        let user = Box::into_raw(handler) as *mut c_void;
        let rc = unsafe { sys::spf_b200_box_graph_spawn(self.raw.as_ptr(), deps.as_ptr(), deps.len(), Some(completion_trampoline), user) };
        if rc == 0 {
            Ok(())
        } else {
            drop(unsafe { Box::from_raw(user as *mut Handler) });
            Err(Error { code: rc, message: box_error(self.ev.raw()) })
        }
    }
    /// Blocks until the last run (callback included) is over and returns its status.
    pub fn wait(&self) -> Result<()> {
        let rc = unsafe { sys::spf_b200_box_graph_wait(self.raw.as_ptr()) };
        if rc == 0 {
            Ok(())
        } else {
            let m = unsafe { CStr::from_ptr(sys::spf_b200_box_graph_status_message(self.raw.as_ptr())) }.to_string_lossy().into_owned();
            Err(Error { code: rc, message: m })
        }
    }
    /// Re-point an `Input*` / `Output*` node at another host buffer or [`BoxCiphertext::as_io`].
    ///
    /// # Safety
    /// `io` must stay valid, and large enough for the node's ciphertext, until the graph has run.
    pub unsafe fn set_io(&mut self, node: usize, io: *mut c_void) -> Result<()> {
        let rc = sys::spf_b200_box_graph_set_io(self.raw.as_ptr(), node, io);
        if rc == 0 { Ok(()) } else { Err(Error { code: rc, message: box_error(self.ev.raw()) }) }
    }
}
impl Drop for BoxGraph {
    fn drop(&mut self) {
        unsafe { sys::spf_b200_box_graph_destroy(self.raw.as_ptr()) }
    }
}

/// Glue for the reference workspace (feature `parasol`): what `parasol_runtime` needs so that
/// `CircuitProcessor::exec_op` runs on the GPU.  Written against spf v0.9.0.
#[cfg(feature = "parasol")]
pub mod parasol {
    use super::*;
    use parasol_runtime::{
        L0LweCiphertext, L1GgswCiphertext, L1GlevCiphertext, L1GlweCiphertext, L1LweCiphertext, Params,
    };

    /// Field-for-field copy of `Params` (`parasol_runtime/src/params.rs:59-91`).
    pub fn params_from(p: &Params) -> spf_params {
        let r = |x: &sunscreen_tfhe::RadixDecomposition| spf_radix { radix_log: x.radix_log.0 as u32, count: x.count.0 as u32 };
        spf_params {
            lwe_n: p.l0_params.dim.0 as u32,
            lwe_std: p.l0_params.std.0,
            glwe_k: p.l1_params.dim.size.0 as u32,
            glwe_n: p.l1_params.dim.polynomial_degree.0 as u32,
            glwe_std: p.l1_params.std.0,
            cbs: r(&p.cbs_radix),
            pbs: r(&p.pbs_radix),
            ks: r(&p.ks_radix),
            pfks: r(&p.pfks_radix),
            ss: r(&p.ss_radix),
            tr: r(&p.tr_radix),
        }
    }
    // Torus<u64> is repr(transparent) over u64 (math/torus.rs:216-220), Complex<f64> is repr(C) (re, im): the casts
    // below are the complete marshalling of every entity (dst.rs:31-33: one contiguous 64-byte aligned array).
    fn torus(x: &[sunscreen_tfhe::Torus<u64>]) -> &[u64] {
        unsafe { std::slice::from_raw_parts(x.as_ptr() as *const u64, x.len()) }
    }
    fn torus_mut(x: &mut [sunscreen_tfhe::Torus<u64>]) -> &mut [u64] {
        unsafe { std::slice::from_raw_parts_mut(x.as_mut_ptr() as *mut u64, x.len()) }
    }
    fn cplx(x: &[num::Complex<f64>]) -> &[f64] {
        unsafe { std::slice::from_raw_parts(x.as_ptr() as *const f64, 2 * x.len()) }
    }
    fn cplx_mut(x: &mut [num::Complex<f64>]) -> &mut [f64] {
        unsafe { std::slice::from_raw_parts_mut(x.as_mut_ptr() as *mut f64, 2 * x.len()) }
    }

    /// The bodies of `Evaluation`'s methods in the GPU build: same signatures as `evaluation.rs`, batch = 1.  With only
    /// these the runtime works unmodified (one op per rayon task); the batching executor is [`Graph`].
    impl Evaluation {
        pub fn circuit_bootstrap_ct(&self, output: &mut L1GgswCiphertext, input: &L0LweCiphertext) {
            self.circuit_bootstrap(cplx_mut(output.0.as_mut_slice()), torus(input.0.as_slice())).expect("circuit_bootstrap")
        }
        pub fn cmux_ct(&self, output: &mut L1GlweCiphertext, sel: &L1GgswCiphertext, a: &L1GlweCiphertext, b: &L1GlweCiphertext) {
            self.cmux(torus_mut(output.0.as_mut_slice()), cplx(sel.0.as_slice()), torus(a.0.as_slice()), torus(b.0.as_slice())).expect("cmux")
        }
        pub fn glev_cmux_ct(&self, output: &mut L1GlevCiphertext, sel: &L1GgswCiphertext, a: &L1GlevCiphertext, b: &L1GlevCiphertext) {
            self.glev_cmux(torus_mut(output.0.as_mut_slice()), cplx(sel.0.as_slice()), torus(a.0.as_slice()), torus(b.0.as_slice())).expect("glev_cmux")
        }
        pub fn multiply_glwe_ggsw_ct(&self, output: &mut L1GlweCiphertext, glwe: &L1GlweCiphertext, ggsw: &L1GgswCiphertext) {
            self.multiply_glwe_ggsw(torus_mut(output.0.as_mut_slice()), torus(glwe.0.as_slice()), cplx(ggsw.0.as_slice())).expect("multiply_glwe_ggsw")
        }
        pub fn keyswitch_lwe_l1_lwe_l0_ct(&self, output: &mut L0LweCiphertext, input: &L1LweCiphertext) {
            self.keyswitch_lwe_l1_lwe_l0(torus_mut(output.0.as_mut_slice()), torus(input.0.as_slice())).expect("keyswitch")
        }
        pub fn sample_extract_l1_ct(&self, output: &mut L1LweCiphertext, input: &L1GlweCiphertext, idx: usize) {
            self.sample_extract_l1(torus_mut(output.0.as_mut_slice()), torus(input.0.as_slice()), idx).expect("sample_extract")
        }
        pub fn scheme_switch_ct(&self, output: &mut L1GgswCiphertext, input: &L1GlevCiphertext) {
            self.scheme_switch(cplx_mut(output.0.as_mut_slice()), torus(input.0.as_slice())).expect("scheme_switch")
        }
        pub fn not_ct(&self, output: &mut L1GlweCiphertext, input: &L1GlweCiphertext) {
            self.not(torus_mut(output.0.as_mut_slice()), torus(input.0.as_slice())).expect("not")
        }
        pub fn xor_ct(&self, output: &mut L1GlweCiphertext, a: &L1GlweCiphertext, b: &L1GlweCiphertext) {
            self.xor(torus_mut(output.0.as_mut_slice()), torus(a.0.as_slice()), torus(b.0.as_slice())).expect("xor")
        }
        pub fn mul_xn_ct(&self, output: &mut L1GlweCiphertext, input: &L1GlweCiphertext, n: usize) {
            self.mul_xn(torus_mut(output.0.as_mut_slice()), torus(input.0.as_slice()), n).expect("mul_xn")
        }
    }

    /// `FheOp` -> `spf_op` (`fhe_circuit.rs:34-127`, same order as the C enum) and `FheCircuit` -> `[spf_node]`:
    /// one node per petgraph node, `in[]` from the incoming `FheEdge`s (`fhe_circuit.rs:174-198`), `io` = the
    /// ciphertext buffer behind an Input / Output op (`Arc<AtomicRefCell<_>>`: borrow for the duration of the run).
    pub fn lower(circuit: &parasol_runtime::FheCircuit) -> Vec<spf_node> {
        use parasol_runtime::{FheEdge, FheOp};
        use petgraph::{visit::EdgeRef, Direction};
        let g = &circuit.graph;
        let index: std::collections::HashMap<_, _> = g.node_indices().enumerate().map(|(i, n)| (n, i as i32)).collect();
        g.node_indices()
            .map(|n| {
                let (op, arg, io): (u32, u32, *mut c_void) = match g.node_weight(n).unwrap() {
                    FheOp::InputLwe0(x) => (sys::SPF_OP_INPUT_LWE0, 0, x.borrow().0.as_slice().as_ptr() as *mut c_void),
                    FheOp::InputLwe1(x) => (sys::SPF_OP_INPUT_LWE1, 0, x.borrow().0.as_slice().as_ptr() as *mut c_void),
                    FheOp::InputGlwe1(x) => (sys::SPF_OP_INPUT_GLWE1, 0, x.borrow().0.as_slice().as_ptr() as *mut c_void),
                    FheOp::InputGgsw1(x) => (sys::SPF_OP_INPUT_GGSW1, 0, x.borrow().0.as_slice().as_ptr() as *mut c_void),
                    FheOp::InputGlev1(x) => (sys::SPF_OP_INPUT_GLEV1, 0, x.borrow().0.as_slice().as_ptr() as *mut c_void),
                    FheOp::OutputLwe0(x) => (sys::SPF_OP_OUTPUT_LWE0, 0, x.borrow_mut().0.as_mut_slice().as_mut_ptr() as *mut c_void),
                    FheOp::OutputLwe1(x) => (sys::SPF_OP_OUTPUT_LWE1, 0, x.borrow_mut().0.as_mut_slice().as_mut_ptr() as *mut c_void),
                    FheOp::OutputGlwe1(x) => (sys::SPF_OP_OUTPUT_GLWE1, 0, x.borrow_mut().0.as_mut_slice().as_mut_ptr() as *mut c_void),
                    FheOp::OutputGgsw1(x) => (sys::SPF_OP_OUTPUT_GGSW1, 0, x.borrow_mut().0.as_mut_slice().as_mut_ptr() as *mut c_void),
                    FheOp::OutputGlev1(x) => (sys::SPF_OP_OUTPUT_GLEV1, 0, x.borrow_mut().0.as_mut_slice().as_mut_ptr() as *mut c_void),
                    FheOp::SampleExtract(i) => (sys::SPF_OP_SAMPLE_EXTRACT, *i as u32, ptr::null_mut()),
                    FheOp::KeyswitchL1toL0 => (sys::SPF_OP_KEYSWITCH_L1_TO_L0, 0, ptr::null_mut()),
                    FheOp::Not => (sys::SPF_OP_NOT, 0, ptr::null_mut()),
                    FheOp::GlweAdd => (sys::SPF_OP_GLWE_ADD, 0, ptr::null_mut()),
                    FheOp::CMux => (sys::SPF_OP_CMUX, 0, ptr::null_mut()),
                    FheOp::GlevCMux => (sys::SPF_OP_GLEV_CMUX, 0, ptr::null_mut()),
                    FheOp::MultiplyGgswGlwe => (sys::SPF_OP_MULTIPLY_GGSW_GLWE, 0, ptr::null_mut()),
                    FheOp::CircuitBootstrap => (sys::SPF_OP_CIRCUIT_BOOTSTRAP, 0, ptr::null_mut()),
                    FheOp::SchemeSwitch => (sys::SPF_OP_SCHEME_SWITCH, 0, ptr::null_mut()),
                    FheOp::ZeroLwe0 => (sys::SPF_OP_ZERO_LWE0, 0, ptr::null_mut()),
                    FheOp::OneLwe0 => (sys::SPF_OP_ONE_LWE0, 0, ptr::null_mut()),
                    FheOp::ZeroGlwe1 => (sys::SPF_OP_ZERO_GLWE1, 0, ptr::null_mut()),
                    FheOp::OneGlwe1 => (sys::SPF_OP_ONE_GLWE1, 0, ptr::null_mut()),
                    FheOp::ZeroGgsw1 => (sys::SPF_OP_ZERO_GGSW1, 0, ptr::null_mut()),
                    FheOp::OneGgsw1 => (sys::SPF_OP_ONE_GGSW1, 0, ptr::null_mut()),
                    FheOp::ZeroGlev1 => (sys::SPF_OP_ZERO_GLEV1, 0, ptr::null_mut()),
                    FheOp::OneGlev1 => (sys::SPF_OP_ONE_GLEV1, 0, ptr::null_mut()),
                    FheOp::Retire => (sys::SPF_OP_RETIRE, 0, ptr::null_mut()),
                    FheOp::Nop => (sys::SPF_OP_NOP, 0, ptr::null_mut()),
                    FheOp::MulXN(k) => (sys::SPF_OP_MUL_XN, *k as u32, ptr::null_mut()),
                };
                let mut inp = [-1i32; 3];
                for e in g.edges_directed(n, Direction::Incoming) {
                    let slot = match e.weight() {
                        FheEdge::Unary | FheEdge::Left | FheEdge::Sel | FheEdge::Glwe => 0,
                        FheEdge::Right | FheEdge::Low | FheEdge::Ggsw => 1,
                        FheEdge::High => 2,
                    };
                    inp[slot] = index[&e.source()];
                }
                spf_node { op, arg, r#in: inp, io }
            })
            .collect()
    }

    /// The evaluator a `CircuitProcessor` dispatches to: one GPU, or every GPU of a box.
    pub enum Evaluator<'a> {
        Single(&'a Evaluation),
        Box(&'a BoxEvaluation),
    }
    /// The graph [`spawn_graph`] returns, on the evaluator it was built for.
    pub enum SpawnedGraph {
        Single(Graph),
        Box(BoxGraph),
    }
    impl SpawnedGraph {
        pub fn wait(&self) -> Result<()> {
            match self {
                SpawnedGraph::Single(g) => g.wait(),
                SpawnedGraph::Box(g) => g.wait(),
            }
        }
    }

    /// Task outputs kept in HBM on a box: the address of a task's ciphertext buffer (the `io` that [`lower`] gives its
    /// `Input*` / `Output*` nodes) -> the [`BoxCiphertext`] that stands for it.  Instruction k's output task and
    /// instruction k + 1's input task then name the same handle, and the hand-off never leaves the devices.
    pub type BoxResident<'a> = std::collections::HashMap<*mut c_void, &'a BoxCiphertext>;

    /// [`lower`], with the io buffers found in `resident` replaced by their box ciphertext handles.
    pub fn lower_resident(circuit: &parasol_runtime::FheCircuit, resident: &BoxResident<'_>) -> Vec<spf_node> {
        let mut nodes = lower(circuit);
        for n in nodes.iter_mut() {
            if let Some(h) = resident.get(&n.io) {
                n.io = h.as_io();
            }
        }
        nodes
    }

    /// `CircuitProcessor::spawn_graph` on the GPU: lower, build, spawn.  Validation errors reach the handler, as in
    /// the reference where they surface through `CompletionHandler::error`.
    pub fn spawn_graph<F>(ev: Evaluator<'_>, circuit: &parasol_runtime::FheCircuit, on_completion: F) -> Option<SpawnedGraph>
    where
        F: FnOnce(Option<Error>) + Send + 'static,
    {
        let nodes = lower(circuit);
        let built = match ev {
            Evaluator::Single(e) => Graph::build(e, &nodes).map(SpawnedGraph::Single),
            Evaluator::Box(b) => BoxGraph::build(b, &nodes).map(SpawnedGraph::Box),
        };
        match built {
            Err(e) => {
                on_completion(Some(e));
                None
            }
            Ok(mut g) => {
                let spawned = match &mut g {
                    SpawnedGraph::Single(s) => s.spawn(&[], on_completion),
                    SpawnedGraph::Box(b) => b.spawn(&[], on_completion),
                };
                if let Err(e) = spawned {
                    panic!("spf_b200: could not spawn a validated graph: {e}");
                }
                Some(g)
            }
        }
    }

    /// [`spawn_graph`] on a box with task outputs in HBM: the io buffers in `resident` are mapped to their
    /// [`BoxCiphertext`]s, and the run is ordered on the devices behind the last runs of `after` (the graphs of the
    /// instructions whose outputs it reads, and of those that read what it writes).  `ranks`: the box ranks the graph
    /// runs on ([`BoxGraph::build_on`]; `None` = every rank), so that independent instructions run on different GPUs.
    pub fn spawn_box_graph<F>(b: &BoxEvaluation, circuit: &parasol_runtime::FheCircuit, resident: &BoxResident<'_>, after: &[&BoxGraph],
                              ranks: Option<&[i32]>, on_completion: F) -> Option<BoxGraph>
    where
        F: FnOnce(Option<Error>) + Send + 'static,
    {
        let nodes = lower_resident(circuit, resident);
        let built = match ranks {
            None => BoxGraph::build(b, &nodes),
            Some(r) => BoxGraph::build_on(b, &nodes, r),
        };
        match built {
            Err(e) => {
                on_completion(Some(e));
                None
            }
            Ok(mut g) => {
                if let Err(e) = g.spawn(after, on_completion) {
                    panic!("spf_b200: could not spawn a validated graph: {e}");
                }
                Some(g)
            }
        }
    }
}
