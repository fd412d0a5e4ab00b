"""Per-op device throughput for the ops of parasol_runtime/benches/fhe_ops.rs:40-85 (cmux, keyswitch,
sample extract, circuit bootstrap, PBS) with inputs resident in HBM, next to the CPU port's
single-thread time per op.  HBM-bound ops are reported against MEASURED_PEAKS.json's copy bandwidth
with the algorithmic bytes of SURVEY.md 8(d).  usage: python tools/op_bench.py [batch]"""
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle as O  # keygen / CPU timing only
import spf_b200
from bench import encrypt_lwe0_numpy

B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
dev = torch.device("cuda", 0)
keys = O.Keys()
client = O.Client(keys)
ev = spf_b200.Evaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft)
stream = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(stream)
s = stream.cuda_stream
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
try:
    hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
except Exception:
    hbm = 6650.0
rng = np.random.default_rng(3)


def timed(fn, reps=3):
    fn()
    ms = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return min(ms)


def rand_u64(*shape):
    return torch.from_numpy(rng.integers(0, 1 << 63, shape, dtype=np.int64)).to(dev)


rows = []
# ---- CMUX: one selector per op (the runtime's CMux nodes), 360 448 algorithmic bytes per op ----
one = client.encrypt_ggsw_l1(1)
sel = torch.from_numpy(np.ascontiguousarray(one).view(np.float64)).to(dev)
d_sel = torch.empty(B * ev.len_ggsw * 2, dtype=torch.float64, device=dev)
ev.dev_fft_rescale(d_sel.data_ptr(), sel.data_ptr(), ev.len_ggsw, to_device=True, stream=s)  # reference -> device scale
d_sel.view(B, -1)[1:] = d_sel.view(B, -1)[0]
a, b, out = rand_u64(B, ev.len_glwe), rand_u64(B, ev.len_glwe), rand_u64(B, ev.len_glwe)
ms = timed(lambda: ev.dev_cmux(out.data_ptr(), d_sel.data_ptr(), ev.len_ggsw, a.data_ptr(), b.data_ptr(), B, stream=s))
bytes_op = ev.len_ggsw * 16 + 3 * ev.len_glwe * 8
rows.append({"op": "cmux", "batch": B, "ms": ms, "ops_per_s": B / ms * 1e3, "algorithmic_gb_s": B * bytes_op / ms / 1e6,
             "hbm_frac": B * bytes_op / ms / 1e6 / hbm})
del d_sel, a, b, out
# ---- keyswitch L1 -> L0: KSK read once per 16 ciphertexts ----
l1 = rand_u64(B, ev.len_lwe_l1)
l0 = torch.empty(B * ev.len_lwe_l0, dtype=torch.int64, device=dev)
ms = timed(lambda: ev.dev_keyswitch_lwe_l1_lwe_l0(l0.data_ptr(), l1.data_ptr(), B, stream=s))
ksk_bytes = keys.ksk.nbytes
alg = ksk_bytes + B * (ev.len_lwe_l1 + ev.len_lwe_l0) * 8
rows.append({"op": "keyswitch_l1_l0", "batch": B, "ms": ms, "ops_per_s": B / ms * 1e3, "algorithmic_gb_s": alg / ms / 1e6,
             "hbm_frac": alg / ms / 1e6 / hbm, "u64_mad_per_s": B * 2048 * 6 * 638 / ms * 1e3,
             "int8_tmac_per_s": B * 2048 * 6 * 640 * 8 / ms / 1e9, "tcgen05_i8_nominal_tmac_per_s": 2250.0,
             "tensor_frac": B * 2048 * 6 * 640 * 8 / ms / 1e9 / 2250.0,
             "note": "8 u8 x u8 -> s32 byte-plane GEMMs on tcgen05.mma kind::i8 (TMEM accumulators); peak = nominal dense "
                     "int8 rate of the part (4.5 POPS); the kernel is bound by the L2 -> SM stream of the key planes"})
# ---- sample extract ----
g = rand_u64(B, ev.len_glwe)
l1o = torch.empty(B * ev.len_lwe_l1, dtype=torch.int64, device=dev)
ms = timed(lambda: ev.dev_sample_extract_l1(l1o.data_ptr(), g.data_ptr(), 0, 0, B, stream=s))
alg = B * (ev.len_glwe // 2 + ev.len_lwe_l1) * 8  # reads the a polynomial + one b coefficient
rows.append({"op": "sample_extract", "batch": B, "ms": ms, "ops_per_s": B / ms * 1e3, "algorithmic_gb_s": alg / ms / 1e6,
             "hbm_frac": alg / ms / 1e6 / hbm})
del g, l1o, l1, l0
# ---- RLWE public-key encryption (exact negacyclic u64 products; 4 194 304 u64 multiply-adds per polynomial, 2 per ciphertext) ----
n = keys.params.glwe_n
pk_d = rand_u64(2 * n)
m_d, e0_d, e1_d = rand_u64(B, n), rand_u64(B, n), rand_u64(B, n)
u_d = torch.from_numpy(rng.integers(0, 2, (B, n), dtype=np.int64)).to(dev)
ct_d = torch.empty(B * 2 * n, dtype=torch.int64, device=dev)
ms = timed(lambda: ev.dev_rlwe_encrypt_public(ct_d.data_ptr(), pk_d.data_ptr(), m_d.data_ptr(), u_d.data_ptr(), e0_d.data_ptr(),
                                              e1_d.data_ptr(), B, stream=s))
rows.append({"op": "rlwe_encrypt_public", "batch": B, "ms": ms, "ops_per_s": B / ms * 1e3, "u64_mad_per_s": B * 2 * n * n / ms * 1e3})
del pk_d, m_d, e0_d, e1_d, u_d, ct_d
# ---- CBS and PBS ----
bits = rng.integers(0, 2, B)
cts = torch.from_numpy(encrypt_lwe0_numpy(keys.lwe0_sk, bits, keys.params.lwe_std, 5).view(np.int64)).to(dev)
ggsw = torch.empty(B * ev.len_ggsw * 2, dtype=torch.float64, device=dev)
ms = timed(lambda: ev.dev_circuit_bootstrap(ggsw.data_ptr(), cts.data_ptr(), B, reference_scale=False, stream=s), reps=2)
rows.append({"op": "circuit_bootstrap", "batch": B, "ms": ms, "ops_per_s": B / ms * 1e3, "fp64_tflops": 293.3e6 * B / ms / 1e9})
# ---- PBS alone (device resident) ----
from bench import cbs_lut
lut = torch.from_numpy(cbs_lut().view(np.int64)).to(dev)
glwe_o = torch.empty(B * ev.len_glwe, dtype=torch.int64, device=dev)
ms = timed(lambda: ev.dev_programmable_bootstrap(glwe_o.data_ptr(), cts.data_ptr(), lut.data_ptr(), 0, 2, B, stream=s), reps=2)
rows.append({"op": "programmable_bootstrap", "batch": B, "ms": ms, "ops_per_s": B / ms * 1e3, "fp64_tflops": 263.5e6 * B / ms / 1e9})
del ggsw, glwe_o
# ---- GLEV cmux and scheme switch: host-pointer API only (copies inside the timed call) ----
nb = min(B, 512)
torch.cuda.synchronize()
glev_a = rng.integers(0, 1 << 63, (nb, ev.len_glev), dtype=np.uint64)
glev_b = rng.integers(0, 1 << 63, (nb, ev.len_glev), dtype=np.uint64)
sel_h = np.broadcast_to(np.ascontiguousarray(one), (nb, ev.len_ggsw)).copy()
ev.glev_cmux(sel_h[:4], glev_a[:4], glev_b[:4])
t0 = time.perf_counter(); ev.glev_cmux(sel_h, glev_a, glev_b); dt = time.perf_counter() - t0
rows.append({"op": "glev_cmux (host pointers, copies inside)", "batch": nb, "ms": 1e3 * dt, "ops_per_s": nb / dt})
glev_in = np.stack([client.encrypt_glev_l1([1])] * 8 + [client.encrypt_glev_l1([0])] * 8)
glev_in = np.ascontiguousarray(np.tile(glev_in, (nb // 16, 1)))
ev.scheme_switch(glev_in[:4])
t0 = time.perf_counter(); ss = ev.scheme_switch(glev_in); dt = time.perf_counter() - t0
rows.append({"op": "scheme_switch (host pointers, copies inside)", "batch": len(glev_in), "ms": 1e3 * dt, "ops_per_s": len(glev_in) / dt,
             "decrypt_ok": bool(client.decrypt_ggsw_l1(ss[0]) == 1 and client.decrypt_ggsw_l1(ss[8]) == 0)})
for r in rows:
    print(json.dumps(r), flush=True)
# ---- CPU port, single thread, one op each (the reference's bench measures exactly these) ----
cpu = {}
g0, g1 = client.encrypt_glwe_l1([0]), client.encrypt_glwe_l1([1])
t0 = time.perf_counter(); O.cmux(keys, g0, g1, one); cpu["cmux_ms"] = 1e3 * (time.perf_counter() - t0)
l1c = O.sample_extract(keys, g1, 0)
t0 = time.perf_counter(); O.sample_extract(keys, g1, 0); cpu["sample_extract_ms"] = 1e3 * (time.perf_counter() - t0)
t0 = time.perf_counter(); l0c = O.keyswitch_lwe(keys, l1c); cpu["keyswitch_ms"] = 1e3 * (time.perf_counter() - t0)
t0 = time.perf_counter(); O.circuit_bootstrap(keys, l0c); cpu["circuit_bootstrap_ms"] = 1e3 * (time.perf_counter() - t0)
t0 = time.perf_counter(); O.cbs_pbs_stage(keys, l0c); cpu["programmable_bootstrap_ms"] = 1e3 * (time.perf_counter() - t0)
ge = client.encrypt_glev_l1([1])
t0 = time.perf_counter(); O.glev_cmux(keys, ge, ge, one); cpu["glev_cmux_ms"] = 1e3 * (time.perf_counter() - t0)
t0 = time.perf_counter(); O.scheme_switch(keys, ge); cpu["scheme_switch_ms"] = 1e3 * (time.perf_counter() - t0)
pkc = client.generate_public_key()
rr = client.rlwe_randomness()
t0 = time.perf_counter(); O.rlwe_encrypt_public(keys.params, g0[:keys.params.glwe_n], pkc, *rr); cpu["rlwe_encrypt_public_ms"] = 1e3 * (time.perf_counter() - t0)
print(json.dumps({"cpu_port_single_thread": cpu}), flush=True)
