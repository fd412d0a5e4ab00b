#!/usr/bin/env python
"""bench.py -- circuit bootstraps / second on B200 (BASELINE.json metric, config 3).

A "step" is one pass of the hot path over one batch of synthetic input: `--batch` (default 4096)
independent L0 LWE ciphertexts -> 4096 L1 GGSW ciphertexts (circuit_bootstrap_via_trace_and_
scheme_switch at DEFAULT_128).  One process per GPU; with N > 1 (torchrun) every rank holds a
replica of the compute key (broadcast once from rank 0 over NCCL/NVLink) and bootstraps its own
batch (weak scaling, no data-path collective: SURVEY.md section 8(e)).

  value     CBS/s, inputs and outputs resident in HBM, CUDA-event time, max over ranks
  e2e       same metric through the reference-facing host-pointer call
            (spf_b200_circuit_bootstrap): pinned host buffers, H2D + D2H inside the timed region
  roofline  the dominant kernel (pbs_kernel, blind rotation) against the FP64 CUDA-core peak
            measured in this run by a DFMA probe (MEASURED_PEAKS.json has no FP64 figure), plus
            its algorithmic HBM bytes against the measured HBM peak
  cpu_baseline  the oracle (C restatement of the reference CPU path; the Rust reference cannot
            be built in this image) on the box's host cores, bounded sample

`--impl reference` times that CPU restatement alone (the reference arm of the contract).
`--dump-outputs DIR` writes a fixed sample of the last timed step's outputs to DIR (see dump_outputs).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "circuit_bootstraps_per_sec"
UNIT = "CBS/s"
# SURVEY.md section 8(d): algorithmic work per unit at DEFAULT_128
FLOP_PER_PBS = 263.5e6
FLOP_PER_CBS = 293.3e6
BSK_BYTES = 83492864
PBS_IO_BYTES = 5104 + 32768  # LWE in + GLWE out per ciphertext


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4096, help="CBS per step per GPU (BASELINE config 3: 4096)")
    ap.add_argument("--impl", default="spf_b200", choices=["spf_b200", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="CBS in the CPU baseline sample (0 = about 10 s of work on all host threads)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-add", action="store_true", help="skip the Parasol program latency measurements (8/32-bit add, mul32 + compare)")
    ap.add_argument("--check", type=int, default=512, help="outputs decrypted with the oracle after the run, spread over every PBS wave (checker only)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the 3-point batch-size sweep (BASELINE config 5)")
    ap.add_argument("--no-sharded-graph", action="store_true", help="N > 1: skip the sharded mul32+compare graph (BASELINE config 4)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a fixed sample of the last step's "
                    "GGSW outputs to DIR/cbs_ggsw_fft.npy (float64, at most 32 MiB)")
    return ap.parse_args()


# ---------------------------------------------------------------------------------------------
# synthetic workload: the harness' own seeds (the reference RNG is unseedable thread_rng())
# ---------------------------------------------------------------------------------------------
def encrypt_lwe0_numpy(sk: np.ndarray, bits: np.ndarray, std: float, seed: int) -> np.ndarray:
    """b = <a,s> + m + e (ops/encryption/lwe_encryption.rs:36-61), vectorised; client-side input
    generation only."""
    rng = np.random.default_rng(seed)
    n = sk.shape[0]
    a = rng.integers(0, 1 << 64, (len(bits), n), dtype=np.uint64)
    e = np.round(rng.normal(0.0, std, len(bits)) * 2.0 ** 64).astype(np.int64).astype(np.uint64)
    b = (a * sk[None, :]).sum(axis=1, dtype=np.uint64) + (bits.astype(np.uint64) << np.uint64(63)) + e
    return np.ascontiguousarray(np.concatenate([a, b[:, None]], axis=1))


def cbs_lut(n: int = 2048) -> np.ndarray:
    """fill_multifunctional_cbs_decomposition_lut (circuit_bootstrapping.rs:430-482) as a trivial GLWE."""
    lut = np.zeros(2 * n, dtype=np.uint64)
    i = np.arange(n)
    pb = 4 * ((i % 4) + 1) + 1
    lut[n:] = (np.uint64(0) - (np.uint64(1) << (64 - pb).astype(np.uint64)))
    return lut


def ncu_traffic(batch: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of one pbs_kernel launch at this batch size, from
    the committed `ncu --set full` capture (profiles/pbs_kernel_dram_traffic.json), or None."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "pbs_kernel_dram_traffic.json")))
        e = t["by_batch"].get(str(batch))
        return None if e is None else {"bytes_per_launch": e["dram_read_bytes"] + e["dram_write_bytes"], **e, "source": t["source"]}
    except Exception:
        return None


def ncu_pipes():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "pbs_kernel_dram_traffic.json"))).get("pipes")
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for nm, v in zip(names, r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------
# CPU baseline (the oracle port, all host threads) -- also the `--impl reference` arm
# ---------------------------------------------------------------------------------------------
def cpu_cbs_rate(keys, cts: np.ndarray, nthreads: int) -> tuple[float, float]:
    """The timed CPU leg runs the FAST flavour of the oracle (oracle/libspf_oracle_fast.so: the same C restatement built
    with -ffp-contract=fast and AVX2/FMA intrinsics for the FFT, the f64 -> torus conversion and the complex MAD), the
    honest stand-in for the reference's +avx2,+fma build; the strict flavour stays the parity checker."""
    import oracle as O

    t0 = time.perf_counter()
    O.circuit_bootstrap_batch(keys, cts, nthreads, fast=True)
    dt = time.perf_counter() - t0
    return len(cts) / dt, dt


CPU_KIND_NOTE = ("oracle/spf_oracle.c built -O3 -march=x86-64-v3 -ffp-contract=fast -DORC_FAST (AVX2/FMA radix-4 Stockham FFT, "
                 "vectorised conversions and complex MADs): a C restatement of the reference CPU path with the reference's "
                 "parallelisation model (one single-threaded op per task over all host threads); the Rust reference itself "
                 "cannot be built in this image")


def cpu_micro(keys, cts: np.ndarray) -> dict:
    """Single-thread figures printed beside the CPU baseline so its class is visible: us per 1024-point (N = 2048)
    forward transform and ms per circuit bootstrap on one core, fast and strict flavours."""
    import oracle as O

    out = {}
    for name, fast in (("fast", True), ("strict", False)):
        out[f"fft1024_us_{name}"] = 1e6 * O.lib(fast).orc_bench_fft_forward(2048, 20000)
    O.circuit_bootstrap_batch(keys, cts[:1], 1, fast=True)
    t0 = time.perf_counter()
    O.circuit_bootstrap_batch(keys, cts[:2], 1, fast=True)
    out["single_thread_ms_per_cbs_fast"] = 1e3 * (time.perf_counter() - t0) / 2
    t0 = time.perf_counter()
    O.circuit_bootstrap_batch(keys, cts[:1], 1, fast=False)
    out["single_thread_ms_per_cbs_strict"] = 1e3 * (time.perf_counter() - t0)
    return out


def cpu_sample_size(rate: float, nt: int, batch: int, seconds: float = 10.0) -> int:
    """CBS in one bounded CPU sample: about `seconds` of work on all host threads, a multiple of the
    thread count, never more than the GPU batch."""
    n = int(rate * seconds) // nt * nt
    return int(max(2 * nt, min(n, batch)))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle as O

    keys = O.Keys()
    nt = O.hw_threads()
    probe_bits = np.random.default_rng(O.INPUT_SEED).integers(0, 2, 2 * nt)
    probe = encrypt_lwe0_numpy(keys.lwe0_sk, probe_bits, keys.params.lwe_std, O.INPUT_SEED)
    rate0, _ = cpu_cbs_rate(keys, probe, nt)  # warm-up pass, also sizes the sample
    sample = args.cpu_sample or cpu_sample_size(rate0, nt, args.batch)
    bits = np.random.default_rng(O.INPUT_SEED).integers(0, 2, sample)
    cts = encrypt_lwe0_numpy(keys.lwe0_sk, bits, keys.params.lwe_std, O.INPUT_SEED)
    total_t = 0.0
    for _ in range(args.steps):
        _, dt = cpu_cbs_rate(keys, cts, nt)
        total_t += dt
    value = sample * args.steps / total_t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total_t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"cbs_batch{args.batch}_default128 (bounded sample of {sample} CBS per step)",
                   "params": "DEFAULT_128", "batch_per_gpu": args.batch},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": nt, "kind": "port",
                         "sample": f"{sample} CBS per step x {args.steps} steps; " + CPU_KIND_NOTE, **cpu_micro(keys, cts)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def cpu_add_latency(keys, a_bits, b_bits, nthreads):
    """The same add on the CPU port with the reference's execution model: every ready op is one
    single-threaded task, independent tasks of a dependency level spread over the host threads."""
    import ctypes as C

    import oracle as O

    l = O.lib(fast=True)
    p = keys.params
    w = len(a_bits)
    t0 = time.perf_counter()
    glwes = np.stack(a_bits + b_bits)
    l1 = np.stack([O.sample_extract(keys, g, 0) for g in glwes])
    l0 = np.zeros((2 * w, keys.lwe0_len), dtype=np.uint64)
    l.orc_keyswitch_lwe_batch(l0, l1, 2 * w, keys.ksk, C.byref(p), nthreads)
    ggsw = O.circuit_bootstrap_batch(keys, l0, nthreads, fast=True)
    sa, sb = ggsw[:w], ggsw[w:]
    zero = np.zeros(keys.glwe_len, dtype=np.uint64)
    one = zero.copy()
    one[p.glwe_k * p.glwe_n] = np.uint64(1 << 63)
    carry, ncarry = zero, one
    outs = []

    def cmux_level(sels, lows, highs):
        out = np.zeros((len(sels), keys.glwe_len), dtype=np.uint64)
        l.orc_cmux_batch(out, np.ascontiguousarray(np.stack(lows)), np.ascontiguousarray(np.stack(highs)),
                         np.ascontiguousarray(np.stack(sels)), len(sels), C.byref(p), min(nthreads, len(sels)))
        return out

    for i in range(w):
        r = cmux_level([sb[i]] * 4, [carry, ncarry, zero, carry], [ncarry, carry, carry, one])
        r2 = cmux_level([sa[i]] * 2, [r[0], r[2]], [r[1], r[3]])
        outs.append(r2[0])
        carry = r2[1]
        ncarry = O.glwe_not(keys, carry)
    outs.append(carry)
    return time.perf_counter() - t0, outs


def cpu_run_graph(keys, circ, nthreads):
    """Any FheCircuit on the CPU port with the reference's execution model (circuit_processor/mod.rs:130-253):
    every ready op is one single-threaded task, the independent tasks of a dependency level are spread over
    the host threads.  Levels come from the host-only planner; the arithmetic is the oracle's.  Returns seconds."""
    import ctypes as C

    import oracle as O
    import spf_b200
    from spf_b200 import OPS

    l = O.lib(fast=True)
    p = keys.params
    level, _ = spf_b200.plan_graph(circ, 1)
    groups = {}
    for v in np.argsort(level, kind="stable").tolist():
        groups.setdefault((int(level[v]), circ.nodes[v][0]), []).append(v)
    zero = np.zeros(keys.glwe_len, dtype=np.uint64)
    one = zero.copy()
    one[p.glwe_k * p.glwe_n] = np.uint64(1 << 63)
    val = {}
    t0 = time.perf_counter()
    for (lv, opc), ids in sorted(groups.items()):
        op = OPS[opc]
        ins = [circ.nodes[v][2] for v in ids]
        if op == "InputGlwe1":
            for v in ids:
                val[v] = circ.nodes[v][3]
        elif op in ("ZeroGlwe1", "OneGlwe1"):
            for v in ids:
                val[v] = zero if op == "ZeroGlwe1" else one
        elif op == "SampleExtract":
            for v, i in zip(ids, ins):
                val[v] = O.sample_extract(keys, val[i[0]], circ.nodes[v][1])
        elif op == "KeyswitchL1toL0":
            out = np.zeros((len(ids), keys.lwe0_len), dtype=np.uint64)
            l.orc_keyswitch_lwe_batch(out, np.stack([val[i[0]] for i in ins]), len(ids), keys.ksk, C.byref(p), min(nthreads, len(ids)))
            for k, v in enumerate(ids):
                val[v] = out[k]
        elif op == "CircuitBootstrap":
            out = O.circuit_bootstrap_batch(keys, np.stack([val[i[0]] for i in ins]), min(nthreads, len(ids)), fast=True)
            for k, v in enumerate(ids):
                val[v] = out[k]
        elif op == "CMux":
            out = np.zeros((len(ids), keys.glwe_len), dtype=np.uint64)
            tab = lambda arrs: (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
            l.orc_cmux_batch_ptrs(tab([out[k] for k in range(len(ids))]), tab([val[i[1]] for i in ins]), tab([val[i[2]] for i in ins]),
                                  tab([val[i[0]] for i in ins]), len(ids), C.byref(p), min(nthreads, len(ids)))
            for k, v in enumerate(ids):
                val[v] = out[k]
        elif op == "Not":
            for v, i in zip(ids, ins):
                val[v] = O.glwe_not(keys, val[i[0]])
        elif op == "OutputGlwe1":
            for v, i in zip(ids, ins):
                circ.nodes[v][3][:] = val[i[0]]
        else:
            raise ValueError(f"cpu_run_graph: op {op} not needed by the benchmark programs")
    return time.perf_counter() - t0


def measure_program_latency(ev, keys, args):
    """BASELINE config 4's program on this GPU: 32-bit multiply (low word) then greater-than, BDD-derived MUX
    circuits (spf_b200.mux_circuits), 45 k CMUX + 192 circuit bootstraps over ~630 dependency levels; wall clock of
    CompiledGraph.run() including the H2D of the 96 input and D2H of the 33 output ciphertexts."""
    import oracle as O  # client-side encrypt/decrypt + the CPU baseline; never on the measured path

    import spf_b200
    from spf_b200.circuits import multiply_then_greater_than

    client = O.Client(keys)
    w, a, b, c = 32, 0xDEADBEEF, 0x12345679, 0x40000000
    slab = iter(spf_b200.pinned_zeros((3 * w + 2 * (w + 1), keys.glwe_len)))  # one page-locked slab for all buffers

    def enc(v):
        out = [next(slab) for _ in range(w)]
        for i, r in enumerate(out):
            r[:] = client.encrypt_glwe_l1([(v >> i) & 1])
        return out

    ab, bb, cb = enc(a), enc(b), enc(c)
    mk_out = lambda: ([[next(slab) for _ in range(w)]], [next(slab)])

    def check(out_prod, out_gt):
        prod = sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(out_prod[0]))
        return prod == (a * b) % (1 << w) and int(client.decrypt_glwe_l1(out_gt[0])[0]) == int(prod > c)

    out_prod, out_gt = mk_out()
    t0 = time.perf_counter()
    circ = multiply_then_greater_than([ab], [bb], [cb], out_prod, out_gt, 1)
    build_ms = 1e3 * (time.perf_counter() - t0)      # cold: includes generating the 16x16 multiplier BDDs (once per process)
    t0 = time.perf_counter()
    circ = multiply_then_greater_than([ab], [bb], [cb], out_prod, out_gt, 1)
    expand_ms = 1e3 * (time.perf_counter() - t0)     # warm: MUX circuits cached, expansion + pruning only
    g = spf_b200.CircuitProcessor(ev).compile(circ)
    g.run()
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        g.run()
        ts.append(time.perf_counter() - t0)
    n_op = lambda name: sum(1 for nd in circ.nodes if nd[0] == spf_b200.OP[name])
    res = {"program": "mul32 (low word) then greater-than", "cmux": n_op("CMux"), "circuit_bootstraps": n_op("CircuitBootstrap"),
           "levels": g.levels, "launches": g.launches, "gpu_ms": 1e3 * float(np.median(ts)), "gpu_ms_min": 1e3 * min(ts),
           "host_graph_build_ms": build_ms, "host_graph_build_warm_ms": expand_ms, "correct": check(out_prod, out_gt)}
    g.close()
    if not args.no_cpu_baseline:
        nt = O.hw_threads()
        out_prod, out_gt = mk_out()
        ccirc = multiply_then_greater_than([ab], [bb], [cb], out_prod, out_gt, 1)
        dt = cpu_run_graph(keys, ccirc, nt)
        res.update({"cpu_port_ms": 1e3 * dt, "cpu_threads": nt, "cpu_correct": check(out_prod, out_gt)})
    return res


def measure_add_latency(ev, keys, args):
    import oracle as O  # client-side encrypt/decrypt + the CPU baseline; never on the measured path

    import spf_b200
    from spf_b200.circuits import ripple_carry_adder

    client = O.Client(keys)
    proc = spf_b200.CircuitProcessor(ev)
    res = {"graph": "hand-built ripple-carry MUX tree (functionally equivalent to mux_circuits' BDD adder, not "
                    "node-for-node; SURVEY.md section 7)", "includes": "H2D of 2w GLWE inputs + D2H of w+1 GLWE outputs"}
    for w, a, b in ((8, 2, 7), (32, 0xDEADBEEF, 0x12345679)):
        slab = spf_b200.pinned_zeros((3 * w + 1, keys.glwe_len))  # one page-locked slab for all 3w + 1 buffers
        ab, bb, outs = list(slab[:w]), list(slab[w:2 * w]), list(slab[2 * w:])
        for i in range(w):
            ab[i][:] = client.encrypt_glwe_l1([(a >> i) & 1])
            bb[i][:] = client.encrypt_glwe_l1([(b >> i) & 1])
        g = proc.compile(ripple_carry_adder(ab, bb, outs))
        g.run()
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            g.run()
            ts.append(time.perf_counter() - t0)
        got = sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(outs))
        entry = {"gpu_ms": 1e3 * float(np.median(ts)), "gpu_ms_min": 1e3 * min(ts), "levels": g.levels,
                 "launches": g.launches, "correct": got == a + b}
        g.close()
        if not args.no_cpu_baseline:
            nt = O.hw_threads()
            dt, couts = cpu_add_latency(keys, ab, bb, nt)
            cgot = sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(couts))
            entry.update({"cpu_port_ms": 1e3 * dt, "cpu_threads": nt, "cpu_correct": cgot == a + b})
        res[f"add{w}"] = entry
        # the same add with the reference's own BDD-derived adder circuit (mux_circuits::add::ripple_carry_adder):
        # more multiplexers (O(w^2): every sum bit carries its own copy of the carry chain), the same depth
        from spf_b200.circuits import bdd_adder

        for o in outs:
            o[:] = 0
        circ = bdd_adder(ab, bb, outs)
        g = proc.compile(circ)
        g.run()
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            g.run()
            ts.append(time.perf_counter() - t0)
        got = sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(outs))
        res[f"add{w}_bdd_circuit"] = {"gpu_ms": 1e3 * float(np.median(ts)), "levels": g.levels, "launches": g.launches,
                                      "cmux": int((circ.ops == spf_b200.OP["CMux"]).sum()), "correct": got == a + b}
        g.close()
    return res


# ---------------------------------------------------------------------------------------------
# end to end the way the reference uses the path: LWE in -> circuit bootstrap -> CMUX -> GLWE out
# ---------------------------------------------------------------------------------------------
class E2EGraphPipeline:
    """The whole batch as a few FheCircuit graphs (InputLwe0 -> CircuitBootstrap -> CMux(sel, a, b) -> OutputGlwe1) on
    the asynchronous executor (spf_b200_graph_spawn): host buffers are rows of page-locked slabs, every graph's H2D /
    D2H copies are inside the timed region and overlap the neighbouring graphs' kernels.  The GGSWs never leave the
    device -- as in the reference, where L1GgswCiphertext is not even serialisable (crypto/encryption.rs:94-98)."""

    def __init__(self, ev, h_lwe: np.ndarray, glwe_len: int, wave: int, mode: str = "double", depth: int = 4):
        import spf_b200

        B = len(h_lwe)
        self.B = B
        self.mode = mode
        self.h_lwe = h_lwe                                         # [B][n + 1], page-locked
        ab = spf_b200.pinned_zeros((2, glwe_len))
        ab[1, glwe_len // 2] = np.uint64(1 << 63)                  # a = trivial 0, b = trivial 1: the output decrypts to the selector
        self.ab = ab
        proc = spf_b200.CircuitProcessor(ev)

        def build(lo, hi, out):
            c = spf_b200.FheCircuit()
            na, nb = c.add("InputGlwe1", io=ab[0]), c.add("InputGlwe1", io=ab[1])
            ins = [c.add("InputLwe0", io=h_lwe[i]) for i in range(lo, hi)]
            sels = [c.add("CircuitBootstrap", x) for x in ins]
            mux = [c.add("CMux", sl, na, nb) for sl in sels]
            for i, m in zip(range(lo, hi), mux):
                c.add("OutputGlwe1", m, io=out[i])
            return proc.compile(c)

        if mode == "double":
            # One graph = one whole step (the executor's own step schedule applies: capi.cu::launch_cbs packs the sub-wave
            # remainder of the blind rotation next to the trace kernels); `depth` such graphs with their own host result
            # buffers take turns: steps k + 1 .. k + depth - 1 are already spawned while step k's results travel to the host,
            # so a blind rotation is always queued when the previous step's trace kernels drain.
            self.depth = max(2, depth)
            if self.depth > 4:
                ev.set_max_in_flight(self.depth)  # the executor's flow control admits 4 spawned graphs by default
            self.h_outs = [spf_b200.pinned_zeros((B, glwe_len)) for _ in range(self.depth)]
            self.graphs = [build(0, B, o) for o in self.h_outs]
            self.h_out = self.h_outs[0]
            self.h2d = int(h_lwe.nbytes + ab.nbytes)
        else:
            self.h_out = spf_b200.pinned_zeros((B, glwe_len))      # [B][2N]
            # chunks: whole PBS waves (3 waves each) so that chunking costs no extra tail; the remainder is its own graph
            per = 3 * wave
            bounds = list(range(0, B, per)) + [B]
            if len(bounds) > 2 and bounds[-1] - bounds[-2] < wave:
                del bounds[-2]  # a remainder below one wave rides with the last chunk
            self.graphs = [build(lo, hi, self.h_out) for lo, hi in zip(bounds[:-1], bounds[1:])]
            self.h2d = int(h_lwe.nbytes + len(self.graphs) * ab.nbytes)
        self.d2h = int(self.h_out.nbytes)

    def step(self):
        for g in self.graphs:  # "double": both whole-step graphs once (warm-up)
            g.spawn()
        for g in self.graphs:
            g.wait()

    def run(self, steps: int):
        """`steps` steps as a stream.  "double": the two whole-step graphs alternate, step k + 1 is spawned before step
        k's results are awaited.  "chunks": a chunk graph is spawned again for the next step as soon as its results of
        this step have arrived on the host.  Either way every step pays all of its H2D and D2H copies."""
        if self.mode == "double":
            d = self.depth
            for k in range(steps):
                if k >= d:
                    self.graphs[k % d].wait()     # step k - d is complete on the host: its consumer may read h_outs[k % d]
                self.graphs[k % d].spawn()
            for k in range(max(0, steps - d), steps):
                self.graphs[k % d].wait()
            self.h_out = self.h_outs[(steps - 1) % d]
            return
        for g in self.graphs:
            g.spawn()
        for _ in range(steps - 1):
            for g in self.graphs:
                g.wait()
                g.spawn()
        for g in self.graphs:
            g.wait()

    def close(self):
        for g in self.graphs:
            g.close()


def measure_sweep(ev, lwe_sk, p, world, rank, dev, stream, flush, batches=(64, 1024, 16384)):
    """BASELINE config 5 in three points: device-resident CBS throughput per batch size, every rank its own batch,
    whole-job rate = world * B / max-over-ranks CUDA-event time."""
    import torch
    import torch.distributed as dist

    rows = []
    for B in batches:
        bits = np.random.default_rng(0x5EE9 + rank).integers(0, 2, B)
        d_in = torch.from_numpy(encrypt_lwe0_numpy(lwe_sk, bits, p.lwe_std, 0x5EE9 + rank).view(np.int64)).to(dev)
        d_out = torch.empty(B * ev.len_ggsw * 2, dtype=torch.float64, device=dev)
        fn = lambda: ev.dev_circuit_bootstrap(d_out.data_ptr(), d_in.data_ptr(), B, reference_scale=False, stream=stream)
        fn()
        ms = []
        for _ in range(3 if B <= 4096 else 2):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        t = torch.tensor([min(ms)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        rows.append({"batch_per_gpu": B, "ms": float(t.item()), "cbs_per_s": world * B / float(t.item()) * 1e3})
        del d_in, d_out
    return rows


def measure_sharded_graph(ev, keys, args, world, rank, dev):
    """BASELINE config 4 under the driver: `world` x (mul32 then greater-than) as ONE graph sharded over the ranks
    (spf_b200_graph_run_sharded): bootstrap levels split evenly, every MUX tree on one rank, level exchange over peer
    memory (NVLink P2P stores fused into the scheme-switch kernel + flag barriers) and, for comparison, NCCL all-gathers;
    rank 0 then runs the same graph alone.  Inputs are encrypted on rank 0 and broadcast; outputs are collected on
    rank 0 and decrypted."""
    import torch
    import torch.distributed as dist

    import spf_b200
    from spf_b200.circuits import multiply_then_greater_than
    from spf_b200.multi import NcclExchange, open_peer_arenas

    w, programs = 32, world
    glwe_len = ev.len_glwe
    n_in, n_out = programs * 3 * w, programs * (w + 1)
    slab = spf_b200.pinned_zeros((n_in + n_out, glwe_len))
    vals = None
    if rank == 0:
        import oracle as O

        client = O.Client(keys)
        rng = np.random.default_rng(2024)
        vals = [(int(rng.integers(0, 1 << w)), int(rng.integers(0, 1 << w)), int(rng.integers(0, 1 << w))) for _ in range(programs)]
        k = 0
        for v in vals:
            for x in v:
                for i in range(w):
                    slab[k] = client.encrypt_glwe_l1([(x >> i) & 1])
                    k += 1
    t_in = torch.from_numpy(slab[:n_in].view(np.int64)).to(dev)
    dist.broadcast(t_in, src=0)
    slab[:n_in] = t_in.cpu().numpy().view(np.uint64)
    rows = iter(slab)
    a, b, c = [], [], []
    for _ in range(programs):
        a.append([next(rows) for _ in range(w)]); b.append([next(rows) for _ in range(w)]); c.append([next(rows) for _ in range(w)])
    out_prod = [[next(rows) for _ in range(w)] for _ in range(programs)]
    out_gt = [next(rows) for _ in range(programs)]
    circ = multiply_then_greater_than(a, b, c, out_prod, out_gt, programs)
    out_nodes = [i for i, nd in enumerate(circ.nodes) if nd[0] == spf_b200.OP["OutputGlwe1"]]
    res = {"workload": f"{programs} x (mul32 low word then greater-than) as one graph, sharded over {world} GPUs",
           "cmux": int((circ.ops == spf_b200.OP["CMux"]).sum()), "circuit_bootstraps": int((circ.ops == spf_b200.OP["CircuitBootstrap"]).sum())}

    def timed(g, runs=3):
        ts = []
        for _ in range(runs + 1):
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            g.run()
            ts.append(1e3 * (time.perf_counter() - t0))
        t = torch.tensor([min(ts[1:])], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def collect_and_check(g):
        """every output lives on one rank (its tree's owner) or on all: sum the owners' copies on rank 0 and decrypt"""
        for node in out_nodes:
            r = g.output_rank(node)
            if not (r == rank or (r < 0 and rank == 0)):
                circ.nodes[node][3][:] = 0
        t = torch.from_numpy(slab[n_in:].view(np.int64)).to(dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        ok = None
        if rank == 0:
            got = t.cpu().numpy().view(np.uint64).reshape(n_out, glwe_len)
            ok, k = True, 0
            dec = [int(client.decrypt_glwe_l1(g_)[0]) for g_ in got]
            prods, gts = dec[:programs * w], dec[programs * w:]
            for p_, (x, y, z) in enumerate(vals):
                prod = sum(bit << i for i, bit in enumerate(prods[p_ * w:(p_ + 1) * w]))
                ok &= prod == (x * y) % (1 << w) and gts[p_] == int(prod > z)
        slab[n_in:] = 0
        return ok

    for mode in ("peer", "nccl"):
        ex = NcclExchange(rank) if mode == "nccl" else None
        g = spf_b200.CompiledGraph(ev, circ, world=world, rank=rank, exchange=ex)
        if mode == "peer":
            open_peer_arenas(g)
        res[f"ms_{mode}"] = timed(g)
        ok = collect_and_check(g)
        if rank == 0:
            res[f"correct_{mode}"] = bool(ok)
        if ex is not None:
            res["exchange_bytes_per_run"] = ex.bytes // 4
            res["exchanges_per_run"] = ex.calls // 4
        res["levels"], res["launches_per_rank"] = g.levels, g.launches
        g.close()
    # the same work on ONE GPU (rank 0; the other ranks wait), and one program alone: the latency floor
    if rank == 0:
        g = spf_b200.CompiledGraph(ev, circ)
        g.run()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter(); g.run(); ts.append(1e3 * (time.perf_counter() - t0))
        res["ms_same_work_1gpu"] = min(ts)
        g.close()
        one = multiply_then_greater_than(a[:1], b[:1], c[:1], out_prod[:1], out_gt[:1], 1)
        g = spf_b200.CompiledGraph(ev, one)
        g.run()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter(); g.run(); ts.append(1e3 * (time.perf_counter() - t0))
        res["ms_one_program_1gpu"] = min(ts)
        g.close()
        best = min(res["ms_peer"], res["ms_nccl"])
        res["speedup_vs_1gpu"] = res["ms_same_work_1gpu"] / best
        res["correct"] = bool(res.get("correct_peer") and res.get("correct_nccl"))
        res["limiter"] = ("per-program latency floor: one program is a chain of ~630 dependency levels (%.1f ms alone on one GPU), "
                          "a sharded run cannot finish before its slowest tree; the level exchange costs %.1f ms (peer) / %.1f ms (nccl) on top"
                          % (res["ms_one_program_1gpu"], res["ms_peer"] - res["ms_one_program_1gpu"], res["ms_nccl"] - res["ms_one_program_1gpu"]))
    dist.barrier()
    return res


def dump_outputs(d_out, B: int, len_ggsw: int, out_dir: str) -> None:
    """What a caller of the timed path receives from one step: B GGSW ciphertexts in the FFT domain at the device scale
    (reference_scale=False), len_ggsw complex128 each, stored as (real, imag) float64 pairs.  A whole step is 256 KiB per
    bootstrap at DEFAULT_128, so only a fixed seeded sample of the batch is written, in ascending batch order: two builds
    run with the same arguments see the same inputs and can be compared output for output."""
    import torch

    n = min(B, max(1, (32 << 20) // (len_ggsw * 16)))
    rows = np.sort(np.random.default_rng(0xD0).choice(B, n, replace=False))
    ggsw = d_out.view(B, len_ggsw, 2)[torch.from_numpy(rows).to(d_out.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "cbs_ggsw_fft.npy"), ggsw)


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist

    import spf_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; spf_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    p = spf_b200.default_128()
    l = spf_b200.lib()
    lens = [l.spf_b200_len_bsk(C.byref(p)), l.spf_b200_len_ksk(C.byref(p)), l.spf_b200_len_ssk(C.byref(p)),
            l.spf_b200_len_ak(C.byref(p))]

    # ---- compute key: generated once on rank 0, replicated to every GPU over NCCL -------------
    keys = None
    if rank == 0:
        import oracle as O  # client-side keygen + the cpu_baseline leg; never on the measured path

        keys = O.Keys()
    d_bsk = torch.empty(lens[0] * 2, dtype=torch.float64, device=dev)
    d_ksk = torch.empty(lens[1], dtype=torch.int64, device=dev)
    d_ssk = torch.empty(lens[2] * 2, dtype=torch.float64, device=dev)
    d_ak = torch.empty(lens[3] * 2, dtype=torch.float64, device=dev)
    sk0 = torch.empty(p.lwe_n, dtype=torch.int64, device=dev)
    if rank == 0:
        d_bsk.copy_(torch.from_numpy(keys.bsk_fft.view(np.float64)))
        d_ksk.copy_(torch.from_numpy(keys.ksk.view(np.int64)))
        d_ssk.copy_(torch.from_numpy(keys.ssk_fft.view(np.float64)))
        d_ak.copy_(torch.from_numpy(keys.ak_fft.view(np.float64)))
        sk0.copy_(torch.from_numpy(keys.lwe0_sk.view(np.int64)))
    key_bcast_ms = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        from spf_b200.multi import broadcast_compute_key

        broadcast_compute_key([d_bsk, d_ksk, d_ssk, d_ak, sk0], src=0)
        torch.cuda.synchronize()
        key_bcast_ms = 1e3 * (time.perf_counter() - t0)
    ev = spf_b200.Evaluation(d_bsk.data_ptr(), d_ksk.data_ptr(), d_ssk.data_ptr(), d_ak.data_ptr(), params=p,
                             device=local, on_device=True)
    del d_bsk, d_ksk, d_ssk, d_ak
    torch.cuda.empty_cache()

    # ---- inputs ---------------------------------------------------------------------------------
    B = args.batch
    lwe_sk = sk0.cpu().numpy().view(np.uint64)
    bits = np.random.default_rng(0xB2000002 + rank).integers(0, 2, B)
    cts = encrypt_lwe0_numpy(lwe_sk, bits, p.lwe_std, 0xB2000002 + rank)
    h_in = torch.from_numpy(cts.view(np.int64)).pin_memory()
    d_in = h_in.to(dev)
    d_out = torch.empty(B * ev.len_ggsw * 2, dtype=torch.float64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    # a dedicated (non-default) stream: kernels are launched on it through the C ABI and the
    # CUDA events below are recorded on it (torch.cuda.Event records on the current stream)
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    def step():
        ev.dev_circuit_bootstrap(d_out.data_ptr(), d_in.data_ptr(), B, reference_scale=False, stream=stream)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()

    # ---- timed region: K steps, CUDA events per step on the launching stream, L2 flushed between --
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = ev.kernel_launches
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    torch.cuda.synchronize()
    wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.zero_()
        starts[i].record()
        step()
        ends[i].record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    launches = ev.kernel_launches - launches0
    dev_ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    clocks = sampler.stop() if sampler else None
    value = world * B * args.steps / (dev_ms * 1e-3)
    if rank == 0 and args.dump_outputs:
        dump_outputs(d_out, B, ev.len_ggsw, args.dump_outputs)

    # ---- roofline of the dominant kernel (pbs_kernel), timed alone with CUDA events ------------
    roofline = None
    if rank == 0:
        lut = torch.from_numpy(cbs_lut().view(np.int64)).to(dev)
        rot = cts.copy()
        rot[:, -1] += np.uint64(1 << 62)
        d_rot = torch.from_numpy(rot.view(np.int64)).to(dev)
        d_glwe = torch.empty(B * ev.len_glwe, dtype=torch.int64, device=dev)
        for _ in range(2):
            ev.dev_programmable_bootstrap(d_glwe.data_ptr(), d_rot.data_ptr(), lut.data_ptr(), 0, 2, B, stream=stream)
        reps = max(2, min(args.steps, 5))
        ks = [torch.cuda.Event(enable_timing=True) for _ in range(reps)]
        ke = [torch.cuda.Event(enable_timing=True) for _ in range(reps)]
        for i in range(reps):
            flush.zero_()
            ks[i].record()
            ev.dev_programmable_bootstrap(d_glwe.data_ptr(), d_rot.data_ptr(), lut.data_ptr(), 0, 2, B, stream=stream)
            ke[i].record()
        torch.cuda.synchronize()
        pbs_ms = sum(a.elapsed_time(b) for a, b in zip(ks, ke)) / reps
        fp64_peak = ev.fp64_peak_tflops()
        achieved = FLOP_PER_PBS * B / (pbs_ms * 1e-3) / 1e12
        hbm_peak = None
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
            hbm_src = "MEASURED_PEAKS.json"
        except Exception:
            hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
        alg_bytes = BSK_BYTES + B * PBS_IO_BYTES
        roofline = {
            "kernel": "pbs_kernel", "bound": "fp64", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
            "frac": achieved / fp64_peak if fp64_peak else None,
            "peak_source": "measured in this run: spf_b200_fp64_peak (dependent-free DFMA probe on all SMs); "
                           "MEASURED_PEAKS.json carries no FP64 figure",
            "flop_per_launch": FLOP_PER_PBS * B, "ms_per_launch": pbs_ms,
            "share_of_step": pbs_ms / (dev_ms / args.steps) if dev_ms else None,
            "note": "timed alone (whole waves on pbs_kernel, a sub-wave remainder on the latency kernel); inside a step the remainder "
                    "runs packed three to an SM concurrently with the trace / scheme-switch kernels (capi.cu::launch_cbs), so the "
                    "step is shorter than this plus the trace kernels",
            "hbm": {"achieved": alg_bytes / (pbs_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                    "frac": alg_bytes / (pbs_ms * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes": alg_bytes,
                    "peak_source": hbm_src},
            # dram__bytes_read.sum + dram__bytes_write.sum of one launch (bytes), from the committed ncu capture
            "traffic": (ncu_traffic(B) or {}).get("bytes_per_launch"), "traffic_detail": ncu_traffic(B),
            # pipe utilisation of the same kernel from the committed ncu capture (what binds it: DESIGN.md K3)
            "ncu_pipes": ncu_pipes(),
        }
        del d_rot, d_glwe, lut

    # ---- end to end (headline): LWE in -> CBS -> CMUX -> GLWE out through the graph API on the asynchronous executor,
    #      host buffers (page-locked slabs), H2D + D2H inside the timed region -----------------------------------------
    e2e = e2e_ggsw = None
    e2e_out = None
    if not args.no_e2e:
        lwe_len = p.lwe_n + 1
        h_lwe = h_in.numpy().view(np.uint64).reshape(B, lwe_len)
        pipe = E2EGraphPipeline(ev, h_lwe, ev.len_glwe, 148 * 3, os.environ.get("SPF_B200_E2E_MODE", "double"),
                                int(os.environ.get("SPF_B200_E2E_DEPTH", "4")))
        pipe.step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e2e_steps = 16  # a stream of whole-step graphs: long enough that the ramp (first H2D, last D2H) does not dominate
        t0 = time.perf_counter()
        pipe.run(e2e_steps)
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
        e2e = {"value": world * B * e2e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": pipe.h2d, "d2h_bytes_per_step": pipe.d2h,
               "steps": e2e_steps, "graphs_per_step": 1 if pipe.mode == "double" else len(pipe.graphs),
               "pipelining": ("%d whole-step graphs with their own page-locked result buffers take turns: the next steps are "
                              "spawned before step k's results are awaited" % pipe.depth if pipe.mode == "double" else
                              "chunk graphs, each re-spawned for step k + 1 once its step-k outputs are on the host"),
               "api": "FheCircuit graphs (InputLwe0 -> CircuitBootstrap -> CMux -> OutputGlwe1) through spf_b200_graph_spawn / "
                      "spf_b200_graph_wait, page-locked host buffers; the GGSWs stay in HBM as in the reference "
                      "(L1GgswCiphertext is not serialisable, crypto/encryption.rs:94-98)"}
        e2e_out = pipe.h_out.copy()
        pipe.close()
        del pipe
        # the round-1 e2e for continuity (1 GPU only): GGSW results shipped to the host, 256 KiB per bootstrap -- a transfer the
        # reference never makes; at 8 GPUs it measures the host's PCIe / memory system (SCALE_r01: 0.85 efficiency)
        if world == 1:
            h_out = torch.empty(B * ev.len_ggsw * 2, dtype=torch.float64).pin_memory()
            lib = spf_b200.lib()

            def host_step():
                rc = lib.spf_b200_circuit_bootstrap(ev.handle, h_out.data_ptr(), h_in.data_ptr(), B)
                if rc != 0:
                    raise RuntimeError(lib.spf_b200_last_error(ev.handle))

            host_step()
            t0 = time.perf_counter()
            n_h = max(1, min(args.steps, 3))
            for _ in range(n_h):
                host_step()
            dt = time.perf_counter() - t0
            e2e_ggsw = {"value": B * n_h / dt, "unit": UNIT, "h2d_bytes_per_step": int(h_in.numel() * 8),
                        "d2h_bytes_per_step": int(h_out.numel() * 8), "steps": n_h,
                        "api": "spf_b200_circuit_bootstrap (host pointers, pinned): GGSW-FFT outputs copied to the host"}
            del h_out

    # ---- checker + CPU baseline (rank 0, N = 1 only for the baseline) --------------------------
    check = None
    cpu_baseline = None
    if rank == 0:
        import oracle as O

        client = O.Client(keys)
        if args.check > 0:
            # outputs spread over every PBS wave (444 ciphertexts each) and both sides of every wave boundary
            nchk = min(args.check, B)
            idx = set(np.linspace(0, B - 1, nchk).astype(int).tolist())
            idx |= {i for w0 in range(444, B, 444) for i in (w0 - 1, w0) if i < B}
            idx = sorted(idx)
            tmp = torch.empty(ev.len_ggsw * 2, dtype=torch.float64, device=dev)
            bad = []
            for i in idx:
                ev.dev_fft_rescale(tmp.data_ptr(), d_out.data_ptr() + i * ev.len_ggsw * 16, ev.len_ggsw, to_device=False, stream=stream)
                torch.cuda.synchronize()
                if client.decrypt_ggsw_l1(tmp.cpu().numpy().view(np.complex128)) != int(bits[i]):
                    bad.append(i)
            check = {"decrypted": len(idx), "ok": not bad, "what": "GGSW outputs of the timed device-resident steps"}
            if e2e_out is not None:
                bad_e = [i for i in idx if int(client.decrypt_glwe_l1(e2e_out[i])[0]) != int(bits[i])]
                check.update({"e2e_decrypted": len(idx), "e2e_ok": not bad_e})
                bad += bad_e
            if bad:
                raise SystemExit(f"bench.py: GPU outputs do not decrypt to the expected plaintexts: {bad[:16]}")
        if world == 1 and not args.no_cpu_baseline:
            nt = O.hw_threads()
            rate0, _ = cpu_cbs_rate(keys, cts[: min(2 * nt, B)], nt)  # warm-up, also sizes the sample
            sample = args.cpu_sample or cpu_sample_size(rate0, nt, B)
            rate, dt = cpu_cbs_rate(keys, cts[: min(sample, B)], nt)
            cpu_baseline = {"value": rate, "unit": UNIT, "cores": nt, "kind": "port",
                            "sample": f"{min(sample, B)} CBS of the same workload in {dt:.1f} s; " + CPU_KIND_NOTE,
                            **cpu_micro(keys, cts)}

    # ---- BASELINE config 5 (3-point batch sweep) and config 4 (sharded program graph, N > 1) ----------------------
    sweep = sharded = None
    if not args.no_sweep:
        sweep = measure_sweep(ev, lwe_sk, p, world, rank, dev, stream, flush)
    if world > 1 and not args.no_sharded_graph:
        sharded = measure_sharded_graph(ev, keys, args, world, rank, dev)

    # ---- Parasol add latency (the metric's second half): encrypted w-bit add through the graph
    #      executor (16/64 x SampleExtract -> Keyswitch -> CBS, then the ripple-carry MUX tree) ------
    add_latency = program_latency = None
    if rank == 0 and world == 1 and not args.no_add:
        add_latency = measure_add_latency(ev, keys, args)
        program_latency = measure_program_latency(ev, keys, args)  # BASELINE config 4's program on one GPU

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"cbs_batch{B}_default128 (BASELINE config 3: batched circuit bootstrapping, "
                                   f"{B} independent LWE inputs per B200)",
                       "params": "DEFAULT_128 (n=637, k=1, N=2048, pbs l=2 logB=16)", "batch_per_gpu": B,
                       "parallelism": f"replicas x{world}, batch sharded, no data-path collective",
                       "l2": "256 MiB memset between timed steps; the 83 MB BSK is re-fetched from HBM every step",
                       "key_broadcast_ms": key_bcast_ms},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
            "cpu_baseline": cpu_baseline, "check": check, "wall_s_timed_region": wall,
            "parasol_add_latency": add_latency, "parasol_mul32_cmp_latency": program_latency,
            "e2e_ggsw_to_host": e2e_ggsw, "throughput_sweep": sweep, "sharded_graph": sharded,
        }
        print(json.dumps(line))
    ev.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
