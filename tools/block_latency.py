"""Fused vs one-by-one: each workload run as ONE InstructionCache.block() graph against the same instructions run one at
a time through InstructionCache (one blocking graph each, results copied to the host and back in between).  Both forms
are warmed up, then timed alternately, --runs times each, on the host clock around the blocking call(s); the median and
spread of each, the levels, launches and circuit bootstraps of the fused graph and of the one-by-one graphs together,
the largest circuit-bootstrap stage of the fused graph and the blind-rotation kernel launch_pbs picks for it
(pbs_quad_kernel up to one ciphertext per SM), and the card's name and power limit.  One JSON document to --out.
Workloads: N independent 32-bit adds (N = 1, 2, 4, 8; 64 N bootstraps in one stage, crossing the SM count between
N = 2 and N = 4), a dependent 16-bit chain (sub, signed compare, select, constant shift), a mixed 8-bit block that
reads its registers several times, and the 8 adds on a two-rank box (both ranks on cuda:0).
usage: python tools/block_latency.py [--runs 20] [--warmup 2] [--out profiles/block_latency_n1.json]"""
import argparse
import collections
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle as O  # input generation only
import spf_b200
from spf_b200.circuits import InstructionCache


class R:
    """A register reference in a workload: the whole register `name`, or one bit of it."""

    def __init__(self, name, bit=None):
        self.name, self.bit = name, bit


def adds(n, w=32):
    regs = {**{f"a{i}": w for i in range(n)}, **{f"b{i}": w for i in range(n)}, **{f"s{i}": w + 1 for i in range(n)}}
    prog = [("add", (R(f"a{i}"), R(f"b{i}"), R(f"s{i}")), {}) for i in range(n)]
    return regs, prog, [f"a{i}" for i in range(n)] + [f"b{i}" for i in range(n)], [f"s{i}" for i in range(n)]


def chain16(w=16):
    regs = {"a": w, "b": w, "c": w, "d": w, "f": 1, "g": w, "h": w}
    prog = [("sub", (R("a"), R("b"), R("d")), {}),
            ("compare", (R("d"), R("c"), R("f", 0), "gt"), {"signed": True}),
            ("select", (R("f", 0), R("a"), R("b"), R("g")), {}),
            ("shift_const", (R("g"), 3, R("h"), True, "arithmetic"), {})]
    return regs, prog, ["a", "b", "c"], ["d", "f", "h"]


def mixed8(w=8):
    """a, b and c are each read by three or four instructions; the fused graph bootstraps each once."""
    regs = {"a": w, "b": w, "c": w, "s": w + 1, "d": w + 1, "ge": 1, "eq": 1, "n": w, "o": w}
    prog = [("add", (R("a"), R("b"), R("s")), {}),
            ("sub", (R("a"), R("c"), R("d")), {}),
            ("compare", (R("a"), R("c"), R("ge", 0), "ge"), {}),
            ("equal", (R("b"), R("c"), R("eq", 0)), {}),
            ("and_", (R("a"), R("b"), R("n")), {}),
            ("or_", (R("b"), R("c"), R("o")), {})]
    return regs, prog, ["a", "b", "c"], ["s", "d", "ge", "eq", "n", "o"]


class Workload:
    """One workload recorded twice: as a Block of `fused_cache`, and as host buffers (or box handles) per register for
    the one-by-one calls of `seq_cache`.  io: (alloc(w) -> w zero ciphertexts, put(ciphertexts) -> bound inputs,
    get(buffer) -> host ciphertext)."""

    def __init__(self, ev, enc, io, regs, prog, ins, outs, rng):
        alloc, put, self.get = io
        self.prog, self.ins, self.outs = prog, ins, outs
        self.fused_cache, self.seq_cache = InstructionCache(ev), InstructionCache(ev)
        self.blk = self.fused_cache.block()
        self.regs = {n: self.blk.reg(w) for n, w in regs.items()}
        for name, args, kw in prog:
            getattr(self.blk, name)(*[self._ref(a, self.regs) for a in args], **kw)
        self.bufs = {n: put(enc(int(rng.integers(0, 1 << regs[n])), regs[n])) if n in ins else alloc(w)
                     for n, w in regs.items()}
        self.fused_out = {n: alloc(regs[n]) for n in outs}

    @staticmethod
    def _ref(a, regs):
        return (regs[a.name] if a.bit is None else regs[a.name][a.bit]) if isinstance(a, R) else a

    def fused(self):
        return self.blk.run({self.regs[n]: self.bufs[n] for n in self.ins}, {self.regs[n]: self.fused_out[n] for n in self.outs})

    def one_by_one(self):
        return [getattr(self.seq_cache, name)(*[self._ref(a, self.bufs) for a in args], **kw) for name, args, kw in self.prog]


def cbs(g):
    return int((g._keep.ops == spf_b200.OP["CircuitBootstrap"]).sum())


def stats(ts):
    ts = np.asarray(ts)
    return {"median_ms": round(float(np.median(ts)), 3), "p10_ms": round(float(np.percentile(ts, 10)), 3),
            "p90_ms": round(float(np.percentile(ts, 90)), 3), "min_ms": round(float(ts.min()), 3),
            "max_ms": round(float(ts.max()), 3)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["unknown, unknown"])[0].split(", ")
    return {"gpu": name, "power_limit": power}


def measure(name, wl, runs, warmup, sm_count, client):
    for _ in range(warmup):
        wl.fused()
        wl.one_by_one()
    tf, ts = [], []
    for _ in range(runs):  # alternate the two forms so drift on a shared host hits both alike
        t0 = time.perf_counter()
        g = wl.fused()
        tf.append(1e3 * (time.perf_counter() - t0))
        t0 = time.perf_counter()
        seq = wl.one_by_one()
        ts.append(1e3 * (time.perf_counter() - t0))
    assert wl.fused_cache.misses == 1
    dec = lambda bufs: [int(client.decrypt_glwe_l1(wl.get(b))[0]) for b in bufs]
    assert all(dec(wl.fused_out[n]) == dec(wl.bufs[n]) for n in wl.outs), f"{name}: fused and one-by-one results differ"
    level, _ = spf_b200.plan_graph(g._keep)
    stages = collections.Counter(level[g._keep.ops == spf_b200.OP["CircuitBootstrap"]].tolist())
    big = max(stages.values())
    row = {"workload": name, "runs": runs,
           "fused": {**stats(tf), "levels": g.levels, "launches": g.launches, "bootstraps": cbs(g),
                     "bootstrap_stages": len(stages), "largest_stage": big,
                     "largest_stage_kernel": "pbs_quad_kernel" if big <= sm_count else "pbs_kernel"},
           "one_by_one": {**stats(ts), "instructions": len(seq), "levels": sum(x.levels for x in seq),
                          "launches": sum(x.launches for x in seq), "bootstraps": sum(cbs(x) for x in seq)}}
    row["speedup"] = round(row["one_by_one"]["median_ms"] / row["fused"]["median_ms"], 2)
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch

    sm_count = torch.cuda.get_device_properties(0).multi_processor_count
    keys = O.Keys()
    client = O.Client(keys)
    enc = lambda v, w: [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]
    host = (lambda w: [np.zeros(4096, np.uint64) for _ in range(w)], lambda cts: cts, lambda b: b)
    rng = np.random.default_rng(1)
    rows = []
    run = lambda name, ev, io, workload: rows.append(
        measure(name, Workload(ev, enc, io, *workload, rng), args.runs, args.warmup, sm_count, client))
    ev = spf_b200.Evaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft)
    for n in (1, 2, 4, 8):
        run(f"add32_x{n}", ev, host, adds(n))
    run("chain16_sub_cmp_select_shiftconst", ev, host, chain16())
    run("mixed8_shared_reads", ev, host, mixed8())
    ev.close()
    box = spf_b200.BoxEvaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft, devices=[0, 0])

    def put(cts):
        hs = [spf_b200.BoxCiphertext.alloc(box, "Glwe1") for _ in cts]
        for h, ct in zip(hs, cts):
            h.write(ct)
        return hs

    handles = (lambda w: put([np.zeros(4096, np.uint64)] * w), put, lambda h: h.read(0))
    run("box2_add32_x8", box, handles, adds(8))
    box.close()
    doc = {**gpu_info(), "device": "cuda:0", "sm_count": sm_count,
           "timing": "host clock around the blocking call(s): Block.run for fused, every InstructionCache call for one_by_one",
           "box": "two ranks on cuda:0", "warmup": args.warmup, "results": rows}
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
