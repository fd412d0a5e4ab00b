"""Blocking latency of instructions with a plaintext operand against the same instructions on two encrypted operands, on
one GPU (cuda:0).  Per instruction and width (8, 16, 32): warm-up calls, then the median and spread of --runs calls of
each form, alternated, each timed on the host around the blocking InstructionCache call; the graph's circuit
bootstraps, CMUX levels (the longest chain of CMux nodes), levels and launches.  The constant of width w is a seeded
random w-bit value (the same for every instruction of that width); the multiplies are also timed by the small constant
10.  Encrypted x encrypted multiplies above 16 bits and shifts by an encrypted amount above 16 bits cannot be built
(their row has "encrypted": null).  Also a block of 8 independent 32-bit x + c against 8 x + y.  The card's name and
power limit are read in the same run.  One JSON document to --out.
usage: python tools/plain_latency.py [--widths 8 16 32] [--runs 20] [--warmup 2] [--out profiles/plain_latency_n1.json]"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle as O  # input generation only
import spf_b200
from isa_latency import gpu_info
from spf_b200.circuits import SHIFT_MAX_WIDTH, InstructionCache, Plain


def instructions(w, k):
    """(name, call(cache, a, b) -> graph, whether the encrypted form exists): b is the second operand, encrypted or
    Plain(k, w); select's plaintext form has a plaintext condition, the shift's a plaintext amount."""
    lg = max(1, (w - 1).bit_length())
    out = lambda n: [np.zeros(4096, np.uint64) for _ in range(n)]
    yield "add", lambda c, a, b: c.add(a, b, out(w + 1)), True
    yield "sub", lambda c, a, b: c.sub(a, b, out(w)), True
    yield "compare_gt", lambda c, a, b: c.compare(a, b, out(1)[0], "gt"), True
    yield "compare_gt_signed", lambda c, a, b: c.compare(a, b, out(1)[0], "gt", signed=True), True
    yield "equal", lambda c, a, b: c.equal(a, b, out(1)[0]), True
    yield "and_", lambda c, a, b: c.and_(a, b, out(w)), True
    yield "or_", lambda c, a, b: c.or_(a, b, out(w)), True
    yield "select", lambda c, a, b: c.select(Plain(k & 1, 1) if isinstance(b, Plain) else b[0], a, a[::-1], out(w)), True
    yield "shift_right_logical", lambda c, a, b: c.shift(a, Plain(k % w, lg) if isinstance(b, Plain) else b[:lg], out(w), True), \
        w <= SHIFT_MAX_WIDTH
    yield "multiply", lambda c, a, b: c.multiply(a, b, out(w)), w <= 16
    yield "multiply_signed", lambda c, a, b: c.multiply_signed(a, b, out(w)), w <= 16


def graph_row(g):
    keep = g._keep
    ops, ins = keep.ops, keep.inputs_of
    depth = np.zeros(len(keep), np.int64)
    cmux = spf_b200.OP["CMux"]
    for i in range(len(keep)):
        srcs = ins[i][ins[i] >= 0]
        depth[i] = (depth[srcs].max() if len(srcs) else 0) + (ops[i] == cmux)
    return {"bootstraps": int((ops == spf_b200.OP["CircuitBootstrap"]).sum()), "cmux_levels": int(depth.max(initial=0)),
            "levels": g.levels, "launches": g.launches}


def timed(forms, runs, warmup):
    """forms: {label: call() -> graph}; warm-up, then alternate.  Returns {label: stats + graph fields}."""
    out = {}
    for label, call in forms.items():
        t0 = time.perf_counter()
        g = call()
        out[label] = {"first_call_ms": round(1e3 * (time.perf_counter() - t0), 1), **graph_row(g)}
        out[label]["_graph"] = g
        for _ in range(warmup):
            call()
    ts = {label: [] for label in forms}
    for _ in range(runs):
        for label, call in forms.items():
            t0 = time.perf_counter()
            call()
            ts[label].append(1e3 * (time.perf_counter() - t0))
    for label, t in ts.items():
        t = np.asarray(t)
        out[label].update({"median_ms": round(float(np.median(t)), 3), "p10_ms": round(float(np.percentile(t, 10)), 3),
                           "p90_ms": round(float(np.percentile(t, 90)), 3), "runs": len(t)})
        out[label].pop("_graph").close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--widths", type=int, nargs="+", default=[8, 16, 32])
    ap.add_argument("--runs", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    keys = O.Keys()
    client = O.Client(keys)
    ev = spf_b200.Evaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft)
    rng = np.random.default_rng(1)
    enc = lambda v, w: [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]
    rows = []
    for w in args.widths:
        a, b, k = enc(int(rng.integers(0, 1 << w)), w), enc(int(rng.integers(0, 1 << w)), w), int(rng.integers(0, 1 << w))
        for name, call, encrypted in instructions(w, k):
            for const in [k] + ([10] if name.startswith("multiply") else []):
                forms = {"plain": lambda call=call, c=InstructionCache(ev), p=Plain(const, w): call(c, a, p)}
                if encrypted:
                    forms["encrypted"] = lambda call=call, c=InstructionCache(ev): call(c, a, b)
                res = timed(forms, args.runs, args.warmup)
                row = {"instruction": name, "width": w, "constant": const, "plain": res["plain"], "encrypted": res.get("encrypted")}
                rows.append(row)
                print(json.dumps(row), flush=True)
    # a block of 8 independent 32-bit x + c against 8 x + y
    blocks = {}
    xs = [enc(int(v), 32) for v in rng.integers(0, 1 << 32, 16, dtype=np.uint64)]
    for label in ("plain", "encrypted"):
        cache = InstructionCache(ev)
        blk = cache.block()
        regs = [blk.reg(32) for _ in range(8 if label == "plain" else 16)]
        sums = [blk.reg(33) for _ in range(8)]
        for i, s in enumerate(sums):
            blk.add(regs[i], Plain(int(rng.integers(0, 1 << 32)), 32) if label == "plain" else regs[8 + i], s)
        bind = {r: x for r, x in zip(regs, xs)}
        outs = {s: [np.zeros(4096, np.uint64) for _ in range(33)] for s in sums}
        blocks[label] = lambda blk=blk, bind=bind, outs=outs: blk.run(bind, outs)
    res = timed(blocks, args.runs, args.warmup)
    block_row = {"block": "8 independent 32-bit adds", "plain": res["plain"], "encrypted": res["encrypted"]}
    print(json.dumps(block_row), flush=True)
    doc = {**gpu_info(), "device": "cuda:0", "timing": "host clock around the blocking InstructionCache call, the two forms alternated",
           "warmup": args.warmup, "results": rows, "block": block_row}
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    ev.close()


if __name__ == "__main__":
    main()
