"""Blocking latency of every InstructionCache instruction on one GPU (cuda:0): per instruction and width (8, 16, 32 where
the instruction allows it), warm-up calls, then the median and spread of --runs calls, each timed on the host around
the blocking call (operand rebinding, copies in and out, the run).  Also records the graph's levels, launches and
circuit-bootstrap count, and the card's name and power limit.  One JSON document to --out.
usage: python tools/isa_latency.py [--widths 8 16 32] [--runs 20] [--warmup 2] [--out profiles/isa_latency_n1.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle as O  # input generation only
import spf_b200
from spf_b200.circuits import SHIFT_MAX_WIDTH, InstructionCache


def instructions(w):
    """(name, call(cache, a, b, sel, amount) -> graph) for width w: a, b w-bit operands, sel one bit, amount w bits."""
    half, lg = w // 2, max(1, (w - 1).bit_length())
    out = lambda n: [np.zeros(4096, np.uint64) for _ in range(n)]
    yield "add", lambda c, a, b, s, k: c.add(a, b, out(w + 1))
    yield "sub", lambda c, a, b, s, k: c.sub(a, b, out(w))
    yield "neg", lambda c, a, b, s, k: c.neg(a, out(w))
    yield "greater_than", lambda c, a, b, s, k: c.greater_than(a, b, out(1)[0])
    for op in ("gt", "ge", "lt", "le"):
        for signed in (False, True):
            yield f"compare_{op}{'_signed' if signed else ''}", lambda c, a, b, s, k, op=op, sg=signed: c.compare(a, b, out(1)[0], op, signed=sg)
    yield "equal", lambda c, a, b, s, k: c.equal(a, b, out(1)[0])
    yield "not_equal", lambda c, a, b, s, k: c.not_equal(a, b, out(1)[0])
    yield "and_", lambda c, a, b, s, k: c.and_(a, b, out(w))
    yield "or_", lambda c, a, b, s, k: c.or_(a, b, out(w))
    yield "xor", lambda c, a, b, s, k: c.xor(a, b, out(w))
    yield "not_", lambda c, a, b, s, k: c.not_(a, out(w))
    for right, mode in ((False, "logical"), (True, "logical"), (True, "arithmetic"), (False, "rotation")):
        if w <= SHIFT_MAX_WIDTH:
            yield f"shift_{'right' if right else 'left'}_{mode}", lambda c, a, b, s, k, r=right, m=mode: c.shift(a, k[:lg], out(w), r, m)
    yield "shift_const_right_logical", lambda c, a, b, s, k: c.shift_const(a, half, out(w), True)
    yield "select", lambda c, a, b, s, k: c.select(s, a, b, out(w))
    yield "zext", lambda c, a, b, s, k: c.zext(a, out(2 * w))
    yield "sext", lambda c, a, b, s, k: c.sext(a, out(2 * w))
    yield "trunc", lambda c, a, b, s, k: c.trunc(a, out(half))
    if w <= 16:
        yield "multiply", lambda c, a, b, s, k: c.multiply(a, b, out(w))
        yield "multiply_signed", lambda c, a, b, s, k: c.multiply_signed(a, b, out(w))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["unknown, unknown"])[0].split(", ")
    return {"gpu": name, "power_limit": power}


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
        a, b = enc(int(rng.integers(0, 1 << w)), w), enc(int(rng.integers(0, 1 << w)), w)
        sel, amount = enc(1, 1)[0], enc(3, w)
        for name, call in instructions(w):
            cache = InstructionCache(ev)
            t0 = time.perf_counter()
            g = call(cache, a, b, sel, amount)
            first = time.perf_counter() - t0
            for _ in range(args.warmup):
                call(cache, a, b, sel, amount)
            ts = []
            for _ in range(args.runs):
                t0 = time.perf_counter()
                call(cache, a, b, sel, amount)
                ts.append(1e3 * (time.perf_counter() - t0))
            assert cache.misses == 1
            ts = np.asarray(ts)
            row = {"instruction": name, "width": w, "median_ms": round(float(np.median(ts)), 3),
                   "p10_ms": round(float(np.percentile(ts, 10)), 3), "p90_ms": round(float(np.percentile(ts, 90)), 3),
                   "min_ms": round(float(ts.min()), 3), "max_ms": round(float(ts.max()), 3), "runs": len(ts),
                   "first_call_ms": round(1e3 * first, 1), "levels": g.levels, "launches": g.launches,
                   "bootstraps": int((g._keep.ops == spf_b200.OP["CircuitBootstrap"]).sum())}
            rows.append(row)
            print(json.dumps(row), flush=True)
            g.close()
    doc = {**gpu_info(), "device": "cuda:0", "timing": "host clock around the blocking InstructionCache call",
           "warmup": args.warmup, "results": rows}
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    ev.close()


if __name__ == "__main__":
    main()
