"""Blocking latency of table lookups (InstructionCache.lookup, select_n) on one GPU (cuda:0): the AES S-box (8 -> 8 bits),
a seeded 4 -> 4, 12 -> 1 and 16 -> 16-bit table, select_n over 16 encrypted 32-bit entries, and the 8-bit product x * y
read from a 16-bit table against InstructionCache.multiply on the same ciphertexts (the two forms alternated).  Per row:
warm-up calls, then the median and spread of --runs calls, each timed on the host around the blocking call; the graph's
circuit bootstraps, CMUX levels, levels, launches and the table bytes copied to the device per run (32 KiB per
polynomial); the result of the last timed call decrypted and checked.  The 16 -> 16 row also times, with CUDA events, a
host-to-device copy of the same number of bytes from one page-locked slab -- the table copy alone.  The card's name and
power limit are read in the same run.  One JSON document to --out.
usage: python tools/lookup_latency.py [--runs 20] [--warmup 2] [--out profiles/lookup_latency_n1.json]"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle as O  # input generation and decryption only
import spf_b200
from isa_latency import gpu_info
from plain_latency import timed
from spf_b200.circuits import InstructionCache


def aes_sbox() -> list[int]:
    """The AES S-box (FIPS-197 5.1.1): the inverse in GF(2^8) mod x^8 + x^4 + x^3 + x + 1, then the affine map."""
    def mul(a, b):
        p = 0
        while b:
            p, a, b = p ^ (a if b & 1 else 0), ((a << 1) ^ 0x11B) if a & 0x80 else a << 1, b >> 1
        return p

    inv = [0] + [next(b for b in range(1, 256) if mul(a, b) == 1) for a in range(1, 256)]
    rot = lambda x, i: ((x << i) | (x >> (8 - i))) & 0xFF
    return [inv[a] ^ rot(inv[a], 1) ^ rot(inv[a], 2) ^ rot(inv[a], 3) ^ rot(inv[a], 4) ^ 0x63 for a in range(256)]


def table_bytes(cache) -> int:
    """Bytes of the table polynomials the one graph of a cache copies per run: its InputGlwe1 nodes the cache does not
    rebind."""
    ((g, ins, _),) = cache._cache.values()
    keep = g._keep
    tables = [i for i in range(len(keep)) if keep.ops[i] == spf_b200.OP["InputGlwe1"] and i not in set(ins)]
    return sum(keep._io[i].nbytes for i in tables)


def h2d_copy_ms(nbytes: int, runs: int) -> dict:
    """CUDA-event time of one host-to-device copy of nbytes from a page-locked slab, median of `runs` after a warm-up."""
    import torch

    src = torch.from_numpy(spf_b200.pinned_zeros((nbytes // 8,)))
    dst = torch.empty(nbytes // 8, dtype=torch.uint64, device="cuda:0")
    dst.copy_(src)
    ts = []
    for _ in range(runs):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        dst.copy_(src, non_blocking=True)
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return {"bytes": nbytes, "median_ms": round(float(np.median(ts)), 3), "runs": runs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    keys = O.Keys()
    client = O.Client(keys)
    ev = spf_b200.Evaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft)
    rng = np.random.default_rng(2)
    enc = lambda v, w: [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]
    dec = lambda bufs: sum(int(client.decrypt_glwe_l1(b)[0]) << i for i, b in enumerate(bufs))
    out = lambda n: [np.zeros(4096, np.uint64) for _ in range(n)]

    def lookup_row(name, table, k, m):
        cache, x, o = InstructionCache(ev), int(rng.integers(0, 1 << k)), out(m)
        xs = enc(x, k)
        res = timed({"lookup": lambda: cache.lookup(table, xs, o)}, args.runs, args.warmup)["lookup"]
        res.update(table_bytes=table_bytes(cache), correct=dec(o) == int(table[x]))   # o: the last timed call's result
        return {"workload": name, "index_bits": k, "result_bits": m, **res}

    rows = []
    rows.append(lookup_row("aes_sbox_8_to_8", aes_sbox(), 8, 8))
    rows.append(lookup_row("table_4_to_4", rng.integers(0, 16, 16), 4, 4))
    rows.append(lookup_row("table_12_to_1", rng.integers(0, 2, 1 << 12), 12, 1))
    rows.append(lookup_row("table_16_to_16", rng.integers(0, 1 << 16, 1 << 16), 16, 16))
    rows[-1]["h2d_table_copy"] = h2d_copy_ms(rows[-1]["table_bytes"], args.runs)
    for r in rows:
        print(json.dumps(r), flush=True)

    # select_n over 16 encrypted 32-bit entries
    cache, vals = InstructionCache(ev), [int(v) for v in rng.integers(0, 1 << 32, 16, dtype=np.uint64)]
    entries, x, o = [enc(v, 32) for v in vals], int(rng.integers(0, 16)), out(32)
    xs = enc(x, 4)
    res = timed({"select_n": lambda: cache.select_n(entries, xs, o)}, args.runs, args.warmup)["select_n"]
    rows.append({"workload": "select_n_16_entries_32_bits", "index_bits": 4, "result_bits": 32, **res,
                 "correct": dec(o) == vals[x]})
    print(json.dumps(rows[-1]), flush=True)

    # x * y at 8 bits: one 16-bit lookup against the multiplier circuit
    i = np.arange(1 << 16)
    product = (i & 0xFF) * (i >> 8) & 0xFF
    x, y = (int(v) for v in rng.integers(0, 256, 2))
    a, b = enc(x, 8), enc(y, 8)
    lc, mc, lo, mo = InstructionCache(ev), InstructionCache(ev), out(8), out(8)
    res = timed({"lookup": lambda: lc.lookup(product, a + b, lo), "multiply": lambda: mc.multiply(a, b, mo)},
                args.runs, args.warmup)
    res["lookup"]["table_bytes"] = table_bytes(lc)
    rows.append({"workload": "mul_8_bit_as_16_bit_lookup", "index_bits": 16, "result_bits": 8, **res,
                 "correct": dec(lo) == dec(mo) == x * y & 0xFF})
    print(json.dumps(rows[-1]), flush=True)

    doc = {**gpu_info(), "device": "cuda:0",
           "timing": "host clock around the blocking InstructionCache call (lookup and multiply alternated)",
           "warmup": args.warmup, "results": rows}
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    ev.close()
    if not all(r["correct"] for r in rows):
        sys.exit("a lookup result decrypted wrong")


if __name__ == "__main__":
    main()
