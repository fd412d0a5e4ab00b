"""One process over the GPUs of a box (spf_b200.BoxEvaluation): key replication, device-resident and end-to-end circuit
bootstrapping, and N x (mul32 then greater-than) in one box graph, blocking and spawned.  Prints one JSON line and
records it under profiles/ (--out).  The same measurements as bench.py's multi-process line, so the two compare.
--chain measures instead a two-instruction program run as two box graphs (mul32, then greater-than on the product),
with the 32 product bits handed over through host buffers or through box ciphertext handles.
--placed K measures K independent mul32-then-greater-than programs spawned as K box graphs, the way a Parasol
processor issues instructions: every graph over all ranks, against program i placed on rank i mod N.

usage: python tools/box_bench.py [--devices 0,1,...] [--batch 4096] [--steps 10] [--out profiles/box_bench_n8.json]
       python tools/box_bench.py --chain [--devices 0,0] [--reps 20] [--out profiles/box_chain_n1.json]
       python tools/box_bench.py --placed 8 [--devices 0,0] [--reps 10] [--out profiles/box_place_n1.json]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_identity(devices):
    """Name and power limit of every GPU of the box, read by the same process that measures."""
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=60)
    rows = {}
    for line in q.stdout.strip().splitlines():
        idx, name, limit = [x.strip() for x in line.split(",")]
        rows[int(idx)] = {"name": name, "power_limit": limit}
    return [rows.get(d, {"name": None, "power_limit": None}) for d in sorted(set(devices))]


def encrypt_lwe0(sk, bits, std, seed):
    """b = <a,s> + m + e, vectorised (client-side input generation only)."""
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 1 << 64, (len(bits), sk.shape[0]), dtype=np.uint64)
    e = np.round(rng.normal(0.0, std, len(bits)) * 2.0 ** 64).astype(np.int64).astype(np.uint64)
    b = (a * sk[None, :]).sum(axis=1, dtype=np.uint64) + (bits.astype(np.uint64) << np.uint64(63)) + e
    return np.ascontiguousarray(np.concatenate([a, b[:, None]], axis=1))


def device_resident(box, cts, batch, steps, warmup):
    """batch CBS per rank per step from device memory through each rank's context, every rank enqueued from this
    thread; CUDA events per device; a step's time is the slowest rank's."""
    import torch

    import spf_b200

    l = spf_b200.lib()
    ranks = []
    for r, (dev, ctx) in enumerate(zip(box.devices, box.contexts)):
        d = torch.device("cuda", dev)
        with torch.cuda.device(d):
            s = torch.cuda.Stream(device=d)
            d_in = torch.from_numpy(cts[r * batch:(r + 1) * batch].view(np.int64)).to(d)
            d_out = torch.empty(batch * box.len_ggsw * 2, dtype=torch.float64, device=d)
            flush = torch.empty(256 << 20, dtype=torch.uint8, device=d)
        ranks.append((d, ctx, s, d_in, d_out, flush))

    def step(events=None):
        for r, (d, ctx, s, d_in, d_out, flush) in enumerate(ranks):
            with torch.cuda.device(d), torch.cuda.stream(s):
                flush.zero_()
                if events:
                    events[r][0].record(s)
                rc = l.spf_b200_dev_circuit_bootstrap(ctx, d_out.data_ptr(), d_in.data_ptr(), batch, 0, s.cuda_stream)
                if rc:
                    raise spf_b200.SpfError(rc, (l.spf_b200_last_error(ctx) or b"").decode())
                if events:
                    events[r][1].record(s)

    for _ in range(max(warmup, 2)):
        step()
    for d, *_ in ranks:
        torch.cuda.synchronize(d)
    per_step = []
    for _ in range(steps):
        ev = []
        for d, *_ in ranks:
            with torch.cuda.device(d):
                ev.append((torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)))
        step(ev)
        for d, *_ in ranks:
            torch.cuda.synchronize(d)
        per_step.append(max(a.elapsed_time(b) for a, b in ev))
    ms = float(np.median(per_step))
    return {"ms_per_step": ms, "cbs_per_s": len(ranks) * batch / (ms * 1e-3)}


def end_to_end(box, cts, steps, warmup):
    """spf_b200_box_circuit_bootstrap from and to page-locked host buffers: host wall clock per call."""
    import spf_b200

    h_in = spf_b200.pinned_zeros(cts.shape)
    h_in[:] = cts
    h_out = spf_b200.pinned_zeros((cts.shape[0], box.len_ggsw), dtype=np.complex128)
    l = spf_b200.lib()

    def call():
        box._check(l.spf_b200_box_circuit_bootstrap(box.handle, h_out.ctypes.data, h_in.ctypes.data, cts.shape[0]))

    for _ in range(max(warmup, 1)):
        call()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        call()
        ts.append(time.perf_counter() - t0)
    s = float(np.median(ts))
    return {"ms_per_call": 1e3 * s, "cbs_per_s": cts.shape[0] / s}, h_out


def programs(box, keys, n_programs, reps):
    """n_programs x (32-bit multiply, low word, then greater-than) in ONE box graph."""
    import oracle as O
    import spf_b200
    from spf_b200.circuits import multiply_then_greater_than

    client = O.Client(keys)
    w = 32
    rng = np.random.default_rng(0xB0C5)
    vals = [tuple(int(x) for x in rng.integers(0, 1 << w, 3)) for _ in range(n_programs)]
    slab = iter(spf_b200.pinned_zeros((n_programs * (3 * w + w + 1), keys.glwe_len)))

    def enc(v):
        out = [next(slab) for _ in range(w)]
        for i, r in enumerate(out):
            r[:] = client.encrypt_glwe_l1([(v >> i) & 1])
        return out

    a, b, c = ([enc(v[k]) for v in vals] for k in range(3))
    out_prod = [[next(slab) for _ in range(w)] for _ in vals]
    out_gt = [next(slab) for _ in vals]
    circ = multiply_then_greater_than(a, b, c, out_prod, out_gt, n_programs)
    g = spf_b200.CircuitProcessor(box).compile(circ)
    g.run()

    def correct():
        ok = True
        for (x, y, z), pb, gt in zip(vals, out_prod, out_gt):
            p = sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(pb))
            ok &= p == (x * y) % (1 << w) and int(client.decrypt_glwe_l1(gt)[0]) == int(p > z)
        return bool(ok)

    blocking = []
    for _ in range(reps):
        t0 = time.perf_counter()
        g.run()
        blocking.append(time.perf_counter() - t0)
    ok_blocking = correct()
    spawned = []
    for _ in range(reps):
        t0 = time.perf_counter()
        g.spawn()
        g.wait()
        spawned.append(time.perf_counter() - t0)
    res = {"programs": n_programs, "levels": g.levels, "launches": g.launches, "blocking_ms": 1e3 * float(np.median(blocking)),
           "spawned_ms": 1e3 * float(np.median(spawned)), "correct": ok_blocking and correct()}
    g.close()
    return res


def chain(box, keys, n_programs, reps, warmup):
    """n_programs x (mul32 | greater-than on the product) as TWO box graphs, the 32 product bits of every program handed
    from the first to the second through page-locked host buffers ("host") or box ciphertext handles ("handle"), each
    run blocking (run, run) and spawned (spawn, spawn after the first, wait).  Times are host clocks around the whole
    program pair up to the end of the second graph (median over reps, rounds of the four ways interleaved); enqueue_ms
    is the host time of the two spawn calls.  PCIe bytes per run follow from the shapes: every rank copies every host
    input, the owner of a product bit copies it out, and the host-buffer hand-off is read back by every rank."""
    import oracle as O
    import spf_b200
    from spf_b200 import FheCircuit
    from spf_b200 import mux_circuits as M
    from spf_b200.circuits import _front

    client = O.Client(keys)
    w = 32
    rng = np.random.default_rng(0xB0C6)
    vals = [tuple(int(x) for x in rng.integers(0, 1 << w, 3)) for _ in range(n_programs)]
    slab = iter(spf_b200.pinned_zeros((n_programs * (3 * w + w + 1), keys.glwe_len)))

    def enc(v):
        out = [next(slab) for _ in range(w)]
        for i, r in enumerate(out):
            r[:] = client.encrypt_glwe_l1([(v >> i) & 1])
        return out

    a, b, c = ([enc(v[k]) for v in vals] for k in range(3))
    mid_host = [[next(slab) for _ in range(w)] for _ in vals]
    out_gt = [next(slab) for _ in vals]
    mid_handle = [[spf_b200.BoxCiphertext.alloc(box, "Glwe1") for _ in range(w)] for _ in vals]

    def graphs(mid):
        c1, c2 = FheCircuit(), FheCircuit()
        keep1, keep2 = [], []
        for p in range(n_programs):
            lo, _hi = M.append_uint_multiply(c1, [_front(c1, x) for x in a[p]], [_front(c1, x) for x in b[p]])
            keep1 += [c1.add("OutputGlwe1", lo[i], io=mid[p][i]) for i in range(w)]
            pairs = [x for pr in zip([_front(c2, x) for x in mid[p]], [_front(c2, x) for x in c[p]]) for x in pr]
            (gt,) = M.insert_mux_circuit(c2, M.compare_or_maybe_equal(w, True, False), pairs)
            keep2.append(c2.add("OutputGlwe1", gt, io=out_gt[p]))
        return spf_b200.BoxGraph(box, M.prune(c1, keep1)[0]), spf_b200.BoxGraph(box, M.prune(c2, keep2)[0])

    pairs = {"host": graphs(mid_host), "handle": graphs(mid_handle)}

    def correct(mode):
        ok = True
        for p, (x, y, z) in enumerate(vals):
            bits = [m if mode == "host" else m.read() for m in (mid_host if mode == "host" else mid_handle)[p]]
            prod = sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(bits))
            ok &= prod == (x * y) % (1 << w) and int(client.decrypt_glwe_l1(out_gt[p])[0]) == int(prod > z)
        return bool(ok)

    def once(mode, spawned):
        g1, g2 = pairs[mode]
        for o in out_gt:
            o[:] = 0
        t0 = time.perf_counter()
        if spawned:
            g1.spawn()
            g2.spawn(after=[g1])
            t_enq = time.perf_counter() - t0
            g2.wait()
            g1.wait()
        else:
            g1.run()
            g2.run()
            t_enq = None
        return time.perf_counter() - t0, t_enq

    ways = [(m, s) for m in ("host", "handle") for s in (False, True)]
    for _ in range(max(warmup, 2)):
        for m, s in ways:
            once(m, s)
    times = {k: [] for k in ways}
    enq = {k: [] for k in ways}
    ok = {m: True for m in pairs}
    for _ in range(reps):
        for m, s in ways:
            t, e = once(m, s)
            times[(m, s)].append(t)
            if e is not None:
                enq[(m, s)].append(e)
            ok[m] &= correct(m)
    glwe, n = keys.glwe_len * 8, box.size
    pcie_in = n * 3 * w * glwe * n_programs + 1 * glwe * n_programs  # operand inputs on every rank, the verdict out
    res = {"programs": n_programs, "ranks": n, "levels": [pairs["host"][0].levels, pairs["host"][1].levels],
           "launches_handle": [g.launches for g in pairs["handle"]], "launches_host": [g.launches for g in pairs["host"]]}
    for m in pairs:
        res[m] = {"pcie_bytes_per_run": pcie_in + (w * glwe + n * w * glwe) * n_programs * (m == "host"), "correct": ok[m]}
        for s in (False, True):
            key = "spawned" if s else "blocking"
            res[m][key + "_ms"] = 1e3 * float(np.median(times[(m, s)]))
            if s:
                res[m]["spawned_enqueue_ms"] = 1e3 * float(np.median(enq[(m, s)]))
    for g in [g for pr in pairs.values() for g in pr]:
        g.close()
    return res


def placed(box, keys, k, reps, warmup):
    """k independent programs (32-bit multiply, low word, then greater-than), one box graph each as programs() builds
    them, with max_in_flight = k: all k graphs spawned, then all k waited for.  Two modes, alternated round by round:
    "all_ranks" builds every graph over the whole box (spf_b200_box_graph_build), "placed" puts program i on rank
    i mod N alone (spf_b200_box_graph_build_on).  Times are host clocks around a batch of k, ending after the last
    wait (median over reps); every output of every timed batch is zeroed before and decrypted after it."""
    import oracle as O
    import spf_b200
    from spf_b200.circuits import multiply_then_greater_than

    client = O.Client(keys)
    w, n = 32, box.size
    rng = np.random.default_rng(0xB0C7)
    vals = [tuple(int(x) for x in rng.integers(0, 1 << w, 3)) for _ in range(k)]
    modes = ("all_ranks", "placed")
    slab = iter(spf_b200.pinned_zeros((k * 3 * w + len(modes) * k * (w + 1), keys.glwe_len)))

    def enc(v):
        out = [next(slab) for _ in range(w)]
        for i, r in enumerate(out):
            r[:] = client.encrypt_glwe_l1([(v >> i) & 1])
        return out

    a, b, c = ([enc(v[j]) for v in vals] for j in range(3))
    outs, graphs = {}, {}
    for m in modes:
        out_prod = [[next(slab) for _ in range(w)] for _ in vals]
        out_gt = [next(slab) for _ in vals]
        outs[m] = (out_prod, out_gt)
        graphs[m] = [spf_b200.BoxGraph(box, multiply_then_greater_than([a[i]], [b[i]], [c[i]], [out_prod[i]], [out_gt[i]], 1),
                                       ranks=None if m == "all_ranks" else [i % n]) for i in range(k)]

    def correct(m):
        ok = True
        out_prod, out_gt = outs[m]
        for (x, y, z), pb, gt in zip(vals, out_prod, out_gt):
            p = sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(pb))
            ok &= p == (x * y) % (1 << w) and int(client.decrypt_glwe_l1(gt)[0]) == int(p > z)
        return bool(ok)

    def batch(m):
        out_prod, out_gt = outs[m]
        for o in [x for pb in out_prod for x in pb] + out_gt:
            o[:] = 0
        fired = []
        t0 = time.perf_counter()
        for g in graphs[m]:
            g.spawn(on_complete=fired.append)
        for g in graphs[m]:
            g.wait()
        t = time.perf_counter() - t0
        return t, len(fired) == k and not any(fired) and correct(m)

    box.set_max_in_flight(k)
    for _ in range(max(warmup, 1)):
        for m in modes:
            batch(m)
    times = {m: [] for m in modes}
    ok = {m: True for m in modes}
    for _ in range(reps):
        for m in modes:
            t, good = batch(m)
            times[m].append(t)
            ok[m] &= good
    res = {"programs": k, "ranks": n, "levels": graphs["all_ranks"][0].levels,
           "placement": [g.ranks for g in graphs["placed"]]}
    for m in modes:
        res[m] = {"batch_ms": 1e3 * float(np.median(times[m])), "batch_ms_min": 1e3 * float(np.min(times[m])),
                  "batch_ms_max": 1e3 * float(np.max(times[m])), "launches": sum(g.launches for g in graphs[m]),
                  "correct": ok[m]}
    for g in [g for gs in graphs.values() for g in gs]:
        g.close()
    box.set_max_in_flight(4)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--devices", default=None, help="comma-separated device list (default: every visible GPU)")
    ap.add_argument("--batch", type=int, default=4096, help="CBS per GPU per step")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5, help="runs of the program graph per mode")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--chain", action="store_true", help="measure the two-graph mul32 | greater-than hand-off only")
    ap.add_argument("--programs", type=int, default=1, help="--chain: programs per graph")
    ap.add_argument("--placed", type=int, default=0, metavar="K",
                    help="measure K independent program graphs over all ranks against placed on rank i mod N")
    args = ap.parse_args()

    import torch

    import oracle as O
    import spf_b200

    if not torch.cuda.is_available():
        raise SystemExit("box_bench.py: no CUDA device; spf_b200 has no CPU fallback")
    devices = [int(x) for x in args.devices.split(",")] if args.devices else list(range(torch.cuda.device_count()))
    metric = "box_chain" if args.chain else "box_place" if args.placed else "box_bench"
    line = {"metric": metric, "devices": devices, "gpus": gpu_identity(devices)}
    keys = O.Keys()
    t0 = time.perf_counter()
    box = spf_b200.BoxEvaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft, devices=devices)
    line["box_create_ms"] = 1e3 * (time.perf_counter() - t0)
    line["key_replication_ms"] = box.key_replication_ms
    n = box.size
    if args.placed:
        line["placed"] = placed(box, keys, args.placed, args.reps, args.warmup)
        box.close()
        emit(line, args.out)
        return
    if args.chain:
        line["chain"] = chain(box, keys, args.programs, max(args.reps, 20), args.warmup)
        box.close()
        emit(line, args.out)
        return
    p = keys.params
    bits = np.random.default_rng(0xB0C4).integers(0, 2, n * args.batch)
    cts = encrypt_lwe0(keys.lwe0_sk.astype(np.uint64), bits, p.lwe_std, 0xB0C4)
    line["device_resident"] = {"batch_per_gpu": args.batch, **device_resident(box, cts, args.batch, args.steps, args.warmup)}
    e2e, h_out = end_to_end(box, cts, args.steps, args.warmup)
    client = O.Client(keys)
    idx = np.linspace(0, len(bits) - 1, 16).astype(int)
    e2e["correct"] = bool(all(client.decrypt_ggsw_l1(h_out[i]) == int(bits[i]) for i in idx))
    line["end_to_end"] = {"batch_per_gpu": args.batch, **e2e}
    line["mul32_then_gt"] = programs(box, keys, n, args.reps)
    box.close()
    emit(line, args.out)


def emit(line, out):
    text = json.dumps(line)
    print(text)
    if out:
        with open(out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
