"""Box graph placement (spf_b200_box_graph_build_on, BoxGraph(..., ranks=...)): a box graph on a chosen, ordered subset
of the box's ranks, whose handle outputs still reach the replica of every rank.  Results are compared with the same
graphs run through host buffers on the same placement, or with a single-context CompiledGraph.  The one-GPU tests put
two ranks on cuda:0 (devices [0, 0]); the multi-device tests put every visible GPU in the box and skip below two."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W = 8
VALS = [(100, 200, 43), (77, 30, 200)]  # (a, b, c): (a + b) mod 2^W > c is 1 for the first program, 0 for the second


def _box(keys, devices):
    import spf_b200

    return spf_b200.BoxEvaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft, devices=devices)


@pytest.fixture(scope="module")
def box2(keys):
    b = _box(keys, [0, 0])
    yield b
    b.close()


@pytest.fixture(scope="module")
def box_all(keys):
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("fewer than two GPUs visible")
    b = _box(keys, list(range(n)))
    yield b
    b.close()


def _enc(client, v, w=W):
    return [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]


def _dec(client, cts):
    return sum(int(client.decrypt_glwe_l1(np.asarray(x))[0]) << i for i, x in enumerate(cts))


def _inputs(client, vals=VALS):
    """[a, b, c]: [programs][W] encrypted bits of every operand."""
    return [[_enc(client, v[k]) for v in vals] for k in range(3)]


def _add_circuit(a, b, sums):
    """sums[p] = a[p] + b[p] (W bits) for every program p."""
    from spf_b200 import FheCircuit
    from spf_b200.circuits import _adder_nodes, _front

    c = FheCircuit()
    for p in range(len(a)):
        s = _adder_nodes(c, [_front(c, x) for x in a[p]], [_front(c, x) for x in b[p]])[:W]
        for i in range(W):
            c.add("OutputGlwe1", s[i], io=sums[p][i])
    return c


def _gt_circuit(sums, cc, gts):
    """gts[p] = sums[p] > cc[p] for every program p."""
    from spf_b200 import FheCircuit
    from spf_b200.circuits import _front, _greater_than_node

    c = FheCircuit()
    for p in range(len(sums)):
        ss, sc = [_front(c, x) for x in sums[p]], [_front(c, x) for x in cc[p]]
        c.add("OutputGlwe1", _greater_than_node(c, ss, sc), io=gts[p])
    return c


def _sums(box, n_programs, mode):
    import spf_b200

    if mode == "host":
        return [[np.zeros(4096, np.uint64) for _ in range(W)] for _ in range(n_programs)]
    return [[spf_b200.BoxCiphertext.alloc(box, "Glwe1") for _ in range(W)] for _ in range(n_programs)]


def _want(vals=VALS):
    s = [(a + b) % (1 << W) for a, b, _ in vals]
    return s, [int(x > c) for x, (_, _, c) in zip(s, vals)]


def _launches(ctx):
    import spf_b200

    return int(spf_b200.lib().spf_b200_kernel_launches(ctx))


def test_placed_on_rank_1_matches_a_single_context(client, evaluation, box2):
    import spf_b200

    a, b, _ = _inputs(client)
    placed_sums, single_sums = _sums(box2, len(VALS), "host"), _sums(box2, len(VALS), "host")
    l0 = _launches(box2.contexts[0])
    g = spf_b200.BoxGraph(box2, _add_circuit(a, b, placed_sums), ranks=[1])
    assert g.ranks == [1]
    g.run()
    g.spawn()
    g.wait()
    assert _launches(box2.contexts[0]) == l0  # rank 0 took no part
    ref = spf_b200.CompiledGraph(evaluation, _add_circuit(a, b, single_sums))
    ref.run()
    assert [[x.tobytes() for x in s] for s in placed_sums] == [[x.tobytes() for x in s] for s in single_sums]
    assert [_dec(client, s) for s in placed_sums] == _want()[0]
    g.close(); ref.close()


def _handoff(box, inputs, producer, consumer, mode):
    """Sums on `producer`, then greater-than on `consumer`, the sums handed over through `mode` ("host" or "handle"),
    spawned with the consumer after the producer."""
    import spf_b200

    a, b, cc = inputs
    sums = _sums(box, len(a), mode)
    gts = [np.zeros(4096, np.uint64) for _ in a]
    ga = spf_b200.BoxGraph(box, _add_circuit(a, b, sums), ranks=producer)
    gb = spf_b200.BoxGraph(box, _gt_circuit(sums, cc, gts), ranks=consumer)
    fired = []
    ga.spawn(on_complete=lambda e: fired.append(("add", e)))
    gb.spawn(after=[ga], on_complete=lambda e: fired.append(("gt", e)))
    gb.wait()
    ga.wait()
    assert fired == [("add", None), ("gt", None)]
    ga.close(); gb.close()
    return sums, gts


def _check_handoff(client, box, producer, consumer):
    inputs = _inputs(client)
    ref_sums, ref_gts = _handoff(box, inputs, producer, consumer, "host")
    sums, gts = _handoff(box, inputs, producer, consumer, "handle")
    want_s, want_g = _want()
    assert [_dec(client, s) for s in ref_sums] == want_s
    assert [int(client.decrypt_glwe_l1(g)[0]) for g in ref_gts] == want_g
    assert [g.tobytes() for g in gts] == [g.tobytes() for g in ref_gts], (producer, consumer)
    for r in range(box.size):  # also the ranks that did not run the producer
        for p in range(len(VALS)):
            assert [x.read(r).tobytes() for x in sums[p]] == [x.tobytes() for x in ref_sums[p]], (producer, consumer, r, p)
    for h in [x for s in sums for x in s]:
        h.close()


def test_handoff_between_ranks(client, box2):
    _check_handoff(client, box2, [0], [1])
    _check_handoff(client, box2, [1], [0])


def test_mixed_placement(client, box2):
    import spf_b200

    a, b, cc = _inputs(client)
    want_s, want_g = _want()

    def fan_in(mode):
        """Program p's sums on rank p alone, both programs' comparisons in one graph over the whole box."""
        sums = _sums(box2, len(VALS), mode)
        gts = [np.zeros(4096, np.uint64) for _ in VALS]
        prod = [spf_b200.BoxGraph(box2, _add_circuit([a[p]], [b[p]], [sums[p]]), ranks=[p]) for p in range(len(VALS))]
        cons = spf_b200.BoxGraph(box2, _gt_circuit(sums, cc, gts))
        assert cons.ranks == [0, 1]
        for g in prod:
            g.spawn()
        cons.spawn(after=prod)
        cons.wait()
        for g in prod + [cons]:
            g.wait()
            g.close()
        return sums, gts

    ref_sums, ref_gts = fan_in("host")
    sums, gts = fan_in("handle")
    assert [int(client.decrypt_glwe_l1(g)[0]) for g in ref_gts] == want_g
    assert [g.tobytes() for g in gts] == [g.tobytes() for g in ref_gts]
    assert [[x.read(r).tobytes() for x in s] for s in sums for r in range(2)] == \
        [[x.tobytes() for x in s] for s in ref_sums for _ in range(2)]

    # an all-rank producer feeds a consumer placed on rank 1
    sums = _sums(box2, len(VALS), "handle")
    gts = [np.zeros(4096, np.uint64) for _ in VALS]
    ga = spf_b200.BoxGraph(box2, _add_circuit(a, b, sums))
    gb = spf_b200.BoxGraph(box2, _gt_circuit(sums, cc, gts), ranks=[1])
    ga.spawn()
    gb.spawn(after=[ga])
    gb.wait()
    assert [int(client.decrypt_glwe_l1(g)[0]) for g in gts] == want_g
    assert [_dec(client, [x.read(r) for x in s]) for s in sums for r in range(2)] == [v for v in want_s for _ in range(2)]
    ga.close(); gb.close()

    # members in the order given: member 0 runs on rank 1, member 1 on rank 0 -- the same shards as over [0, 1]
    host = _sums(box2, len(VALS), "host")
    handles = _sums(box2, len(VALS), "handle")
    ref = spf_b200.BoxGraph(box2, _add_circuit(a, b, host))
    rev = spf_b200.BoxGraph(box2, _add_circuit(a, b, handles), ranks=[1, 0])
    assert rev.ranks == [1, 0] and rev.levels == ref.levels
    ref.run()
    rev.run()
    for r in range(2):
        assert [[x.read(r).tobytes() for x in s] for s in handles] == [[x.tobytes() for x in s] for s in host], r
    assert [_dec(client, s) for s in host] == want_s
    ref.close(); rev.close()


def _check_concurrent(client, box, k):
    """k independent programs, program i placed on rank i mod N, all spawned before any wait."""
    import spf_b200
    from spf_b200.circuits import _front, _greater_than_node

    rng = np.random.default_rng(0x9A7)
    vals = [tuple(int(x) for x in rng.integers(0, 1 << W, 3)) for _ in range(k)]
    a, b, cc = _inputs(client, vals)
    sums = _sums(box, k, "handle")
    gts = [np.zeros(4096, np.uint64) for _ in range(k)]
    graphs = []
    for i in range(k):
        c = _add_circuit([a[i]], [b[i]], [sums[i]])
        c.add("OutputGlwe1", _greater_than_node(c, [_front(c, x) for x in a[i]], [_front(c, x) for x in cc[i]]), io=gts[i])
        graphs.append(spf_b200.BoxGraph(box, c, ranks=[i % box.size]))
    fired = {i: [] for i in range(k)}
    box.set_max_in_flight(k)
    try:
        for i, g in enumerate(graphs):
            g.spawn(on_complete=lambda e, i=i: fired[i].append(e))
        for g in graphs:
            g.wait()
    finally:
        box.set_max_in_flight(4)
    assert fired == {i: [None] for i in range(k)}
    want_s, _ = _want(vals)
    for i in range(k):
        for r in range(box.size):
            assert _dec(client, [x.read(r) for x in sums[i]]) == want_s[i], (i, r)
        assert int(client.decrypt_glwe_l1(gts[i])[0]) == int(vals[i][0] > vals[i][2]), i
    for g in graphs:
        g.close()


def test_concurrent_independent_graphs(client, box2):
    _check_concurrent(client, box2, 6)


def test_failed_dependency_of_a_placed_graph(keys, client, box2):
    """A placed run whose dependency failed retires as a no-op with the dependency's error; a one-member graph is not
    poisoned by a failed run."""
    import spf_b200
    from spf_b200 import FheCircuit

    other = _box(keys, [0])
    graphs, outs = [], []
    for ev, ranks in ((other, None), (box2, [1]), (box2, [0])):
        c = FheCircuit()
        outs.append(np.zeros(keys.glwe_len, dtype=np.uint64))
        c.add("OutputGlwe1", c.add("Not", c.add("InputGlwe1", io=client.encrypt_glwe_l1([1]))), io=outs[-1])
        graphs.append(spf_b200.CircuitProcessor(ev).compile(c, ranks=ranks))
    foreign, bad, dependent = graphs
    errs, dep_errs = [], []
    bad.spawn(after=[foreign], on_complete=errs.append)
    dependent.spawn(after=[bad], on_complete=dep_errs.append)
    with pytest.raises(spf_b200.SpfError):
        bad.wait()
    with pytest.raises(spf_b200.SpfError) as e:
        dependent.wait()
    assert "dependency" in str(e.value)
    assert len(errs) == 1 and isinstance(errs[0], spf_b200.SpfError) and "another box" in str(errs[0])
    assert len(dep_errs) == 1 and isinstance(dep_errs[0], spf_b200.SpfError) and "dependency" in str(dep_errs[0])
    assert not outs[1].any() and not outs[2].any()  # no-ops: nothing was written
    bad.run()
    dependent.spawn(after=[bad])
    dependent.wait()
    assert [int(client.decrypt_glwe_l1(o)[0]) for o in outs[1:]] == [0, 0]
    for g in graphs:
        g.close()
    other.close()


def test_argument_errors_leave_the_box_usable(client, evaluation, box2):
    import spf_b200

    l = spf_b200.lib()
    x = client.encrypt_glwe_l1([1])
    out = np.zeros(4096, np.uint64)

    def circuit():
        from spf_b200 import FheCircuit

        c = FheCircuit()
        c.add("OutputGlwe1", c.add("Not", c.add("InputGlwe1", io=x)), io=out)
        return c

    c = circuit()
    cases = [((), 0, "n_ranks"), ((0, 1, 0), 3, "n_ranks"), ((2,), 1, "not a rank"), ((-1,), 1, "not a rank"),
             ((1, 1), 2, "twice"), (None, 1, "NULL")]
    for ranks, n, msg in cases:
        g = C.c_void_p(0x1234)
        arr = None if ranks is None else (C.c_int * max(len(ranks), 1))(*ranks)
        rc = l.spf_b200_box_graph_build_on(box2.handle, c._pack(), len(c.nodes), arr, n, C.byref(g))
        err = (l.spf_b200_box_last_error(box2.handle) or b"").decode()
        assert rc == -1 and g.value is None and msg in err, (ranks, n, rc, err)
    for ranks in ([], [2], [1, 1]):
        with pytest.raises(spf_b200.SpfError) as e:
            spf_b200.BoxGraph(box2, c, ranks=ranks)
        assert e.value.code == -1
    with pytest.raises(spf_b200.SpfError) as e:
        spf_b200.CircuitProcessor(evaluation).compile(c, ranks=[0])
    assert e.value.code == -1
    g = spf_b200.CircuitProcessor(box2).compile(circuit(), ranks=[1])
    g.run()
    assert int(client.decrypt_glwe_l1(out)[0]) == 0
    g.close()


def test_multi_device_handoff(client, box_all):
    n = box_all.size
    _check_handoff(client, box_all, [0], [1])
    _check_handoff(client, box_all, [1], [0])
    _check_handoff(client, box_all, [n - 1], list(range(n)))


def test_multi_device_concurrent(client, box_all):
    _check_concurrent(client, box_all, 2 * box_all.size)
