"""Box ciphertext handles (spf_b200_box_ciphertext_*, spf_b200.BoxCiphertext): box graphs that hand their outputs to
the next graph in HBM, one replica per rank.  Every result is compared with the same graphs run through host buffers.
The one-GPU tests put two ranks on cuda:0 (devices [0, 0]); the multi-device tests use every visible GPU and skip below
two."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W = 8
VALS = [(100, 200, 43), (77, 30, 200)]  # (a, b, c): (a + b) mod 2^W > c is 1 for the first program, 0 for the second


def _n_devices():
    import torch

    return torch.cuda.device_count()


def _box(keys, devices):
    import spf_b200

    return spf_b200.BoxEvaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft, devices=devices)


@pytest.fixture(scope="module")
def box2(keys):
    b = _box(keys, [0, 0])
    yield b
    b.close()


@pytest.fixture(scope="module")
def box1(keys):
    b = _box(keys, [0])
    yield b
    b.close()


@pytest.fixture(scope="module")
def box_all(keys):
    n = _n_devices()
    if n < 2:
        pytest.skip("fewer than two GPUs visible")
    b = _box(keys, list(range(n)))
    yield b
    b.close()


def _enc(client, v, w=W):
    return [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]


def _dec(client, cts):
    return sum(int(client.decrypt_glwe_l1(np.asarray(x))[0]) << i for i, x in enumerate(cts))


def _add_graph(a, b, sums, echo):
    """Instruction 1 of every program: sums[p] = a[p] + b[p] (W bits); echo = program 0's a bit 0, passed through."""
    from spf_b200 import FheCircuit
    from spf_b200.circuits import _adder_nodes, _front

    c = FheCircuit()
    for p in range(len(a)):
        s = _adder_nodes(c, [_front(c, x) for x in a[p]], [_front(c, x) for x in b[p]])[:W]
        for i in range(W):
            c.add("OutputGlwe1", s[i], io=sums[p][i])
    c.add("OutputGlwe1", c.add("InputGlwe1", io=a[0][0]), io=echo)
    return c


def _gt_graph(sums, cc, gts):
    """Instruction 2 of every program: gts[p] = sums[p] > cc[p]."""
    from spf_b200 import FheCircuit
    from spf_b200.circuits import _front, _greater_than_node

    c = FheCircuit()
    for p in range(len(sums)):
        ss, sc = [_front(c, x) for x in sums[p]], [_front(c, x) for x in cc[p]]
        c.add("OutputGlwe1", _greater_than_node(c, ss, sc), io=gts[p])
    return c


def _chain(box, inputs, mode, spawned):
    """The two-instruction programs with the W sum bits handed over through `mode` ("host" or "handle")."""
    import spf_b200

    a, b, cc = inputs
    if mode == "host":
        slab = spf_b200.pinned_zeros((len(VALS) * W + 1, 4096))
        sums = [[slab[p * W + i] for i in range(W)] for p in range(len(VALS))]
        echo = slab[len(VALS) * W]
    else:
        sums = [[spf_b200.BoxCiphertext.alloc(box, "Glwe1") for _ in range(W)] for _ in VALS]
        echo = spf_b200.BoxCiphertext.alloc(box, "Glwe1")
    gts = [np.zeros(4096, np.uint64) for _ in VALS]
    ga = spf_b200.BoxGraph(box, _add_graph(a, b, sums, echo))
    gb = spf_b200.BoxGraph(box, _gt_graph(sums, cc, gts))
    if spawned:
        order = []
        ga.spawn(on_complete=lambda e: order.append(("add", e)))
        gb.spawn(after=[ga], on_complete=lambda e: order.append(("gt", e)))
        gb.wait()
        ga.wait()
        assert order == [("add", None), ("gt", None)]
    else:
        ga.run()
        gb.run()
    ga.close(); gb.close()
    return sums, echo, gts


def _check_chain(client, box):
    inputs = [[_enc(client, v[k]) for v in VALS] for k in range(3)]
    ref_sums, ref_echo, ref_gts = _chain(box, inputs, "host", spawned=False)
    want_s = [(a + b) % (1 << W) for a, b, _ in VALS]
    want_g = [int(s > c) for s, (_, _, c) in zip(want_s, VALS)]
    assert [_dec(client, s) for s in ref_sums] == want_s
    assert [int(client.decrypt_glwe_l1(g)[0]) for g in ref_gts] == want_g
    for mode, spawned in (("host", True), ("handle", False), ("handle", True)):
        sums, echo, gts = _chain(box, inputs, mode, spawned)
        assert [g.tobytes() for g in gts] == [g.tobytes() for g in ref_gts], (mode, spawned)
        if mode == "host":
            assert [[x.tobytes() for x in s] for s in sums] == [[x.tobytes() for x in s] for s in ref_sums]
            continue
        for r in range(box.size):  # owned (the sum bits) and replicated (echo) values reach every rank's replica
            for p in range(len(VALS)):
                assert [x.read(r).tobytes() for x in sums[p]] == [x.tobytes() for x in ref_sums[p]], (spawned, r, p)
            assert echo.read(r).tobytes() == inputs[0][0][0].tobytes() == ref_echo.tobytes(), (spawned, r)
        assert [_dec(client, [x.read() for x in s]) for s in sums] == want_s
        for h in [x for s in sums for x in s] + [echo]:
            h.close()


def _check_sum_trees_on_every_rank(box):
    """Both programs' adders are owned by different ranks, so owners push replicas to their peers."""
    import spf_b200

    c = _add_graph([[np.zeros(4096, np.uint64)] * W] * 2, [[np.zeros(4096, np.uint64)] * W] * 2,
                   [[np.zeros(4096, np.uint64)] * W] * 2, np.zeros(4096, np.uint64))
    _, owner = spf_b200.plan_graph(c, world=box.size)
    outs = [i for i, n in enumerate(c.nodes) if n[0] == spf_b200.OP["OutputGlwe1"]][:-1]
    assert {int(owner[c.nodes[i][2][0]]) for i in outs} == set(range(min(box.size, 2)))


def test_chain_through_handles_matches_host_buffers(client, box2):
    _check_sum_trees_on_every_rank(box2)
    _check_chain(client, box2)


def test_single_rank_box_chain(client, box1):
    _check_chain(client, box1)


def test_multi_device_chain(client, box_all):
    _check_sum_trees_on_every_rank(box_all)
    _check_chain(client, box_all)


def _ggsw_pair(box, cts, sel_io):
    """CircuitBootstrap -> OutputGgsw1 (sel_io), then a second graph CMux(sel, 0, 1) from InputGgsw1 (sel_io)."""
    import spf_b200
    from spf_b200 import FheCircuit
    from spf_b200.circuits import _front

    ca, cb = FheCircuit(), FheCircuit()
    for ct, sel in zip(cts, sel_io):
        ca.add("OutputGgsw1", _front(ca, ct), io=sel)
    zero, one = cb.add("ZeroGlwe1"), cb.add("OneGlwe1")
    outs = [np.zeros(4096, np.uint64) for _ in cts]
    for k in range(len(cts)):
        cb.add("OutputGlwe1", cb.add("CMux", cb.add("InputGgsw1", io=sel_io[k]), zero, one), io=outs[k])
    for c in (ca, cb):
        g = spf_b200.BoxGraph(box, c)
        g.run()
        g.close()
    return outs


def test_ggsw_handle_feeds_a_cmux_selector(client, box2):
    import spf_b200

    bits = [1, 0, 1]
    n = spf_b200.io_bytes("Ggsw1") // 16
    cts = [client.encrypt_glwe_l1([b]) for b in bits]
    host = [np.zeros(n, np.complex128) for _ in bits]
    ref = _ggsw_pair(box2, cts, host)
    handles = [spf_b200.BoxCiphertext.alloc(box2, "Ggsw1") for _ in bits]
    got = _ggsw_pair(box2, cts, handles)
    assert [x.tobytes() for x in got] == [x.tobytes() for x in ref]
    assert [int(client.decrypt_glwe_l1(x)[0]) for x in got] == bits
    for h, want in zip(handles, host):
        for r in range(box2.size):
            assert h.read(r).tobytes() == want.tobytes(), r  # the reference scale, as the host output
    # write() takes the reference scale and read() gives it back
    again = spf_b200.BoxCiphertext.alloc(box2, "Ggsw1")
    again.write(host[0])
    assert again.read(1).tobytes() == host[0].tobytes()


def _not_graph(ins, outs):
    from spf_b200 import FheCircuit

    c = FheCircuit()
    for x, y in zip(ins, outs):
        c.add("OutputGlwe1", c.add("Not", c.add("InputGlwe1", io=x)), io=y)
    return c


def _check_in_place(client, box):
    import spf_b200

    bits = [1, 0]  # two Not trees: one per rank on a two-rank box
    host = [client.encrypt_glwe_l1([b]) for b in bits]
    hs = [spf_b200.BoxCiphertext.alloc(box, "Glwe1") for _ in bits]
    for h, x in zip(hs, host):
        h.write(x)
    g = spf_b200.BoxGraph(box, _not_graph(hs, hs))
    host_out = [np.zeros(4096, np.uint64) for _ in bits]
    gh = spf_b200.BoxGraph(box, _not_graph(host, host_out))
    for k in range(3):
        g.run()
        gh.run()
        for x, y in zip(host, host_out):
            x[:] = y
        for r in range(box.size):
            assert [h.read(r).tobytes() for h in hs] == [x.tobytes() for x in host], (k, r)
        assert [int(client.decrypt_glwe_l1(h.read())[0]) for h in hs] == [b ^ ((k + 1) & 1) for b in bits]
    g.close(); gh.close()


def test_in_place_handle_without_bootstrap(client, box2):
    _check_in_place(client, box2)


def test_multi_device_in_place(client, box_all):
    _check_in_place(client, box_all)


def test_spawned_chain_under_flow_control(client, box2):
    import spf_b200

    hs = [spf_b200.BoxCiphertext.alloc(box2, "Glwe1") for _ in range(4)]
    hs[0].write(client.encrypt_glwe_l1([1]))
    graphs = [spf_b200.BoxGraph(box2, _not_graph([hs[k]], [hs[k + 1]])) for k in range(3)]
    order = []
    box2.set_max_in_flight(1)
    try:
        for k, g in enumerate(graphs):
            g.spawn(after=graphs[k - 1:k], on_complete=lambda e, k=k: order.append((k, e)))
        graphs[-1].wait()
    finally:
        box2.set_max_in_flight(4)
    assert order == [(0, None), (1, None), (2, None)]
    assert [int(client.decrypt_glwe_l1(h.read(r))[0]) for h in hs[1:] for r in range(2)] == [0, 0, 1, 1, 0, 0]
    for g in graphs:
        g.close()


def test_set_io_rebinds_between_spawned_runs(client, box2):
    import spf_b200
    from spf_b200.circuits import InstructionCache

    x, y = (spf_b200.BoxCiphertext.alloc(box2, "Glwe1") for _ in range(2))
    ox, oy = (spf_b200.BoxCiphertext.alloc(box2, "Glwe1") for _ in range(2))
    x.write(client.encrypt_glwe_l1([1]))
    y.write(client.encrypt_glwe_l1([0]))
    g = spf_b200.BoxGraph(box2, _not_graph([x], [ox]))
    g.spawn()
    g.set_io(0, y)  # the run in flight keeps its own bindings
    g.set_io(2, oy)
    g.spawn()
    g.wait()
    assert [int(client.decrypt_glwe_l1(h.read(1))[0]) for h in (ox, oy)] == [0, 1]
    g.close()
    # InstructionCache on a box with handle operands: one graph, rebound per call
    cache = InstructionCache(box2)
    w = 4
    for a, b in ((5, 9), (15, 15)):
        ha, hb = ([spf_b200.BoxCiphertext.alloc(box2, "Glwe1") for _ in range(w)] for _ in range(2))
        out = [spf_b200.BoxCiphertext.alloc(box2, "Glwe1") for _ in range(w + 1)]
        for hs, v in ((ha, a), (hb, b)):
            for h, ct in zip(hs, _enc(client, v, w)):
                h.write(ct)
        cache.add(ha, hb, out)
        assert _dec(client, [o.read(1) for o in out]) == a + b
    assert (cache.hits, cache.misses) == (1, 1)


def test_handle_errors_leave_the_graph_usable(client, evaluation, keys, box2):
    import torch

    import spf_b200
    from spf_b200 import DeviceCiphertext

    other = _box(keys, [0])
    foreign = spf_b200.BoxCiphertext.alloc(other, "Glwe1")
    x, out = spf_b200.BoxCiphertext.alloc(box2, "Glwe1"), spf_b200.BoxCiphertext.alloc(box2, "Glwe1")
    x.write(client.encrypt_glwe_l1([0]))
    with pytest.raises(spf_b200.SpfError) as e:
        spf_b200.BoxGraph(box2, _not_graph([foreign], [out]))
    assert e.value.code == -1 and "another box" in str(e.value)
    g = spf_b200.BoxGraph(box2, _not_graph([x], [out]))
    lwe0 = spf_b200.BoxCiphertext.alloc(box2, "Lwe0")
    dev = DeviceCiphertext(torch.zeros(keys.glwe_len, dtype=torch.int64, device="cuda:0"))  # a raw device pointer
    with pytest.raises(spf_b200.SpfError) as e:
        g.set_io(0, foreign)
    assert e.value.code == -1 and "another box" in str(e.value)
    rc = spf_b200.lib().spf_b200_box_graph_set_io(g._h, 0, lwe0.ptr)  # past the Python kind check
    assert rc == -1 and b"kind mismatch" in spf_b200.lib().spf_b200_box_last_error(box2.handle)
    with pytest.raises(spf_b200.SpfError) as e:
        g.set_io(0, dev)
    assert e.value.code == -1 and "device-memory" in str(e.value) and "box ciphertext handle" in str(e.value)
    g.run()
    assert int(client.decrypt_glwe_l1(out.read(1))[0]) == 1
    # single-context graphs refuse handles
    with pytest.raises(spf_b200.SpfError) as e:
        spf_b200.CompiledGraph(evaluation, _not_graph([x], [np.zeros(4096, np.uint64)]))
    assert e.value.code == -1 and "box graphs only" in str(e.value)
    # a dependency's failure still propagates through `after`
    bad = spf_b200.BoxGraph(other, _not_graph([foreign], [spf_b200.BoxCiphertext.alloc(other, "Glwe1")]))
    errs, dep_errs = [], []
    g.spawn(after=[bad], on_complete=errs.append)
    g2 = spf_b200.BoxGraph(box2, _not_graph([out], [x]))
    g2.spawn(after=[g], on_complete=dep_errs.append)
    with pytest.raises(spf_b200.SpfError):
        g2.wait()
    assert len(errs) == 1 and "another box" in str(errs[0])
    assert len(dep_errs) == 1 and "dependency" in str(dep_errs[0])
    for q in (g, g2, bad):
        q.close()
    other.close()


def test_closed_handle_lives_while_a_graph_binds_it(client, box2):
    import spf_b200

    l = spf_b200.lib()
    x = spf_b200.BoxCiphertext.alloc(box2, "Glwe1")
    x.write(client.encrypt_glwe_l1([1]))
    out = np.zeros(4096, np.uint64)
    g = spf_b200.BoxGraph(box2, _not_graph([x], [out]))
    ptr = x.ptr
    x.close()
    with pytest.raises(spf_b200.SpfError, match="closed"):
        x.read()
    g.run()
    assert int(client.decrypt_glwe_l1(out)[0]) == 0
    buf = np.zeros(4096, np.uint64)
    assert l.spf_b200_box_ciphertext_read(ptr, 1, buf.ctypes.data) == 0  # still a live handle: the graph holds it
    g.close()
    assert l.spf_b200_box_ciphertext_read(ptr, 1, buf.ctypes.data) == -1  # gone with the graph's reference
