"""One process over several ranks of a box (spf_b200_box_*): BoxEvaluation's batched ops, box graphs through the
blocking and the spawned path, dependencies, errors.  The one-GPU tests put two ranks on cuda:0 (devices [0, 0]); the
multi-device tests use every visible GPU and skip below two."""
import ctypes as C
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _n_devices():
    import torch

    return torch.cuda.device_count()


@pytest.fixture(scope="module")
def box2(keys):
    import spf_b200

    b = spf_b200.BoxEvaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft, devices=[0, 0])
    yield b
    b.close()


@pytest.fixture(scope="module")
def box_all(keys):
    import spf_b200

    n = _n_devices()
    if n < 2:
        pytest.skip("fewer than two GPUs visible")
    b = spf_b200.BoxEvaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft, devices=list(range(n)))
    yield b
    b.close()


def _multiply_program(client, keys, w, vals):
    from spf_b200.circuits import multiply_then_greater_than

    enc = lambda v: [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]
    a, b, c = ([enc(v[k]) for v in vals] for k in range(3))
    out_prod = [[np.zeros(keys.glwe_len, dtype=np.uint64) for _ in range(w)] for _ in vals]
    out_gt = [np.zeros(keys.glwe_len, dtype=np.uint64) for _ in vals]
    return multiply_then_greater_than(a, b, c, out_prod, out_gt, len(vals)), out_prod, out_gt


def _decrypt_multiply(client, out_prod, out_gt):
    prods = [sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(p)) for p in out_prod]
    return prods, [int(client.decrypt_glwe_l1(g)[0]) for g in out_gt]


def _check_key_replicas(box, keys):
    host = [np.ascontiguousarray(keys.bsk_fft).reshape(-1), np.ascontiguousarray(keys.ksk).reshape(-1),
            np.ascontiguousarray(keys.ssk_fft).reshape(-1), np.ascontiguousarray(keys.ak_fft).reshape(-1)]
    for r in range(box.size):
        for which, h in enumerate(host):
            for off in (0, h.size // 2, h.size - 4096):
                got = box.key_slice(r, which, off, 4096)
                assert got.tobytes() == h[off:off + 4096].tobytes(), (r, which, off)


def _check_cbs_against_slices(box, evaluation, client, bits):
    import spf_b200

    cts = client.encrypt_lwe_l0_batch(bits)
    got = box.circuit_bootstrap(cts)
    for r in range(box.size):
        s, k = spf_b200.box_shard(len(bits), box.size, r)
        assert np.array_equal(got[s:s + k], evaluation.circuit_bootstrap(cts[s:s + k])), r
    for g, bit in zip(got, bits):
        assert np.array_equal(client.ggsw_level_messages(g), client.ggsw_expected_messages(bit))


def test_box_reports_its_ranks_and_replicated_key(keys, box2):
    assert box2.size == 2 and box2.devices == [0, 0]
    ctxs = box2.contexts
    assert all(ctxs) and ctxs[0] != ctxs[1]
    assert box2.key_replication_ms > 0
    _check_key_replicas(box2, keys)


def test_box_cbs_bit_identical_to_single_context_slices(client, evaluation, box2):
    rng = np.random.default_rng(71)
    _check_cbs_against_slices(box2, evaluation, client, [int(x) for x in rng.integers(0, 2, 301)])


def test_box_pbs_and_keyswitch_bit_identical(oracle, keys, client, evaluation, box2):
    import spf_b200

    p = keys.params
    lut = oracle.generate_lut(p, [lambda x: (x + 3) % 8], 3)
    msgs = [m % 8 for m in range(37)]
    cts = np.zeros((len(msgs), keys.lwe0_len), dtype=np.uint64)
    for i, m in enumerate(msgs):
        oracle.lib().orc_encrypt_lwe(C.byref(client.rng), cts[i], keys.lwe0_sk, p.lwe_n, p.lwe_std, m << 60)
    out = box2.programmable_bootstrap(cts, lut)
    bits = [m & 1 for m in msgs]
    l1 = np.stack([client.encrypt_lwe_l1(b) for b in bits])
    l0 = box2.keyswitch_lwe_l1_lwe_l0(l1)
    for r in range(2):
        s, k = spf_b200.box_shard(len(msgs), 2, r)
        assert np.array_equal(out[s:s + k], evaluation.programmable_bootstrap(cts[s:s + k], lut))
        assert np.array_equal(l0[s:s + k], evaluation.keyswitch_lwe_l1_lwe_l0(l1[s:s + k]))
    for i, m in enumerate(msgs):
        assert int(oracle.decode(client.decrypt_glwe_l1_raw(out[i])[:1], 3)[0]) == (m + 3) % 8
    assert [client.decrypt_lwe_l0(x) for x in l0] == bits


def test_box_cmux_matches_single_context(client, evaluation, box2):
    bits = [1, 0, 0, 1, 1]
    sel = evaluation.circuit_bootstrap(client.encrypt_lwe_l0_batch(bits))
    a = np.stack([client.encrypt_glwe_l1([0])] * len(bits))
    b = np.stack([client.encrypt_glwe_l1([1])] * len(bits))
    got = box2.cmux(sel, a, b)
    assert np.array_equal(got, evaluation.cmux(sel, a, b))
    assert [int(client.decrypt_glwe_l1(x)[0]) for x in got] == bits


def _graph_check(keys, client, evaluation, box, spawn_too=True):
    import spf_b200

    w, vals = 8, [(13, 11, 100), (255, 255, 0)]
    circ, out_prod, out_gt = _multiply_program(client, keys, w, vals)
    want_p, want_g = [(a * b) % (1 << w) for a, b, _ in vals], [int((a * b) % (1 << w) > c) for a, b, c in vals]
    g = spf_b200.CircuitProcessor(box).compile(circ)
    assert isinstance(g, spf_b200.BoxGraph) and g.levels > 0
    g.run()
    assert _decrypt_multiply(client, out_prod, out_gt) == (want_p, want_g)
    assert g.launches > 0
    # the same program on one context (world = 1) decrypts to the same values
    circ1, out_prod1, out_gt1 = _multiply_program(client, keys, w, vals)
    g1 = spf_b200.CompiledGraph(evaluation, circ1)
    g1.run()
    assert _decrypt_multiply(client, out_prod1, out_gt1) == (want_p, want_g)
    g1.close()
    if spawn_too:
        for _ in range(2):  # a second run of the same box graph, spawned
            for x in [x for p in out_prod for x in p] + out_gt:
                x[:] = 0
            calls = []
            g.spawn(on_complete=calls.append)
            g.wait()
            assert calls == [None]
            assert _decrypt_multiply(client, out_prod, out_gt) == (want_p, want_g)
    g.close()


def test_box_graph_multiply_then_compare(keys, client, evaluation, box2):
    _graph_check(keys, client, evaluation, box2)


def _refresh_graph(c, src, out, invert):
    """InputGlwe1 -> SampleExtract -> KeyswitchL1toL0 -> CircuitBootstrap -> CMux(sel, 0, 1) [-> Not] -> OutputGlwe1"""
    from spf_b200.circuits import _front

    sels = [_front(c, x) for x in src]
    zero, one = c.add("ZeroGlwe1"), c.add("OneGlwe1")
    for s, o in zip(sels, out):
        x = c.add("CMux", s, zero, one)
        c.add("OutputGlwe1", c.add("Not", x) if invert else x, io=o)


def test_box_graphs_chained_with_after(keys, client, box2):
    """Graph B reads the host buffers graph A writes; `after=[A]` orders B behind A on every rank's stream.  The
    buffers between them are page-locked, so A's copies land before B's copies read them."""
    import spf_b200
    from spf_b200 import FheCircuit

    bits = [1, 0, 1, 1]
    mid = spf_b200.pinned_zeros((len(bits), keys.glwe_len))
    out = [np.zeros(keys.glwe_len, dtype=np.uint64) for _ in bits]
    ca, cb = FheCircuit(), FheCircuit()
    _refresh_graph(ca, [client.encrypt_glwe_l1([b]) for b in bits], list(mid), invert=False)
    _refresh_graph(cb, list(mid), out, invert=True)
    proc = spf_b200.CircuitProcessor(box2)
    order = []
    ga = proc.spawn_graph(ca, on_completion=lambda e: order.append(("a", e)))
    gb = proc.spawn_graph(cb, on_completion=lambda e: order.append(("b", e)), after=[ga])
    gb.wait()
    ga.wait()
    assert order == [("a", None), ("b", None)]
    assert [int(client.decrypt_glwe_l1(x)[0]) for x in mid] == bits
    assert [int(client.decrypt_glwe_l1(x)[0]) for x in out] == [1 - b for b in bits]
    ga.close(); gb.close()


def test_failed_dependency_is_reported(keys, client, box2):
    """A run that cannot start (its dependency belongs to another box) fails through its completion handler; a run
    spawned after it retires as a no-op with a dependency error."""
    import spf_b200
    from spf_b200 import FheCircuit

    other = spf_b200.BoxEvaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft, devices=[0])
    graphs, errs = [], []
    for ev in (other, box2, box2):
        c = FheCircuit()
        c.add("OutputGlwe1", c.add("Not", c.add("InputGlwe1", io=client.encrypt_glwe_l1([1]))),
              io=np.zeros(keys.glwe_len, dtype=np.uint64))
        graphs.append(spf_b200.CircuitProcessor(ev).compile(c))
    foreign, bad, dependent = graphs
    dep_errs = []
    bad.spawn(after=[foreign], on_complete=errs.append)
    dependent.spawn(after=[bad], on_complete=dep_errs.append)
    with pytest.raises(spf_b200.SpfError):
        bad.wait()
    with pytest.raises(spf_b200.SpfError) as e:
        dependent.wait()
    assert "dependency" in str(e.value)
    assert len(errs) == 1 and isinstance(errs[0], spf_b200.SpfError) and "another box" in str(errs[0])
    assert len(dep_errs) == 1 and isinstance(dep_errs[0], spf_b200.SpfError) and "dependency" in str(dep_errs[0])
    for g in graphs:
        g.close()
    other.close()


def test_box_graph_errors(keys, client, evaluation, box2):
    import spf_b200
    from spf_b200 import DeviceCiphertext, FheCircuit

    bad = FheCircuit()
    bad.add("SampleExtract", bad.add("ZeroLwe0"), arg=1)  # wrong ciphertext kind
    with pytest.raises(spf_b200.SpfError) as e:
        spf_b200.BoxGraph(box2, bad)
    assert e.value.code == -4
    h = DeviceCiphertext.alloc(evaluation, keys.glwe_len * 8)
    c = FheCircuit()
    c.add("OutputGlwe1", c.add("Not", c.add("InputGlwe1", io=h)), io=np.zeros(keys.glwe_len, dtype=np.uint64))
    with pytest.raises(spf_b200.SpfError) as e:
        spf_b200.BoxGraph(box2, c)
    assert e.value.code == -1 and "device-memory" in str(e.value)


def test_destroy_with_a_spawned_run_in_flight(keys, client, box2):
    import spf_b200

    w, vals = 8, [(7, 9, 10)]
    circ, out_prod, out_gt = _multiply_program(client, keys, w, vals)
    g = spf_b200.BoxGraph(box2, circ)
    fired = []
    done = threading.Event()
    g.spawn(on_complete=lambda e: (fired.append(e), done.set()))
    g.close()  # waits for the run
    assert done.is_set() and fired == [None]
    assert _decrypt_multiply(client, out_prod, out_gt) == ([63], [1])


# ---- several GPUs --------------------------------------------------------------------------------------------------
def test_multi_device_key_replicas_are_byte_equal(keys, box_all):
    _check_key_replicas(box_all, keys)


def test_multi_device_cbs(client, evaluation, box_all):
    rng = np.random.default_rng(72)
    _check_cbs_against_slices(box_all, evaluation, client, [int(x) for x in rng.integers(0, 2, 64 * box_all.size + 3)])


def test_multi_device_graph(keys, client, evaluation, box_all):
    _graph_check(keys, client, evaluation, box_all)


def test_multi_device_instruction_cache_add_32bit(keys, client, box_all):
    from spf_b200.circuits import InstructionCache

    w, a, b = 32, 0xDEADBEEF, 0x12345678
    enc = lambda v: [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]
    out = [np.zeros(keys.glwe_len, dtype=np.uint64) for _ in range(w + 1)]
    cache = InstructionCache(box_all)
    cache.add(enc(a), enc(b), out)
    assert sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(out)) == a + b
