"""The level-synchronous graph executor (spf_b200_graph_*; CircuitProcessor equivalent) on the GPU,
modelled on parasol_runtime/src/circuit_processor/tests/{mod.rs,faults.rs}."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def proc(evaluation):
    import spf_b200

    return spf_b200.CircuitProcessor(evaluation)


def test_copy_and_constants(keys, client, proc):
    """circuit_processor/tests/mod.rs:53-120: Input -> Output copies; Zero/One constants."""
    import spf_b200

    g_in = client.encrypt_glwe_l1([1, 0, 1])
    l0_in = client.encrypt_lwe_l0(1)
    g_out = np.zeros_like(g_in)
    l0_out = np.zeros_like(l0_in)
    z, o = np.zeros(keys.glwe_len, dtype=np.uint64), np.zeros(keys.glwe_len, dtype=np.uint64)
    gz, go = np.zeros(keys.ggsw_fft_len, dtype=np.complex128), np.zeros(keys.ggsw_fft_len, dtype=np.complex128)
    c = spf_b200.FheCircuit()
    c.add("OutputGlwe1", c.add("InputGlwe1", io=g_in), io=g_out)
    c.add("OutputLwe0", c.add("InputLwe0", io=l0_in), io=l0_out)
    c.add("OutputGlwe1", c.add("ZeroGlwe1"), io=z)
    c.add("OutputGlwe1", c.add("OneGlwe1"), io=o)
    c.add("OutputGgsw1", c.add("ZeroGgsw1"), io=gz)
    c.add("OutputGgsw1", c.add("OneGgsw1"), io=go)
    c.add("Nop")
    proc.run_graph_blocking(c)
    assert np.array_equal(g_out, g_in) and np.array_equal(l0_out, l0_in)
    assert client.decrypt_glwe_l1(z)[:2].tolist() == [0, 0] and client.decrypt_glwe_l1(o)[:2].tolist() == [1, 0]
    assert client.decrypt_ggsw_l1(gz) == 0 and client.decrypt_ggsw_l1(go) == 1


def test_sample_extract_keyswitch_cbs_cmux(oracle, keys, client, proc):
    """mod.rs:122-193: sample extract, keyswitch, CBS + CMux through the graph; every intermediate
    stays on the device.  Integer nodes are bit-exact against the oracle."""
    import spf_b200

    bits = [1, 0, 1, 1]
    src = client.encrypt_glwe_l1(bits)
    a, b = client.encrypt_glwe_l1([0]), client.encrypt_glwe_l1([1])
    outs = [np.zeros(keys.glwe_len, dtype=np.uint64) for _ in bits]
    l0s = [np.zeros(keys.lwe0_len, dtype=np.uint64) for _ in bits]
    c = spf_b200.FheCircuit()
    x = c.add("InputGlwe1", io=src)
    na, nb = c.add("InputGlwe1", io=a), c.add("InputGlwe1", io=b)
    for i in range(len(bits)):
        l0 = c.add("KeyswitchL1toL0", c.add("SampleExtract", x, arg=i))
        c.add("OutputLwe0", l0, io=l0s[i])
        sel = c.add("CircuitBootstrap", l0)
        c.add("OutputGlwe1", c.add("CMux", sel, na, nb), io=outs[i])
    g = proc.compile(c)
    g.run()
    assert g.levels == 6
    for i, bit in enumerate(bits):
        assert np.array_equal(l0s[i], oracle.keyswitch_lwe(keys, oracle.sample_extract(keys, src, i)))
        assert client.decrypt_glwe_l1(outs[i])[0] == bit
    launches = g.launches
    g.run()  # re-running a compiled graph re-reads the inputs
    assert g.launches == launches
    g.close()
    # 4 chains, but one launch per (level, op) group: SE, KS, PBS + trace/SS, CMUX, and one gather of the outputs
    assert launches <= 7


def test_not_add_mulxn_multiply(oracle, keys, client, proc):
    import spf_b200

    a, b = client.encrypt_glwe_l1([1, 0, 1, 0]), client.encrypt_glwe_l1([1, 1, 0, 0])
    ggsw = client.encrypt_ggsw_l1(1)
    o = [np.zeros(keys.glwe_len, dtype=np.uint64) for _ in range(4)]
    c = spf_b200.FheCircuit()
    na, nb, ng = c.add("InputGlwe1", io=a), c.add("InputGlwe1", io=b), c.add("InputGgsw1", io=ggsw)
    c.add("OutputGlwe1", c.add("Not", na), io=o[0])
    c.add("OutputGlwe1", c.add("GlweAdd", na, nb), io=o[1])
    c.add("OutputGlwe1", c.add("MulXN", na, arg=2), io=o[2])
    c.add("OutputGlwe1", c.add("MultiplyGgswGlwe", na, ng), io=o[3])
    proc.run_graph_blocking(c)
    assert np.array_equal(o[0], oracle.glwe_not(keys, a))
    assert np.array_equal(o[1], a + b)
    assert np.array_equal(o[2], oracle.glwe_mul_xn(keys, a, 2))
    assert oracle.torus_distance(o[3], oracle.multiply_glwe_ggsw(keys, a, ggsw)).max() <= 2.0 ** -30


def test_glev_cmux_and_scheme_switch_nodes(oracle, keys, client, proc):
    import spf_b200

    d0, d1 = client.encrypt_glev_l1([0, 1]), client.encrypt_glev_l1([1, 1])
    sel = client.encrypt_ggsw_l1(1)
    out_glev = np.zeros(keys.glev_len, dtype=np.uint64)
    out_ggsw = np.zeros(keys.ggsw_fft_len, dtype=np.complex128)
    c = spf_b200.FheCircuit()
    n0, n1, ns = c.add("InputGlev1", io=d0), c.add("InputGlev1", io=d1), c.add("InputGgsw1", io=sel)
    m = c.add("GlevCMux", ns, n0, n1)
    c.add("OutputGlev1", m, io=out_glev)
    c.add("OutputGgsw1", c.add("SchemeSwitch", m), io=out_ggsw)
    proc.run_graph_blocking(c)
    assert oracle.torus_distance(out_glev, oracle.glev_cmux(keys, d0, d1, sel)).max() <= 2.0 ** -30
    # the selected GLEV encrypts [1, 1]: as a GGSW its last-row level-0 GLWE decodes to 1 at coeffs 0, 1
    msgs = client.ggsw_level_messages(out_ggsw)
    assert msgs[1, 0, :3].tolist() == [1, 1, 0]


@pytest.mark.parametrize("a,b", [(2, 7), (255, 1), (170, 85), (0, 0)])
def test_basic_add_8bit(keys, client, proc, a, b):
    """BASELINE config 1 (examples/basic_add: encrypted uint8 a + b; parasol_cpu/src/proc/ops/add.rs:13-80):
    16 x (SampleExtract -> KeyswitchL1toL0 -> CircuitBootstrap) + a ripple-carry MUX tree."""
    from spf_b200.circuits import ripple_carry_adder

    w = 8
    ab = [client.encrypt_glwe_l1([(a >> i) & 1]) for i in range(w)]
    bb = [client.encrypt_glwe_l1([(b >> i) & 1]) for i in range(w)]
    outs = [np.zeros(keys.glwe_len, dtype=np.uint64) for _ in range(w + 1)]
    g = proc.compile(ripple_carry_adder(ab, bb, outs))
    g.run()
    got = sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(outs))
    assert got == a + b
    assert g.levels <= 4 + 3 * w + 1  # front end (4) + <= 3 levels per bit (2 CMUX + Not) + outputs
    assert g.launches <= 2 * g.levels  # one launch per (level, op) group, not per node
    g.close()


def test_malformed_graphs(keys, client, proc):
    """circuit_processor/tests/faults.rs:10-118 -> SPF_E_GRAPH (-4) with a message."""
    import spf_b200

    glwe = client.encrypt_glwe_l1([1])
    lwe0 = client.encrypt_lwe_l0(1)

    def expect(c, text):
        with pytest.raises(spf_b200.SpfError) as e:
            proc.run_graph_blocking(c)
        assert e.value.code == -4 and text in str(e.value), str(e.value)

    c = spf_b200.FheCircuit()
    c.add("CircuitBootstrap", c.add("InputGlwe1", io=glwe))  # GLWE into an LWE0 port
    expect(c, "wrong ciphertext kind")
    c = spf_b200.FheCircuit()
    c.add("CMux", c.add("InputGlwe1", io=glwe), -1, -1)  # missing inputs
    expect(c, "missing ciphertext input")
    c = spf_b200.FheCircuit()
    c.add("SampleExtract", c.add("InputGlwe1", io=glwe), arg=2048)
    expect(c, "illegal sample extract")
    c = spf_b200.FheCircuit()
    c.nodes.append((spf_b200.OP["Not"], 0, (1, -1, -1), None))  # 0 <- 1 <- 0
    c.nodes.append((spf_b200.OP["Not"], 0, (0, -1, -1), None))
    expect(c, "cycle")
    c = spf_b200.FheCircuit()
    c.add("KeyswitchL1toL0", c.add("InputLwe0", io=lwe0))
    expect(c, "wrong ciphertext kind")


def _two_level_program(client, keys, w, programs, rng):
    import spf_b200
    from spf_b200.circuits import add_then_greater_than

    vals = [(int(rng.integers(0, 1 << w)), int(rng.integers(0, 1 << w)), int(rng.integers(0, 1 << w))) for _ in range(programs)]
    enc = lambda v: [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]
    a, b, c = ([enc(v[k]) for v in vals] for k in range(3))
    out_sum = [[np.zeros(keys.glwe_len, dtype=np.uint64) for _ in range(w)] for _ in range(programs)]
    out_gt = [np.zeros(keys.glwe_len, dtype=np.uint64) for _ in range(programs)]
    return vals, add_then_greater_than(a, b, c, out_sum, out_gt, programs), out_sum, out_gt


def _check_program(client, vals, w, out_sum, out_gt):
    for (a, b, c), s_bits, gt in zip(vals, out_sum, out_gt):
        s = sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(s_bits))
        assert s == (a + b) % (1 << w)
        assert int(client.decrypt_glwe_l1(gt)[0]) == int(s > c)


def test_add_then_compare_two_level_program(keys, client, proc):
    """A two-instruction program (add, then greater-than on the refreshed sum bits): two circuit-
    bootstrap levels in one graph, as in BASELINE config 4's multi-level programs."""
    rng = np.random.default_rng(11)
    w = 6
    vals, circ, out_sum, out_gt = _two_level_program(client, keys, w, 2, rng)
    g = proc.compile(circ)
    g.run()
    _check_program(client, vals, w, out_sum, out_gt)
    g.close()


def test_sharded_run_emulated_on_one_gpu(keys, client, evaluation):
    """spf_b200_graph_run_sharded with world = 2, both ranks emulated on this GPU: rank r computes
    chunk r of every CircuitBootstrap level and the MUX trees it owns; the exchange callback parks the
    rank's own chunk and fills in the peer's chunk from the peer's previous pass.  After (exchanges + 1)
    alternating passes every exchange has seen correct peer data; every output is written by its owning
    rank into the shared host buffers, which must then decrypt correctly."""
    import ctypes as C

    import spf_b200

    rng = np.random.default_rng(12)
    w, world = 4, 2
    vals, circ, out_sum, out_gt = _two_level_program(client, keys, w, 1, rng)
    cudart = C.CDLL("libcudart.so.12")
    parked = {0: {}, 1: {}}  # rank -> exchange index -> host copy of that rank's chunk
    counter = {"i": 0}

    def make_exchange(rank):
        def exchange(d_buf, chunk_bytes, world_, stream):
            assert world_ == world
            i = counter["i"]
            counter["i"] += 1
            assert cudart.cudaStreamSynchronize(C.c_void_p(stream)) == 0
            mine = np.empty(chunk_bytes, dtype=np.uint8)
            assert cudart.cudaMemcpy(C.c_void_p(mine.ctypes.data), C.c_void_p(d_buf + rank * chunk_bytes), C.c_size_t(chunk_bytes), 2) == 0
            parked[rank][i] = mine
            peer = parked[1 - rank].get(i)
            if peer is not None:
                assert cudart.cudaMemcpy(C.c_void_p(d_buf + (1 - rank) * chunk_bytes), C.c_void_p(peer.ctypes.data), C.c_size_t(chunk_bytes), 1) == 0
        return exchange

    graphs = [spf_b200.CompiledGraph(evaluation, circ, world=world, rank=r, exchange=make_exchange(r)) for r in range(world)]
    for _ in range(5):  # four dependent exchanges -> correct after five alternating passes
        for r in (1, 0):
            counter["i"] = 0
            graphs[r].run()
    assert counter["i"] == 4  # per bootstrap level: keyswitch outputs, then the GGSWs
    _check_program(client, vals, w, out_sum, out_gt)
    out_nodes = [i for i, nd in enumerate(circ.nodes) if nd[0] == spf_b200.OP["OutputGlwe1"]]
    ranks = {graphs[0].output_rank(i) for i in out_nodes}
    assert ranks <= {0, 1} and all(graphs[0].output_rank(i) == graphs[1].output_rank(i) for i in out_nodes)
    with pytest.raises(spf_b200.SpfError):
        graphs[0].output_rank(0)
    # a graph laid out for a sharded run refuses the unsharded entry point
    assert spf_b200.lib().spf_b200_graph_run(graphs[0]._h) == -1
    for g in graphs:
        g.close()


def test_instruction_cache_reuses_compiled_graph(keys, client, evaluation):
    """SURVEY.md 8(f).3: one compiled graph per (instruction, width), re-bound per invocation."""
    import spf_b200
    from spf_b200.circuits import InstructionCache

    cache = InstructionCache(evaluation)
    w = 5
    for a, b in ((3, 9), (31, 31), (0, 17)):
        ab = [client.encrypt_glwe_l1([(a >> i) & 1]) for i in range(w)]
        bb = [client.encrypt_glwe_l1([(b >> i) & 1]) for i in range(w)]
        outs = [np.zeros(keys.glwe_len, dtype=np.uint64) for _ in range(w + 1)]
        cache.add(ab, bb, outs)
        assert sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(outs)) == a + b
    assert (cache.misses, cache.hits) == (1, 2)
    g = cache._cache[("add", w)][0]
    with pytest.raises(spf_b200.SpfError):
        g.set_io(10 ** 6, np.zeros(4, dtype=np.uint64))  # not a node


def test_instruction_cache_multiply_and_compare(keys, client, evaluation):
    """The cached ISA instructions built from BDD-derived MUX circuits: 6-bit unsigned multiply (low word)
    and greater-than, two invocations each on ONE compiled graph."""
    from spf_b200.circuits import InstructionCache

    cache = InstructionCache(evaluation)
    w = 6
    enc = lambda v: [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]
    for a, b in ((13, 11), (63, 63)):
        outs = [np.zeros(keys.glwe_len, dtype=np.uint64) for _ in range(w)]
        cache.multiply(enc(a), enc(b), outs)
        assert sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(outs)) == (a * b) % (1 << w)
        gt = np.zeros(keys.glwe_len, dtype=np.uint64)
        cache.greater_than(enc(a), enc(b), gt)
        assert int(client.decrypt_glwe_l1(gt)[0]) == int(a > b)
    assert (cache.misses, cache.hits) == (2, 2)
    with pytest.raises(ValueError):
        cache.multiply(enc(1) * 4, enc(1) * 4, [np.zeros(keys.glwe_len, dtype=np.uint64)] * (4 * w))


def test_glev_round_trip_then_mux_circuit(keys, client, proc):
    """The reference's ciphertext conversions in a graph (fhe_circuit.rs:562-619): selectors go GGSW -> GLEV
    (GlevCMux(sel, ZeroGlev1, OneGlev1)) -> GGSW (SchemeSwitch, no circuit bootstrap) and then drive a BDD-derived
    2-bit AND with a second operand.  (Deeper GLEV-mode trees are outside the noise budget of DEFAULT_128: one
    CMux with cbs_radix (l = 4, logB = 4) leaves ~2^-13 of decomposition noise, which already swamps the two finest
    GLEV levels -- `tools/glev_debug.py` shows the levels decoding to garbage after two GlevCMux.)"""
    import spf_b200
    from spf_b200 import mux_circuits as M

    for a, b in ((0b11, 0b01), (0b10, 0b11), (0b00, 0b10)):
        c = spf_b200.FheCircuit()
        front = lambda v: [M.insert_ciphertext_conversion(c, c.add("InputGlwe1", io=client.encrypt_glwe_l1([(v >> i) & 1])), "glwe", "ggsw")
                           for i in range(2)]
        sa, sb = front(a), front(b)
        sa_rt = [M.insert_ciphertext_conversion(c, M.insert_ciphertext_conversion(c, x, "ggsw", "glev"), "glev", "ggsw") for x in sa]
        and_out = M.insert_mux_circuit(c, M.make_and_circuit(2), [sa_rt[0], sb[0], sa_rt[1], sb[1]])
        outs = [np.zeros(keys.glwe_len, dtype=np.uint64) for _ in range(2)]
        for n, buf in zip(and_out, outs):
            c.add("OutputGlwe1", n, io=buf)
        ops = [spf_b200.OPS[n[0]] for n in c.nodes]
        assert ops.count("CircuitBootstrap") == 4 and ops.count("SchemeSwitch") == 2 and ops.count("GlevCMux") == 2
        proc.run_graph_blocking(c)
        got = sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(outs))
        assert got == a & b, (a, b, got)


def test_signed_multiply_4bit(keys, client, proc):
    """append_int_multiply (parasol_runtime/src/circuits/mul.rs:19-73) on encrypted 4-bit two's-complement operands:
    abs -> unsigned multiplier -> conditional negate, three bootstrap levels; the 8 product bits decrypt to a * b."""
    import spf_b200
    from spf_b200 import mux_circuits as M

    w = 4
    for a, b in ((-3, 5), (-8, -8), (7, -1)):
        c = spf_b200.FheCircuit()
        front = lambda v: [M.insert_ciphertext_conversion(c, c.add("InputGlwe1", io=client.encrypt_glwe_l1([(v >> i) & 1])), "glwe", "ggsw")
                           for i in range(w)]
        lo, hi = M.append_int_multiply(c, front(a & 0xF), front(b & 0xF))
        outs = [np.zeros(keys.glwe_len, dtype=np.uint64) for _ in range(2 * w)]
        for n, buf in zip(lo + hi, outs):
            c.add("OutputGlwe1", n, io=buf)
        proc.run_graph_blocking(c)
        got = sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(outs))
        assert got == (a * b) % 256, (a, b, got)


def test_pinned_slab_buffers(keys, client, proc):
    """spf_b200_host_alloc: ciphertext buffers sliced from one page-locked slab work as graph IO (and are not
    registered again); the slab is released with the array."""
    import spf_b200

    slab = spf_b200.pinned_zeros((3, keys.glwe_len))
    assert slab.flags["C_CONTIGUOUS"] and not slab.any()
    slab[0][:] = client.encrypt_glwe_l1([1, 0, 1])
    c = spf_b200.FheCircuit()
    x = c.add("InputGlwe1", io=slab[0])
    c.add("OutputGlwe1", x, io=slab[1])
    c.add("OutputGlwe1", c.add("Not", x), io=slab[2])
    g = proc.compile(c)
    g.run()
    assert np.array_equal(slab[1], slab[0])
    assert client.decrypt_glwe_l1(slab[2])[:3].tolist() == [0, 0, 1]   # Not adds a trivial one: only coefficient 0 flips
    g.close()
    with pytest.raises(spf_b200.SpfError):
        spf_b200.pinned_zeros((1 << 50,), np.uint8)


def test_pack_unpack_roundtrip(oracle, keys, client, proc):
    """SURVEY.md 8(f).4: the fluent layer's pack (MulXN + GlweAdd tree) and unpack (SampleExtract(i)) graph
    shapes on the executor; the unpacked bits are refreshed through keyswitch + CBS and used as selectors."""
    import spf_b200
    from spf_b200.circuits import pack, unpack

    value, w = 0b1011001, 7
    bits = [(value >> i) & 1 for i in range(w)]
    c = spf_b200.FheCircuit()
    ins = [c.add("InputGlwe1", io=client.encrypt_glwe_l1([b])) for b in bits]
    packed = pack(c, ins)
    packed_out = np.zeros(keys.glwe_len, dtype=np.uint64)
    c.add("OutputGlwe1", packed, io=packed_out)
    lwes = unpack(c, packed, w)
    l1_out = [np.zeros(keys.lwe1_len, dtype=np.uint64) for _ in range(w)]
    zero, one = c.add("ZeroGlwe1"), c.add("OneGlwe1")
    mux_out = [np.zeros(keys.glwe_len, dtype=np.uint64) for _ in range(w)]
    for i, n in enumerate(lwes):
        c.add("OutputLwe1", n, io=l1_out[i])
        sel = c.add("CircuitBootstrap", c.add("KeyswitchL1toL0", n))
        c.add("OutputGlwe1", c.add("CMux", sel, zero, one), io=mux_out[i])
    proc.run_graph_blocking(c)
    assert client.decrypt_glwe_l1(packed_out)[:w].tolist() == bits          # bit i sits in coefficient i
    assert [client.decrypt_lwe_l1(x) for x in l1_out] == bits
    assert [int(client.decrypt_glwe_l1(x)[0]) for x in mux_out] == bits


def test_peer_memory_exchange_two_ranks_on_one_gpu(keys, client, evaluation):
    """The fused exchange of a sharded run (spf_b200_graph_set_peers): two ranks as two contexts on this GPU, run
    concurrently from two host threads; the scheme-switch kernel of each rank stores its GGSWs into both arenas,
    keyswitch outputs are broadcast, levels are separated by the peer-memory flag barrier.  Each output is written
    by its owner rank into the shared host buffers."""
    import threading

    import spf_b200

    ev1 = spf_b200.Evaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft, device=0)
    rng = np.random.default_rng(31)
    w, world = 4, 2
    vals, circ, out_sum, out_gt = _two_level_program(client, keys, w, 2, rng)
    graphs = [spf_b200.CompiledGraph(e, circ, world=world, rank=r) for r, e in enumerate((evaluation, ev1))]
    with pytest.raises(spf_b200.SpfError):
        graphs[0].run()  # neither an exchange callable nor peers
    arenas = [g.arena for g in graphs]
    assert all(arenas) and arenas[0] != arenas[1]
    for g in graphs:
        g.set_peers(arenas)
    for _ in range(2):  # twice: the start-of-run barrier orders run k + 1 after every rank's run k
        for buf in [b for p_ in out_sum for b in p_] + out_gt:
            buf[:] = 0
        errs = []

        def go(g):
            try:
                g.run()
            except Exception as e:  # surfaced below
                errs.append(e)

        ths = [threading.Thread(target=go, args=(g,)) for g in graphs]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        assert not errs, errs
        _check_program(client, vals, w, out_sum, out_gt)
    for g in graphs:
        g.close()
    ev1.close()


def test_peer_barrier_times_out_instead_of_hanging(keys, client, evaluation):
    """A rank that never arrives: the peer-memory barrier gives up after its device-side timeout (5 s) and the run
    fails with SPF_E_GRAPH -- the GPU is not left spinning."""
    import time

    import spf_b200

    rng = np.random.default_rng(33)
    vals, circ, out_sum, out_gt = _two_level_program(client, keys, 2, 1, rng)
    graphs = [spf_b200.CompiledGraph(evaluation, circ, world=2, rank=r) for r in range(2)]
    for g in graphs:
        g.set_peers([x.arena for x in graphs])
    t0 = time.perf_counter()
    with pytest.raises(spf_b200.SpfError) as e:
        graphs[0].run()   # rank 1 never runs
    assert "peer barrier timed out" in str(e.value) and e.value.code == -4
    assert 4.0 < time.perf_counter() - t0 < 12.0   # one timeout, not one per barrier
    for g in graphs:
        g.close()


def _multiply_program(client, keys, w, vals):
    from spf_b200.circuits import multiply_then_greater_than

    enc = lambda v: [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]
    a, b, c = ([enc(v[k]) for v in vals] for k in range(3))
    out_prod = [[np.zeros(keys.glwe_len, dtype=np.uint64) for _ in range(w)] for _ in vals]
    out_gt = [np.zeros(keys.glwe_len, dtype=np.uint64) for _ in vals]
    return multiply_then_greater_than(a, b, c, out_prod, out_gt, len(vals)), out_prod, out_gt


def _check_multiply(client, vals, w, out_prod, out_gt):
    for (a, b, c), p_bits, gt in zip(vals, out_prod, out_gt):
        p = sum(int(client.decrypt_glwe_l1(o)[0]) << i for i, o in enumerate(p_bits))
        assert p == (a * b) % (1 << w), (a, b, p)
        assert int(client.decrypt_glwe_l1(gt)[0]) == int(p > c)


def test_multiply_then_compare_8bit(keys, client, proc):
    """The ISA's unsigned multiply (parasol_cpu/src/proc/tests/mul.rs) on 8-bit operands: one BDD-derived
    8x8 multiplier block (the low word keeps 639 of its 3228 multiplexers after pruning), then CmpGt on the
    refreshed product bits."""
    w = 8
    vals = [(13, 11, 100), (255, 255, 0), (0, 77, 0)]
    circ, out_prod, out_gt = _multiply_program(client, keys, w, vals)
    g = proc.compile(circ)
    g.run()
    _check_multiply(client, vals, w, out_prod, out_gt)
    g.close()


def test_multiply_then_compare_32bit(keys, client, proc):
    """BASELINE config 4's program on one GPU: 32-bit multiply (four 16x16 blocks + grade-school reduction,
    45 k CMUX nodes over ~600 dependency levels, three circuit-bootstrap levels of 96 / 64 / 32) then
    greater-than; decrypts to the plain product and comparison."""
    w = 32
    rng = np.random.default_rng(21)
    vals = [(int(rng.integers(0, 1 << w)), int(rng.integers(0, 1 << w)), int(rng.integers(0, 1 << w))), (0xFFFFFFFF, 0xFFFFFFFF, 0)]
    for v in vals:
        circ, out_prod, out_gt = _multiply_program(client, keys, w, [v])
        g = proc.compile(circ)
        g.run()
        _check_multiply(client, [v], w, out_prod, out_gt)
        g.close()
