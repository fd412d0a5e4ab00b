"""MUX-circuit generator (spf_b200/csrc/muxgen.cpp through the C ABI) and its expansion into
FheCircuit graphs: the reference's own test strategy for mux_circuits (random operands against plain
integer arithmetic, mux_circuits/src/{add,sub,neg,comparisons,mul}.rs `mod tests`), the multiplexer
counts of the reference's shipped pre-generated circuits as golden values, and the serialized
MuxCircuit format.  No GPU needed."""
import numpy as np
import pytest

from spf_b200 import FheCircuit, OP, SpfError
from spf_b200 import OPS as spf_b200_ops
from spf_b200 import mux_circuits as M


def bits(v, w):
    return [(v >> i) & 1 for i in range(w)]


def value(b):
    return sum(int(x) << i for i, x in enumerate(b))


def rand(rng, w):
    return int.from_bytes(rng.bytes(16), "little") % (1 << w)


@pytest.mark.parametrize("n,m,cin", [(8, 8, False), (8, 8, True), (5, 9, False), (9, 5, True), (32, 32, False), (1, 1, True)])
def test_ripple_carry_adder(n, m, cin):
    c = M.ripple_carry_adder(n, m, cin)
    assert c.metrics()["inputs"] == n + m + cin and c.metrics()["outputs"] == max(n, m) + 1
    rng = np.random.default_rng(n * 100 + m)
    lo = min(n, m)
    for _ in range(50):
        a, b, ci = rand(rng, n), rand(rng, m), int(rng.integers(0, 2)) if cin else 0
        ab, bb = bits(a, n), bits(b, m)
        inp = ([ci] if cin else []) + [x for p in zip(ab[:lo], bb[:lo]) for x in p] + (ab[lo:] if n > m else bb[lo:])
        assert value(c.evaluate(inp)) == a + b + ci


@pytest.mark.parametrize("n,bin_", [(8, False), (8, True), (32, False)])
def test_full_subtractor(n, bin_):
    c = M.full_subtractor(n, bin_)
    rng = np.random.default_rng(n)
    for _ in range(50):
        a, b, bi = rand(rng, n), rand(rng, n), int(rng.integers(0, 2)) if bin_ else 0
        inp = ([bi] if bin_ else []) + [x for p in zip(bits(a, n), bits(b, n)) for x in p]
        out = c.evaluate(inp)
        assert value(out[:n]) == (a - b - bi) % (1 << n) and out[n] == int(a - b - bi < 0)


def test_negator():
    c = M.negator(16)
    for a in (0, 1, 2, 0x8000, 0xFFFF, 12345):
        assert value(c.evaluate(bits(a, 16))) == (-a) % (1 << 16)


@pytest.mark.parametrize("greater", [False, True])
@pytest.mark.parametrize("or_equal", [False, True])
def test_comparisons(greater, or_equal):
    n = 8
    cu, cs = M.compare_or_maybe_equal(n, greater, or_equal), M.compare_or_maybe_equal_signed(n, greater, or_equal)
    rng = np.random.default_rng(3)
    cases = [(rand(rng, n), rand(rng, n)) for _ in range(100)] + [(7, 7), (0, 255), (255, 0), (128, 127)]
    for a, b in cases:
        inp = [x for p in zip(bits(a, n), bits(b, n)) for x in p]
        want = (a > b if greater else a < b) or (or_equal and a == b)
        assert cu.evaluate(inp) == [int(want)]
        sa, sb = a - 256 * (a >> 7), b - 256 * (b >> 7)
        want = (sa > sb if greater else sa < sb) or (or_equal and sa == sb)
        assert cs.evaluate(inp) == [int(want)]


def test_equality_and_bitwise():
    n = 8
    eq, ne, an, orr = M.compare_equal(n), M.compare_not_equal(n), M.make_and_circuit(n), M.make_or_circuit(n)
    rng = np.random.default_rng(4)
    for a, b in [(rand(rng, n), rand(rng, n)) for _ in range(50)] + [(9, 9), (0, 0)]:
        inp = [x for p in zip(bits(a, n), bits(b, n)) for x in p]
        assert eq.evaluate(inp) == [int(a == b)] and ne.evaluate(inp) == [int(a != b)]
        assert value(an.evaluate(inp)) == a & b and value(orr.evaluate(inp)) == a | b


# multiplexer counts of the circuits the reference ships pre-generated (mux_circuits/src/data/
# multiplier-n8-m8, multiplier-n16-m16, gradeschool-reduction-n64-m64, loaded by mul.rs:62-68,393-400)
GOLDEN_MUX_GATES = {("unsigned_multiplier", 8, 8): 3228, ("unsigned_multiplier", 16, 16): 29500,
                    ("gradeschool_reduce", 64, 64): 36888}


@pytest.mark.parametrize("n,m", [(1, 1), (4, 4), (5, 3), (3, 7), (8, 8), (16, 16)])
def test_unsigned_multiplier(n, m):
    c = M.unsigned_multiplier(n, m)
    assert c.metrics()["inputs"] == n + m and c.metrics()["outputs"] == n + m
    if ("unsigned_multiplier", n, m) in GOLDEN_MUX_GATES:
        assert c.metrics()["mux_gates"] == GOLDEN_MUX_GATES[("unsigned_multiplier", n, m)]
    rng = np.random.default_rng(n * 64 + m)
    cases = [(rand(rng, n), rand(rng, m)) for _ in range(20 if n < 16 else 6)] + [((1 << n) - 1, (1 << m) - 1), (0, 1)]
    for a, b in cases:
        assert value(c.evaluate(bits(a, n) + bits(b, m))) == a * b


@pytest.mark.parametrize("n,m", [(32, 32), (64, 64), (40, 24), (20, 18)])
def test_gradeschool_reduce(n, m):
    c = M.gradeschool_reduce(n, m)
    assert c.metrics()["inputs"] == 2 * (n + m) and c.metrics()["outputs"] == n + m
    if ("gradeschool_reduce", n, m) in GOLDEN_MUX_GATES:
        assert c.metrics()["mux_gates"] == GOLDEN_MUX_GATES[("gradeschool_reduce", n, m)]
    (a_lo, a_hi), (b_lo, b_hi) = M.partition_integer(n), M.partition_integer(m)
    rng = np.random.default_rng(n)
    for x, y in [(rand(rng, n), rand(rng, m)) for _ in range(8)] + [((1 << n) - 1, (1 << m) - 1)]:
        xl, xh, yl, yh = x & ((1 << a_lo) - 1), x >> a_lo, y & ((1 << b_lo) - 1), y >> b_lo
        inp = M.encode_gradeschool_reduction(n, m, bits(xl * yl, a_lo + b_lo), bits(xl * yh, a_lo + b_hi),
                                             bits(xh * yl, a_hi + b_lo), bits(xh * yh, a_hi + b_hi))
        assert value(c.evaluate(inp)) == x * y


def test_generator_rejects_bad_sizes():
    for args in [("unsigned_multiplier", 0, 4), ("unsigned_multiplier", 4, 0), ("unsigned_multiplier", 256, 256),
                 ("gradeschool_reduce", 16, 32), ("ripple_carry_adder", 4, 0)]:
        with pytest.raises(SpfError):
            M.MuxCircuit.generate(*args)


def test_bincode_round_trip_and_errors():
    c = M.unsigned_multiplier(4, 4)
    blob = c.to_bincode()
    d = M.MuxCircuit.from_bincode(blob)
    assert d.metrics() == c.metrics()
    for a, b in [(3, 5), (15, 15), (9, 0)]:
        assert value(d.evaluate(bits(a, 4) + bits(b, 4))) == a * b
    with pytest.raises(SpfError):
        M.MuxCircuit.from_bincode(blob[:-3])
    with pytest.raises(SpfError):
        M.MuxCircuit.from_bincode(b"\xff" * 8 + blob[8:])


def _plain_run(c: FheCircuit, ggsw_bits: dict[int, int]) -> dict[int, int]:
    """Evaluate the Boolean skeleton of a FheCircuit (CMux / constants / conversions) on plaintext bits."""
    val = {}
    for i, (op, arg, ins, io) in enumerate(c.nodes):
        if i in ggsw_bits:
            val[i] = ggsw_bits[i]
        elif op == OP["CMux"]:
            val[i] = val[ins[2]] if val[ins[0]] else val[ins[1]]
        elif op in (OP["ZeroGlwe1"], OP["ZeroGgsw1"]):
            val[i] = 0
        elif op in (OP["OneGlwe1"], OP["OneGgsw1"]):
            val[i] = 1
        elif op in (OP["SampleExtract"], OP["KeyswitchL1toL0"], OP["CircuitBootstrap"]):
            val[i] = val[ins[0]]
        elif op == OP["MultiplyGgswGlwe"]:   # in[0] = Glwe, in[1] = Ggsw
            val[i] = val[ins[0]] & val[ins[1]]
    return val


@pytest.mark.parametrize("w", [8, 32, 24])
def test_append_uint_multiply_structure(w):
    """circuits/mul.rs: a w x w product expands to 16x16 blocks + one reduction behind a bootstrap
    level (w > 16) or a single block (w <= 16); the graph's Boolean skeleton multiplies."""
    c = FheCircuit()
    a = [c.add("OneGgsw1") for _ in range(w)]   # stand-ins for the operands' GGSW producers
    b = [c.add("OneGgsw1") for _ in range(w)]
    lo, hi = M.append_uint_multiply(c, a, b)
    assert len(lo) == w and len(hi) == w
    n_cbs = sum(1 for n in c.nodes if n[0] == OP["CircuitBootstrap"])
    assert n_cbs == (0 if w <= 16 else 4 * w)
    rng = np.random.default_rng(w)
    for x, y in [(rand(rng, w), rand(rng, w)), ((1 << w) - 1, (1 << w) - 1)]:
        assign = {n: bt for n, bt in zip(a + b, bits(x, w) + bits(y, w))}
        val = _plain_run(c, assign)
        assert value([val[n] for n in lo + hi]) == x * y
    pruned, ren = M.prune(c, lo)
    assert len(pruned.nodes) < len(c.nodes)
    x, y = rand(rng, w), rand(rng, w)
    # inputs that survive pruning keep their meaning
    assign = {ren[n]: bt for n, bt in zip(a + b, bits(x, w) + bits(y, w)) if n in ren}
    val = _plain_run(pruned, assign)
    assert value([val[ren[n]] for n in lo]) == (x * y) % (1 << w)


def test_insert_mux_circuit_validates_inputs():
    c = FheCircuit()
    z = c.add("ZeroGlwe1")
    with pytest.raises(SpfError):
        M.insert_mux_circuit(c, M.make_and_circuit(1), [z, z])
    g = c.add("OneGgsw1")
    with pytest.raises(SpfError):
        M.insert_mux_circuit(c, M.make_and_circuit(1), [g])


def test_low_word_of_a_multiplier():
    """circuits._keep_outputs: the ISA Mul keeps the low word only (parasol_cpu/src/proc/ops/mul.rs:106-108)."""
    from spf_b200.circuits import _keep_outputs

    w = 6
    c = _keep_outputs(M.unsigned_multiplier(w, w), w)
    assert c.metrics()["outputs"] == w and c.metrics()["inputs"] == 2 * w
    for a, b in [(13, 11), (63, 63), (0, 5), (32, 2)]:
        assert value(c.evaluate(bits(a, w) + bits(b, w))) == (a * b) % (1 << w)


@pytest.mark.parametrize("right,mode", [(False, "logical"), (True, "logical"), (True, "arithmetic"), (False, "rotation"), (True, "rotation")])
def test_bitshift(right, mode):
    """mux_circuits/src/bitshift.rs tests: every value/shift pair of an 8-bit barrel shifter (big-endian inputs)."""
    w = 8
    c = M.bitshift(w, w, right, mode)
    be = lambda v: [(v >> (w - 1 - i)) & 1 for i in range(w)]
    from_be = lambda b: sum(int(x) << (w - 1 - i) for i, x in enumerate(b))
    for v in (0x00, 0x01, 0x80, 0xA5, 0xFF, 0x3C):
        for sh in list(range(0, 10)) + [16, 255]:
            got = from_be(c.evaluate(be(v) + be(sh)))
            if mode == "rotation":
                k = sh % w
                want = ((v >> k) | (v << (w - k))) & 0xFF if right else ((v << k) | (v >> (w - k))) & 0xFF
            elif mode == "logical":
                want = 0 if sh >= w else ((v >> sh) if right else (v << sh) & 0xFF)
            else:
                sv = v - 256 * (v >> 7)
                want = (sv >> min(sh, w - 1)) & 0xFF
            assert got == want, (v, sh, got, want)


def test_bitshift_rejects_what_the_reference_panics_on():
    for args in [(6, 6, False, "rotation"), (8, 8, False, "arithmetic"), (8, 2, True, "logical")]:
        with pytest.raises(SpfError):
            M.bitshift(*args)


def test_small_circuits_exhaustively():
    """Every input of a 3 x 3 multiplier, a 3 + 3 adder with carry-in and the 3-bit comparisons."""
    mul, add = M.unsigned_multiplier(3, 3), M.ripple_carry_adder(3, 3, True)
    for a in range(8):
        for b in range(8):
            assert value(mul.evaluate(bits(a, 3) + bits(b, 3))) == a * b
            inter = [x for p in zip(bits(a, 3), bits(b, 3)) for x in p]
            for cin in (0, 1):
                assert value(add.evaluate([cin] + inter)) == a + b + cin
            for greater in (False, True):
                for or_eq in (False, True):
                    want = (a > b if greater else a < b) or (or_eq and a == b)
                    assert M.compare_or_maybe_equal(3, greater, or_eq).evaluate(inter) == [int(want)]


def test_random_widths_property():
    """hypothesis: for random small widths the generated adder / subtractor / multiplier agree with integer arithmetic."""
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=40, deadline=None)
    @given(st.integers(1, 6), st.integers(1, 6), st.integers(0, 2 ** 12 - 1), st.integers(0, 2 ** 12 - 1))
    def check(n, m, x, y):
        a, b = x % (1 << n), y % (1 << m)
        assert value(M.unsigned_multiplier(n, m).evaluate(bits(a, n) + bits(b, m))) == a * b
        lo = min(n, m)
        ab, bb = bits(a, n), bits(b, m)
        inp = [v for p in zip(ab[:lo], bb[:lo]) for v in p] + (ab[lo:] if n > m else bb[lo:])
        assert value(M.ripple_carry_adder(n, m).evaluate(inp)) == a + b
        b2 = y % (1 << n)
        out = M.full_subtractor(n).evaluate([v for p in zip(bits(a, n), bits(b2, n)) for v in p])
        assert value(out[:n]) == (a - b2) % (1 << n) and out[n] == int(a < b2)

    check()


def test_ciphertext_conversions_and_glev_mode():
    """insert_ciphertext_conversion (fhe_circuit.rs:562-619) chains and MuxMode::Glev expansion; the planner accepts
    the result (kinds line up)."""
    from spf_b200 import plan_graph

    c = FheCircuit()
    g = c.add("OneGgsw1")
    assert M.insert_ciphertext_conversion(c, g, "ggsw", "ggsw") == g
    l0 = M.insert_ciphertext_conversion(c, g, "ggsw", "lwe0")      # MultiplyGgswGlwe -> SampleExtract -> Keyswitch
    back = M.insert_ciphertext_conversion(c, l0, "lwe0", "glev")   # CircuitBootstrap -> GlevCMux
    again = M.insert_ciphertext_conversion(c, back, "glev", "glwe")  # SchemeSwitch -> MultiplyGgswGlwe
    names = [spf_b200_ops[n[0]] for n in c.nodes]
    assert names == ["OneGgsw1", "OneGlwe1", "MultiplyGgswGlwe", "SampleExtract", "KeyswitchL1toL0", "CircuitBootstrap",
                     "ZeroGlev1", "OneGlev1", "GlevCMux", "SchemeSwitch", "OneGlwe1", "MultiplyGgswGlwe"]
    assert again == len(c) - 1
    outs = M.insert_mux_circuit(c, M.make_and_circuit(2), [g, g, g, g], mux_mode="glev")
    sel = [M.insert_ciphertext_conversion(c, o, "glev", "ggsw") for o in outs]
    M.insert_mux_circuit(c, M.make_or_circuit(1), sel)
    level, owner = plan_graph(c, 2)   # validates the kinds of every edge
    assert sum(1 for n in c.nodes if spf_b200_ops[n[0]] == "GlevCMux") >= 3
    with pytest.raises(SpfError):
        M.insert_ciphertext_conversion(c, g, "ggsw", "nonsense")


@pytest.mark.parametrize("w", [4, 6])
def test_append_int_multiply_structure(w):
    """circuits/mul.rs:19-73: the signed product's Boolean skeleton over every pair of w-bit two's-complement values."""
    c = FheCircuit()
    a = [c.add("OneGgsw1") for _ in range(w)]
    b = [c.add("OneGgsw1") for _ in range(w)]
    lo, hi = M.append_int_multiply(c, a, b)
    assert len(lo) == w and len(hi) == w
    signed = lambda v: v - (1 << w) * (v >> (w - 1))
    step = 1 if w == 4 else 5
    for x in range(0, 1 << w, step):
        for y in range(0, 1 << w, step):
            val = _plain_run(c, {n: bt for n, bt in zip(a + b, bits(x, w) + bits(y, w))})
            assert value([val[n] for n in lo + hi]) == (signed(x) * signed(y)) % (1 << (2 * w)), (x, y)


def test_program_graph_skeletons():
    """circuits.{bdd_adder, ripple_carry_adder, multiply_then_greater_than}: the Boolean skeletons of the program graphs
    (front ends passed through) compute a + b and (a * b mod 2^w, > c) on plaintext bits."""
    from spf_b200.circuits import bdd_adder, multiply_then_greater_than, ripple_carry_adder

    def run(c, in_bits):
        ins = [i for i, n in enumerate(c.nodes) if n[0] == OP["InputGlwe1"]]
        assert len(ins) == len(in_bits)
        val = {}
        for i, (op, arg, src, io) in enumerate(c.nodes):
            if op == OP["InputGlwe1"]:
                val[i] = in_bits[ins.index(i)]
            elif op == OP["CMux"]:
                val[i] = val[src[2]] if val[src[0]] else val[src[1]]
            elif op == OP["Not"]:
                val[i] = 1 - val[src[0]]
            elif op == OP["ZeroGlwe1"]:
                val[i] = 0
            elif op == OP["OneGlwe1"]:
                val[i] = 1
            elif op != OP["OutputGlwe1"]:
                val[i] = val[src[0]]
        return [val[src[0]] for op, arg, src, io in c.nodes if op == OP["OutputGlwe1"]]

    buf = lambda: np.zeros(4096, np.uint64)
    w = 6
    for build in (bdd_adder, ripple_carry_adder):
        c = build([buf() for _ in range(w)], [buf() for _ in range(w)], [buf() for _ in range(w + 1)])
        for a, b in ((13, 50), (63, 63), (0, 0), (32, 31)):
            assert value(run(c, bits(a, w) + bits(b, w))) == a + b, build.__name__
    mk = lambda: [[buf() for _ in range(w)]]
    c = multiply_then_greater_than(mk(), mk(), mk(), mk(), [buf()], 1)
    for a, b, d in ((13, 11, 9), (63, 63, 0), (7, 9, 63), (0, 5, 0)):
        out = run(c, bits(a, w) + bits(b, w) + bits(d, w))
        assert value(out[:w]) == (a * b) % (1 << w) and out[w] == int((a * b) % (1 << w) > d)
