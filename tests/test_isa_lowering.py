"""InstructionCache lowering of the Parasol integer instructions, checked without a GPU: the cache's compile step is
replaced by a plaintext interpreter of the graph's Boolean skeleton, so every call goes through the shipped builder and
through the cache's own rebinding (operand-bit / result-bit node maps) and is compared with Python integer semantics,
exhaustively at w = 4.  Plaintext "ciphertexts" carry their bit in coefficient 0."""
import numpy as np
import pytest

from spf_b200 import OP, OPS, plan_graph
from spf_b200.circuits import InstructionCache

W = 4
MASK = (1 << W) - 1
_PASS = {OP[n] for n in ("SampleExtract", "KeyswitchL1toL0", "CircuitBootstrap", "SchemeSwitch")}
_ZERO = {OP[n] for n in OPS if n.startswith("Zero")}
_ONE = {OP[n] for n in OPS if n.startswith("One")}


class PlainGraph:
    """Stands in for CompiledGraph: set_io binds buffers to Input/Output nodes, run() evaluates the graph on the bits in
    coefficient 0 of the bound inputs and writes the result bits the same way.  An unbound io node is an error."""

    def __init__(self, ev, circuit):
        self.circuit = circuit
        self.nodes = list(circuit.nodes)
        self.io = {}

    def set_io(self, node, buf):
        assert OPS[self.nodes[node][0]].startswith(("Input", "Output")), node
        self.io[node] = buf

    def run(self):
        v = [0] * len(self.nodes)
        for i, (op, arg, ins, _) in enumerate(self.nodes):
            if op == OP["InputGlwe1"]:
                v[i] = int(self.io[i][0])
            elif op == OP["OutputGlwe1"]:
                self.io[i][0] = v[ins[0]]
            elif op in _PASS:
                assert op != OP["SampleExtract"] or arg == 0
                v[i] = v[ins[0]]
            elif op == OP["CMux"]:
                v[i] = v[ins[2]] if v[ins[0]] else v[ins[1]]
            elif op == OP["Not"]:
                v[i] = 1 - v[ins[0]]
            elif op == OP["GlweAdd"]:
                v[i] = v[ins[0]] ^ v[ins[1]]
            elif op == OP["MultiplyGgswGlwe"]:  # (glwe, ggsw): the signed multiply's GGSW -> GLWE conversion
                v[i] = v[ins[0]] & v[ins[1]]
            elif op in _ZERO:
                v[i] = 0
            elif op in _ONE:
                v[i] = 1
            else:
                raise AssertionError(f"unexpected node {OPS[op]}")


def plain_cache():
    cache = InstructionCache(None)
    cache._compile = PlainGraph
    return cache


def enc(v, w=W):
    bufs = [np.zeros(4096, np.uint64) for _ in range(w)]
    for i, b in enumerate(bufs):
        b[0] = (v >> i) & 1
    return bufs


def outs(n):
    return [np.zeros(4096, np.uint64) for _ in range(n)]


def dec(bufs):
    return sum(int(b[0]) << i for i, b in enumerate(bufs))


def signed(v, w=W):
    return v - ((v >> (w - 1)) << w)


def n_cbs(g):
    return int((g.circuit.ops == OP["CircuitBootstrap"]).sum())


def check_graph(cache, g, cbs):
    """The graph is the one cached, has `cbs` circuit bootstraps and passes the host planner."""
    assert any(entry[0] is g for entry in cache._cache.values())
    assert n_cbs(g) == cbs, n_cbs(g)
    plan_graph(g.circuit)


PAIRS = [(a, b) for a in range(1 << W) for b in range(1 << W)]


@pytest.mark.parametrize("borrow", [False, True])
def test_sub(borrow):
    cache = plain_cache()
    for a, b in PAIRS:
        o = outs(W + borrow)
        g = cache.sub(enc(a), enc(b), o)
        assert dec(o[:W]) == (a - b) & MASK, (a, b)
        if borrow:
            assert int(o[W][0]) == int(a < b), (a, b)
    check_graph(cache, g, 2 * W)
    assert (cache.misses, cache.hits) == (1, len(PAIRS) - 1)


def test_neg_not_xor_and_or():
    cache = plain_cache()
    for a in range(1 << W):
        o = outs(W)
        check_graph(cache, cache.neg(enc(a), o), W)
        assert dec(o) == (-a) & MASK
        o = outs(W)
        check_graph(cache, cache.not_(enc(a), o), 0)
        assert dec(o) == ~a & MASK
    for a, b in PAIRS:
        for name, want, cbs in (("and_", a & b, 2 * W), ("or_", a | b, 2 * W), ("xor", a ^ b, 0)):
            o = outs(W)
            check_graph(cache, getattr(cache, name)(enc(a), enc(b), o), cbs)
            assert dec(o) == want, (name, a, b)
    assert cache.misses == 5


@pytest.mark.parametrize("op", ["gt", "ge", "lt", "le"])
@pytest.mark.parametrize("is_signed", [False, True])
def test_compare(op, is_signed):
    cache = plain_cache()
    rel = {"gt": lambda x, y: x > y, "ge": lambda x, y: x >= y, "lt": lambda x, y: x < y, "le": lambda x, y: x <= y}[op]
    for a, b in PAIRS:
        o = outs(1)
        g = cache.compare(enc(a), enc(b), o[0], op, signed=is_signed)
        x, y = (signed(a), signed(b)) if is_signed else (a, b)
        assert int(o[0][0]) == int(rel(x, y)), (a, b)
        if op == "gt" and not is_signed:
            gt = outs(1)
            cache.greater_than(enc(a), enc(b), gt[0])
            assert int(gt[0][0]) == int(o[0][0])
    check_graph(cache, g, 2 * W)


def test_equality():
    cache = plain_cache()
    for a, b in PAIRS:
        eq, ne = outs(1), outs(1)
        check_graph(cache, cache.equal(enc(a), enc(b), eq[0]), 2 * W)
        check_graph(cache, cache.not_equal(enc(a), enc(b), ne[0]), 2 * W)
        assert (int(eq[0][0]), int(ne[0][0])) == (int(a == b), int(a != b))


def _shifted(v, k, right, mode):
    if mode == "rotation":
        k %= W
        return ((v >> k) | (v << (W - k))) & MASK if right else ((v << k) | (v >> (W - k))) & MASK
    if mode == "arithmetic":
        return (signed(v) >> min(k, W)) & MASK
    return (v >> k if right else v << k) & MASK if k < W else 0


SHIFTS = [(False, "logical"), (True, "logical"), (True, "arithmetic"), (False, "rotation"), (True, "rotation")]


@pytest.mark.parametrize("right,mode", SHIFTS)
@pytest.mark.parametrize("amount_bits", [2, 3])
def test_shift_by_encrypted_amount(right, mode, amount_bits):
    cache = plain_cache()
    for v in range(1 << W):
        for k in range(1 << amount_bits):
            o = outs(W)
            g = cache.shift(enc(v), enc(k, amount_bits), o, right, mode)
            assert dec(o) == _shifted(v, k, right, mode), (v, k)
    # a rotation reads only the low log2(W) amount bits (the count is mod W): the others are pruned, unbound
    read = 2 if mode == "rotation" else amount_bits
    check_graph(cache, g, W + read)
    ins = cache._cache[("shift", W, amount_bits, right, mode)][1]
    # slots are value then amount, each most significant bit first, as the barrel shifter takes them
    assert [n >= 0 for n in ins] == [True] * W + [False] * (amount_bits - read) + [True] * read
    assert cache.misses == 1


@pytest.mark.parametrize("right,mode", SHIFTS)
def test_shift_by_constant(right, mode):
    cache = plain_cache()
    for k in range(W + 1):
        for v in range(1 << W):
            o = outs(W)
            g = cache.shift_const(enc(v), k, o, right, mode)
            assert dec(o) == _shifted(v, k, right, mode), (v, k)
        check_graph(cache, g, 0)
        _, ins, res = cache._cache[("shift_const", W, k, right, mode)]
        live = sum(n >= 0 for n in ins)
        assert live == (W if mode == "rotation" else W - k + (mode == "arithmetic" and k == W)), (k, ins)
    assert cache.misses == W + 1


def test_select():
    cache = plain_cache()
    for cond in (0, 1):
        for a, b in PAIRS:
            o = outs(W)
            g = cache.select(enc(cond, 1)[0], enc(a), enc(b), o)
            assert dec(o) == (b if cond else a)
    check_graph(cache, g, 1)
    assert (cache.misses, cache.hits) == (1, 2 * len(PAIRS) - 1)


def test_width_casts():
    cache = plain_cache()
    for v in range(1 << W):
        for n in (W, W + 2, 2 * W):
            o = outs(n)
            check_graph(cache, cache.zext(enc(v), o), 0)
            assert dec(o) == v
            o = outs(n)
            check_graph(cache, cache.sext(enc(v), o), 0)
            assert dec(o) == signed(v) & ((1 << n) - 1)
        for n in range(1, W + 1):
            o = outs(n)
            check_graph(cache, cache.trunc(enc(v), o), 0)
            assert dec(o) == v & ((1 << n) - 1)
    # truncation prunes the high operand bits; sign extension has several results read one operand bit
    assert cache._cache[("trunc", W, 1)][1] == [0] + [-1] * (W - 1)
    sext_outs = cache._cache[("sext", W, 2 * W)][2]
    g = cache._cache[("sext", W, 2 * W)][0]
    assert len({g.nodes[n][2][0] for n in sext_outs[W - 1:]}) == 1


def test_add_multiply_and_signed_multiply():
    cache = plain_cache()
    for a, b in PAIRS:
        o = outs(W + 1)
        g_add = cache.add(enc(a), enc(b), o)
        assert dec(o) == a + b
        o = outs(W)
        g_mul = cache.multiply(enc(a), enc(b), o)
        assert dec(o) == (a * b) & MASK
        o = outs(W)
        g_smul = cache.multiply_signed(enc(a), enc(b), o)
        assert dec(o) == (signed(a) * signed(b)) & MASK, (a, b)
    check_graph(cache, g_add, 2 * W)
    check_graph(cache, g_mul, 2 * W)
    # operand bits, then |a| and |b| refreshed, then the low word of |a| * |b| refreshed for the conditional negate
    check_graph(cache, g_smul, 5 * W)
    assert cache.misses == 3


def test_bad_widths_are_rejected_before_anything_is_built():
    cache = plain_cache()
    a, b3 = enc(1), enc(1, 3)
    bad = [
        lambda: cache.sub(a, b3, outs(W)),
        lambda: cache.sub(a, enc(1), outs(W + 2)),
        lambda: cache.sub([], [], outs(1)),
        lambda: cache.add(a, b3, outs(W + 1)),
        lambda: cache.add(a, enc(1), outs(W)),
        lambda: cache.greater_than(a, b3, outs(1)[0]),
        lambda: cache.compare(a, enc(1), outs(1)[0], "eq"),
        lambda: cache.compare(a, b3, outs(1)[0], "lt", signed=True),
        lambda: cache.equal(a, b3, outs(1)[0]),
        lambda: cache.and_(a, enc(1), outs(W - 1)),
        lambda: cache.xor(a, b3, outs(W)),
        lambda: cache.not_([], []),
        lambda: cache.neg(a, outs(W + 1)),
        lambda: cache.select(outs(1)[0], a, b3, outs(W)),
        lambda: cache.shift(a, enc(1, 1), outs(W), True),                  # too few amount bits for 4 bits
        lambda: cache.shift(a, enc(1, 2), outs(W), False, "arithmetic"),
        lambda: cache.shift(enc(1, 6), enc(1, 3), outs(6), True, "rotation"),
        lambda: cache.shift(a, enc(1, 2), outs(W), True, "circular"),
        lambda: cache.shift(enc(1, 17), enc(1, 5), outs(17), True),          # the barrel shifter grows as 2^w
        lambda: cache.shift_const(a, W + 1, outs(W), True),
        lambda: cache.shift_const(a, -1, outs(W), False),
        lambda: cache.shift_const(a, 1, outs(W), False, "arithmetic"),
        lambda: cache.zext(a, outs(W - 1)),
        lambda: cache.sext(a, outs(W - 1)),
        lambda: cache.trunc(a, outs(W + 1)),
        lambda: cache.trunc(a, []),
        lambda: cache.multiply_signed(enc(1, 17), enc(1, 17), outs(17)),
        lambda: cache.multiply_signed(a, enc(1), outs(2 * W)),
        lambda: cache.multiply(enc(1, 24), enc(1, 24), outs(24)),
    ]
    for k, call in enumerate(bad):
        with pytest.raises(ValueError):
            call()
        assert (cache.misses, cache.hits, cache._cache) == (0, 0, {}), k

