"""Plaintext operands (circuits.Plain, Block.const) and the constant folding behind them, checked without a GPU through
the plaintext graph interpreter of test_isa_lowering (PlainGraph): exhaustively at w = 4 every instruction and flag
with the plaintext operand in each position (and all of them plaintext), against Python integer semantics and the same
call on encrypted bits; bootstrap counts against the operand bits the result depends on; no multiplexer left with a
constant selector or equal branches; the constant multiplier of the MUX generator; random blocks with const registers;
the new argument checks; and cache keys per constant."""
import itertools

import numpy as np
import pytest

from spf_b200 import OP, OPS
from spf_b200 import mux_circuits as M
from spf_b200.circuits import Plain, PlainBit
from test_isa_block import RandomBlock, semantics
from test_isa_lowering import W, _shifted, dec, enc, n_cbs, outs, plain_cache, signed

MASK = (1 << W) - 1
_REL = {"gt": lambda x, y: x > y, "ge": lambda x, y: x >= y, "lt": lambda x, y: x < y, "le": lambda x, y: x <= y}
_CONST_GGSW = {OP["ZeroGgsw1"], OP["OneGgsw1"]}


def _shape(name, widths, n_out, call, want, cbs="read"):
    return pytest.param(widths, n_out, call, want, cbs, id=name)


def _shapes():
    """(operand widths, result bits, call(cache, operands, out), integer semantics, bootstraps): bootstraps "read" = one
    per encrypted operand bit the result depends on, "cond" the same for select's condition alone (a and b are only
    rewired), "shift" like "read" but "none" with a plaintext amount (that is shift_const), "none" for the rewiring
    instructions, "signed" for the signed
    multiply, which also refreshes |a| and the unsigned product (at most 3 per encrypted operand bit, none when the result
    reads none)."""
    o1 = lambda out: out[0]
    yield _shape("add", (W, W), W + 1, lambda c, x, o: c.add(*x, o), lambda a, b: a + b)
    for borrow in (0, 1):
        yield _shape(f"sub{'_borrow' if borrow else ''}", (W, W), W + borrow, lambda c, x, o: c.sub(*x, o),
                     lambda a, b, n=W + borrow: (a - b) % (1 << n))
    yield _shape("neg", (W,), W, lambda c, x, o: c.neg(*x, o), lambda a: -a & MASK)
    yield _shape("greater_than", (W, W), 1, lambda c, x, o: c.greater_than(*x, o1(o)), lambda a, b: int(a > b))
    for op in _REL:
        for sg in (False, True):
            yield _shape(f"compare_{op}{'_signed' if sg else ''}", (W, W), 1,
                         lambda c, x, o, op=op, sg=sg: c.compare(*x, o1(o), op, signed=sg),
                         lambda a, b, op=op, sg=sg: int(_REL[op](signed(a), signed(b)) if sg else _REL[op](a, b)))
    yield _shape("equal", (W, W), 1, lambda c, x, o: c.equal(*x, o1(o)), lambda a, b: int(a == b))
    yield _shape("not_equal", (W, W), 1, lambda c, x, o: c.not_equal(*x, o1(o)), lambda a, b: int(a != b))
    yield _shape("and_", (W, W), W, lambda c, x, o: c.and_(*x, o), lambda a, b: a & b)
    yield _shape("or_", (W, W), W, lambda c, x, o: c.or_(*x, o), lambda a, b: a | b)
    yield _shape("xor", (W, W), W, lambda c, x, o: c.xor(*x, o), lambda a, b: a ^ b, "none")
    yield _shape("not_", (W,), W, lambda c, x, o: c.not_(*x, o), lambda a: ~a & MASK, "none")
    yield _shape("multiply", (W, W), W, lambda c, x, o: c.multiply(*x, o), lambda a, b: a * b & MASK)
    yield _shape("multiply_signed", (W, W), W, lambda c, x, o: c.multiply_signed(*x, o),
                 lambda a, b: signed(a) * signed(b) & MASK, "signed")
    yield _shape("select", (1, W, W), W, lambda c, x, o: c.select(x[0] if isinstance(x[0], Plain) else x[0][0], x[1], x[2], o),
                 lambda s, a, b: b if s else a, "cond")
    for right, mode in ((False, "logical"), (True, "logical"), (True, "arithmetic"), (False, "rotation"), (True, "rotation")):
        for k in (2, 3):
            yield _shape(f"shift_{'right' if right else 'left'}_{mode}_{k}", (W, k), W,
                         lambda c, x, o, r=right, m=mode: c.shift(*x, o, r, m),
                         lambda a, s, r=right, m=mode: _shifted(a, s, r, m), "shift")
    for k in range(W + 1):
        yield _shape(f"shift_const_{k}", (W,), W, lambda c, x, o, k=k: c.shift_const(*x, k, o, True, "arithmetic"),
                     lambda a, k=k: _shifted(a, k, True, "arithmetic"), "none")
    yield _shape("zext", (W,), W + 2, lambda c, x, o: c.zext(*x, o), lambda a: a, "none")
    yield _shape("sext", (W,), W + 2, lambda c, x, o: c.sext(*x, o), lambda a: signed(a) & 0x3F, "none")
    yield _shape("trunc", (W,), 2, lambda c, x, o: c.trunc(*x, o), lambda a: a & 3, "none")


def check_folded(g):
    """No CMux left with a constant selector or with one node on both branches."""
    for op, _, (s, lo, hi), _ in g.nodes:
        if op == OP["CMux"]:
            assert g.nodes[s][0] not in _CONST_GGSW and lo != hi


def read_bits(table, widths, enc_pos):
    """The encrypted operand bits the result depends on, from {operand values: result} of one constant."""
    read = 0
    for p in enc_pos:
        for j in range(widths[p]):
            read += any(table[v] != table[v[:p] + (v[p] ^ 1 << j,) + v[p + 1:]] for v in table)
    return read


@pytest.mark.parametrize("widths,n_out,call,want,cbs", list(_shapes()))
def test_every_instruction_with_plaintext_operands(widths, n_out, call, want, cbs):
    cache, encrypted = plain_cache(), plain_cache()
    n = len(widths)
    for plain_pos in (s for r in range(1, n + 1) for s in itertools.combinations(range(n), r)):
        enc_pos = [p for p in range(n) if p not in plain_pos]
        for consts in itertools.product(*[range(1 << widths[p]) for p in plain_pos]):
            table, graph = {}, None
            for evals in itertools.product(*[range(1 << widths[p]) for p in enc_pos]):
                vals = [0] * n
                for p, v in zip(plain_pos + tuple(enc_pos), consts + evals):
                    vals[p] = v
                o, ref = outs(n_out), outs(n_out)
                graph = call(cache, [Plain(v, w) if p in plain_pos else enc(v, w) for p, (v, w) in enumerate(zip(vals, widths))], o)
                call(encrypted, [enc(v, w) for v, w in zip(vals, widths)], ref)
                table[tuple(vals)] = dec(o)
                assert dec(o) == want(*vals) % (1 << n_out) == dec(ref), (plain_pos, vals)
            check_folded(graph.circuit)
            read = read_bits(table, widths, enc_pos)
            if cbs == "signed":
                assert n_cbs(graph) <= 3 * sum(widths[p] for p in enc_pos) * (read > 0), (plain_pos, consts, n_cbs(graph), read)
            else:
                if cbs == "cond":
                    read = read_bits(table, widths, [p for p in enc_pos if p == 0])
                if cbs == "shift" and 1 in plain_pos:
                    cbs = "none"
                assert n_cbs(graph) == (0 if cbs == "none" else read), (plain_pos, consts, n_cbs(graph), read)
    assert encrypted.misses == 1


def test_shift_by_plain_amount_is_shift_const():
    cache = plain_cache()
    for right, mode in (("right", "logical"), ("left", "logical"), ("right", "arithmetic"), ("left", "rotation")):
        for w in (4, 24):
            for k in range(w + 1):
                a = enc(5, w)
                g1 = cache.shift_const(a, k % w if mode == "rotation" else k, outs(w), right == "right", mode)
                g2 = cache.shift(a, Plain(k, max(1, k.bit_length())), outs(w), right == "right", mode)
                assert g1 is g2   # the same cached graph
    # and node for node when built apart; amounts of w and more clear, fill or wrap
    for k, want in ((3, 3), (9, 4), (15, 4)):
        c1, c2 = plain_cache(), plain_cache()
        a = enc(0b1011)
        g1 = c1.shift_const(a, want, outs(W), True, "arithmetic")
        g2 = c2.shift(a, Plain(k, 4), outs(W), True, "arithmetic")
        assert [n[:3] for n in g1.circuit.nodes] == [n[:3] for n in g2.circuit.nodes]
    o = outs(W)
    plain_cache().shift(enc(0b0110), Plain(5, 3), o, False, "rotation")
    assert dec(o) == _shifted(0b0110, 5, False, "rotation")


@pytest.mark.parametrize("n", [16, 32])
def test_const_multiplier(n):
    rng = np.random.default_rng(n)
    for k in [0, 1, (1 << n) - 1, 1 << (n - 1)] + [int(x) for x in rng.integers(0, 1 << n, 2, dtype=np.uint64)]:
        m = M.const_multiplier(n, k)
        assert m.depth() <= n and len(m.inputs) == len(m.outputs) == n
        for x in [0, (1 << n) - 1] + [int(v) for v in rng.integers(0, 1 << n, 10, dtype=np.uint64)]:
            got = m.evaluate([(x >> i) & 1 for i in range(n)])
            assert sum(b << i for i, b in enumerate(got)) == x * k % (1 << n), (k, x)


def test_multiply_by_a_constant_is_shallow():
    cache = plain_cache()
    for w, k in ((16, 12345), (32, 77)):
        o = outs(w)
        x = int(np.random.default_rng(w).integers(0, 1 << w))
        g = cache.multiply(enc(x, w), Plain(k, w), o)
        assert dec(o) == x * k % (1 << w) and n_cbs(g) == w
        o = outs(w)
        g = cache.multiply_signed(Plain(-k, w), enc(x, w), o)
        assert dec(o) == signed(x, w) * -k % (1 << w)
        check_folded(g.circuit)


class ConstBlock(RandomBlock):
    """RandomBlock whose operand windows also come from two const registers."""

    def __init__(self, blk, rng):
        self.consts = [blk.const(W, int(rng.integers(0, 1 << W))), blk.const(2 * W, int(rng.integers(0, 1 << 2 * W)))]
        super().__init__(blk, rng)

    def _window(self, n):
        regs = self.inputs + self.results + self.consts
        avail = self.avail | {b for r in self.consts for b in r}
        cands = [r[i:i + n] for r in regs for i in range(len(r) - n + 1) if all(b in avail for b in r[i:i + n])]
        return cands[int(self.rng.integers(len(cands)))]


@pytest.mark.parametrize("seed", range(30))
def test_random_blocks_with_const_registers(seed):
    rng = np.random.default_rng(1000 + seed)
    cache, single = plain_cache(), plain_cache()
    rb = ConstBlock(cache.block(), rng)
    for values in [[int(rng.integers(0, 1 << len(r))) for r in rb.inputs] for _ in range(3)]:
        want = _sequential_with(rb, values)
        one = _one_at_a_time_with(single, rb, values)
        results = {r: outs(len(r)) for r in rb.outputs}
        g = rb.blk.run({r: enc(v, len(r)) for r, v in zip(rb.inputs, values)}, results)
        for r, o in results.items():
            assert dec(o) == sum(want[b] << i for i, b in enumerate(r)) == dec([one[b] for b in r]), (seed, values, r)
    assert cache.misses == 1
    check_folded(g.circuit)


def _sequential_with(rb, values):
    bits = {b: b.value for r in rb.consts for b in r}
    for r, v in zip(rb.inputs, values):
        bits.update((b, (v >> i) & 1) for i, b in enumerate(r))
    val = lambda x: bits[x] if not hasattr(x, "__len__") else sum(bits[b] << i for i, b in enumerate(x))
    for name, args, kw, out in rb.program:
        v = semantics(name, args, kw, val)
        bits.update((b, (v >> i) & 1) for i, b in enumerate(out))
    return bits


def _one_at_a_time_with(cache, rb, values):
    """test_isa_block._one_at_a_time with the const bits passed as they are (PlainBits are plaintext operand bits)."""
    from spf_b200.circuits import Bit, Reg

    bufs = {b: b for r in rb.consts for b in r}
    for r, v in zip(rb.inputs, values):
        bufs.update(zip(r, enc(v, len(r))))
    host = lambda x: bufs[x] if isinstance(x, (Bit, PlainBit)) else [bufs[b] for b in x] if isinstance(x, Reg) else x
    for name, args, kw, out in rb.program:
        o = outs(len(out))
        bufs.update(zip(out, o))
        getattr(cache, name)(*map(host, args), **kw)
    return bufs


def test_results_of_constants_fold_into_later_instructions():
    """t = 5 + 3 is a constant, so u = t + x bootstraps x alone, and u > 2 bootstraps u; and(x, 0) reads nothing."""
    blk = plain_cache().block()
    x, t, u, gt, z = blk.reg(W), blk.reg(W + 1), blk.reg(W + 1), blk.reg(1), blk.reg(W)
    blk.add(blk.const(W, 5), blk.const(W, 3), t)
    blk.add(t[:W], x, u)
    blk.compare(u[:W], blk.const(W, 2), gt[0], "gt")
    blk.and_(x, Plain(0, W), z)
    for v in range(1 << W):
        res = {u: outs(W + 1), gt: outs(1), z: outs(W)}
        g = blk.run({x: enc(v)}, res)
        assert (dec(res[u]), dec(res[gt]), dec(res[z])) == (8 + v, int((8 + v) & MASK > 2), 0)
    assert n_cbs(g) == 2 * W
    check_folded(g.circuit)


def test_a_graph_of_constants_only():
    cache = plain_cache()
    o = outs(W + 1)
    g = cache.add(Plain(9, W), Plain(12, W), o)
    assert dec(o) == 21 and n_cbs(g) == 0
    assert {OPS[op] for op, *_ in g.circuit.nodes} <= {"ZeroGlwe1", "OneGlwe1", "OutputGlwe1"}


def test_new_argument_errors_are_raised_before_anything_is_built():
    cache = plain_cache()
    a = enc(1)

    def block(*steps):
        def run():
            blk = cache.block()
            x, s, k = blk.reg(W), blk.reg(W), blk.const(W, 3)
            for step in steps:
                step(blk, x, s, k)
        return run

    bad = [
        lambda: Plain(16, W), lambda: Plain(-9, W), lambda: Plain(0, 0), lambda: Plain(1, -1),
        lambda: cache.add(a, Plain(1, W), Plain(0, W + 1)),                   # a plaintext result
        lambda: cache.greater_than(a, Plain(1, W), Plain(0, 1)),
        lambda: cache.not_(a, list(Plain(0, W))),
        lambda: cache.select(Plain(1, 2), a, enc(2), outs(W)),                # a two-bit condition
        lambda: cache.multiply(enc(1, 33), Plain(1, 33), outs(33)),           # 32 bits at most with a constant
        lambda: cache.multiply_signed(Plain(1, 33), enc(1, 33), outs(33)),
        lambda: cache.multiply(enc(1, 20), enc(1, 20), outs(20)),             # encrypted: 16 bits as before
        lambda: cache.multiply(enc(1, 20), Plain(1, 19), outs(20)),
        lambda: cache.shift(enc(1, 20), enc(1, 5), outs(20), True),           # an encrypted amount: 16 bits as before
        lambda: cache.shift(a, Plain(1, 2), outs(W), False, "arithmetic"),
        lambda: cache.shift(a, Plain(1, 2), outs(W), True, "circular"),
        block(lambda b, x, s, k: b.not_(x, k)),                                # writes a const register
        block(lambda b, x, s, k: b.add(x, k, Plain(0, W + 1))),
        block(lambda b, x, s, k: b.not_(x, s), lambda b, x, s, k: b.run({x: enc(1), k: enc(3)}, {s: outs(W)})),
        block(lambda b, x, s, k: b.not_(x, s), lambda b, x, s, k: b.run({x: enc(1)}, {s: outs(W), k: outs(W)})),
        block(lambda b, x, s, k: b.const(0, 0)),
        block(lambda b, x, s, k: b.const(W, 1 << W)),
    ]
    for i, call in enumerate(bad):
        with pytest.raises(ValueError):
            call()
        assert (cache.misses, cache.hits, cache._cache) == (0, 0, {}), i


def test_cache_keys_per_constant():
    cache = plain_cache()
    x = enc(6)
    add = lambda a, b: cache.add(a, b, outs(W + 1))
    g3 = add(x, Plain(3, W))
    assert add(enc(9), Plain(3, W)) is g3 and (cache.misses, cache.hits) == (1, 1)    # same constant, same place: hit
    assert add(x, Plain(4, W)) is not g3 and cache.misses == 2                         # another constant
    assert add(Plain(3, W), x) is not g3 and cache.misses == 3                         # the same constant elsewhere
    g15 = add(x, Plain(15, W))
    assert add(x, Plain(-1, W)) is g15 and cache.hits == 2                             # -1 is 15 in four bits
    add(x, enc(3))                                                                     # encrypted: the unchanged key
    assert ("add", W) in cache._cache and cache.misses == 5
    g = cache.shift_const(x, 2, outs(W), True)
    assert cache.shift(x, Plain(2, 3), outs(W), True) is g and cache.hits == 3         # shift_const's graph
    blk = cache.block()
    a, s = blk.reg(W), blk.reg(W + 1)
    blk.add(a, blk.const(W, 3), s)
    g = blk.run({a: enc(1)}, {s: outs(W + 1)})
    blk2 = cache.block()
    a2, s2 = blk2.reg(W), blk2.reg(W + 1)
    blk2.add(a2, Plain(3, W), s2)                                                      # a const register is a Plain
    assert blk2.run({a2: enc(2)}, {s2: outs(W + 1)}) is g
    blk3 = cache.block()
    a3, s3 = blk3.reg(W), blk3.reg(W + 1)
    blk3.add(a3, blk3.const(W, 5), s3)
    assert blk3.run({a3: enc(2)}, {s3: outs(W + 1)}) is not g
    assert (cache.misses, cache.hits) == (8, 4)
