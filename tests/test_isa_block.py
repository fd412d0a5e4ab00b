"""InstructionCache.block(): straight-line instruction sequences over registers lowered into one graph, checked without
a GPU through the plaintext graph interpreter of test_isa_lowering (PlainGraph).  Seeded random blocks at w = 4 drawn
from every instruction and flag, compared with Python integer semantics of sequential execution and with the same
instructions run one at a time through the cache; bootstrap counts and CBS stages of fused graphs; cache keys; and
the checks that reject a malformed block before anything is built."""
import numpy as np
import pytest

from spf_b200 import OP, plan_graph
from spf_b200.circuits import Bit, Reg
from test_isa_lowering import W, _shifted, dec, enc, n_cbs, outs, plain_cache, signed

MASK = (1 << W) - 1
_REL = {"gt": lambda x, y: x > y, "ge": lambda x, y: x >= y, "lt": lambda x, y: x < y, "le": lambda x, y: x <= y}


def semantics(name, args, kw, val):
    """Python integer result of one instruction (before truncation to its result width); val(x) reads a Reg or Bit."""
    if name == "select":
        cond, a, b, _ = args
        return val(b) if val(cond) else val(a)
    a = val(args[0])
    if name in ("neg", "not_", "zext", "sext", "trunc"):
        return {"neg": -a, "not_": ~a, "zext": a, "sext": signed(a), "trunc": a}[name]
    if name in ("shift", "shift_const"):
        k = val(args[1]) if name == "shift" else args[1]
        return _shifted(a, k, *args[3:])
    b = val(args[1])
    if name == "compare":
        x, y = (signed(a), signed(b)) if kw["signed"] else (a, b)
        return int(_REL[args[3]](x, y))
    return {"add": a + b, "sub": a - b, "multiply": a * b, "multiply_signed": signed(a) * signed(b),
            "greater_than": int(a > b), "equal": int(a == b), "not_equal": int(a != b),
            "and_": a & b, "or_": a | b, "xor": a ^ b}[name]


class RandomBlock:
    """A seeded random program: inputs x, y (4 bits) and z (8 bits, read through 4-bit windows); every instruction
    writes a fresh register (a single-bit result: bit 0 of a fresh 1-bit register).  Operands are drawn from every
    fully-available window of every register, so results are re-read, sliced and used as conditions and amounts."""

    def __init__(self, blk, rng):
        self.blk, self.rng = blk, rng
        self.inputs = [blk.reg(W), blk.reg(W), blk.reg(2 * W)]
        self.avail = {b for r in self.inputs for b in r}
        self.results, self.program = [], []
        for _ in range(int(rng.integers(3, 13))):
            self._one()
        k = int(rng.integers(1, len(self.results) + 1))
        self.outputs = [self.results[i] for i in sorted(rng.choice(len(self.results), k, replace=False))]

    def _window(self, n):
        regs = self.inputs + self.results
        cands = [r[i:i + n] for r in regs for i in range(len(r) - n + 1) if all(b in self.avail for b in r[i:i + n])]
        return cands[int(self.rng.integers(len(cands)))]

    def _bit(self):
        return self._window(1)[0]

    def _one(self):
        rng, blk = self.rng, self.blk
        pick = lambda xs: xs[int(rng.integers(len(xs)))]
        name = pick(["add", "sub", "multiply", "multiply_signed", "neg", "greater_than", "compare", "equal",
                     "not_equal", "and_", "or_", "xor", "not_", "shift", "shift_const", "select", "zext", "sext", "trunc"])
        a, kw = self._window(W), {}
        n_out = {"add": W + 1, "sub": pick([W, W + 1]), "zext": pick([W, W + 2, 2 * W]), "sext": pick([W, W + 1, 2 * W]),
                 "trunc": pick(list(range(1, W + 1)))}.get(name, W)
        if name in ("greater_than", "compare", "equal", "not_equal"):
            out = blk.reg(1)
            args = [a, self._window(W), out[0]]
            if name == "compare":
                args.append(pick(sorted(_REL)))
                kw["signed"] = bool(rng.integers(2))
        else:
            out = blk.reg(n_out)
            if name in ("neg", "not_", "zext", "sext", "trunc"):
                args = [a, out]
            elif name == "select":
                args = [self._bit(), a, self._window(W), out]
            elif name in ("shift", "shift_const"):
                right, mode = pick([(False, "logical"), (True, "logical"), (True, "arithmetic"), (False, "rotation"),
                                    (True, "rotation")])
                amount = self._window(int(rng.integers(2, 4))) if name == "shift" else int(rng.integers(0, W + 1))
                args = [a, amount, out, right, mode]
            else:
                args = [a, self._window(W), out]
        getattr(blk, name)(*args, **kw)
        self.program.append((name, args, kw, out))
        self.results.append(out)
        self.avail.update(out)


def _sequential(rb, values):
    """Python integer semantics of the block in program order: bit -> value."""
    bits = {}
    for r, v in zip(rb.inputs, values):
        bits.update((b, (v >> i) & 1) for i, b in enumerate(r))
    val = lambda x: bits[x] if isinstance(x, Bit) else sum(bits[b] << i for i, b in enumerate(x))
    for name, args, kw, out in rb.program:
        v = semantics(name, args, kw, val)
        bits.update((b, (v >> i) & 1) for i, b in enumerate(out))
    return bits


def _one_at_a_time(cache, rb, values):
    """The same instructions through InstructionCache, one graph per instruction, host buffers in between."""
    bufs = {}
    for r, v in zip(rb.inputs, values):
        bufs.update(zip(r, enc(v, len(r))))
    host = lambda x: bufs[x] if isinstance(x, Bit) else [bufs[b] for b in x] if isinstance(x, Reg) else x
    for name, args, kw, out in rb.program:
        o = outs(len(out))
        bufs.update(zip(out, o))
        getattr(cache, name)(*map(host, args), **kw)
    return bufs


@pytest.mark.parametrize("seed", range(40))
def test_random_blocks_match_sequential_semantics_and_the_single_instruction_path(seed):
    rng = np.random.default_rng(seed)
    cache, single = plain_cache(), plain_cache()
    rb = RandomBlock(cache.block(), rng)
    sets = [[int(rng.integers(0, 1 << len(r))) for r in rb.inputs] for _ in range(3)]
    for values in sets:
        want = _sequential(rb, values)
        one = _one_at_a_time(single, rb, values)
        results = {r: outs(len(r)) for r in rb.outputs}
        g = rb.blk.run({r: enc(v, len(r)) for r, v in zip(rb.inputs, values)}, results)
        for r, o in results.items():
            assert dec(o) == sum(want[b] << i for i, b in enumerate(r)) == dec([one[b] for b in r]), (seed, values, r)
    assert (cache.misses, cache.hits) == (1, len(sets) - 1)
    plan_graph(g.circuit)
    # a bit is bootstrapped at most once: no two CircuitBootstrap chains start from the same node
    srcs = [g.circuit.nodes[g.circuit.nodes[g.circuit.nodes[i][2][0]][2][0]][2][0]
            for i in np.flatnonzero(g.circuit.ops == OP["CircuitBootstrap"])]
    assert len(srcs) == len(set(srcs))


def record_mixed(blk, w):
    """A mixed w-bit block that reads a, c and k more than once (also run on encrypted operands by the GPU tests):
    d = a + b, e = a - c with borrow, f = (d mod 2^w) > c signed, g = f ? b : a (an intermediate), m = g * c,
    sh = m << k (encrypted amount), x = sext of the low half of sh.  Returns (inputs, outputs) registers."""
    lg = (w - 1).bit_length()
    a, b, c, k = blk.reg(w), blk.reg(w), blk.reg(w), blk.reg(lg)
    d, e, f, g, m, sh, x = blk.reg(w + 1), blk.reg(w + 1), blk.reg(1), blk.reg(w), blk.reg(w), blk.reg(w), blk.reg(w)
    blk.add(a, b, d)
    blk.sub(a, c, e)
    blk.compare(d[:w], c, f[0], "gt", signed=True)
    blk.select(f[0], a, b, g)
    blk.multiply(g, c, m)
    blk.shift(m, k, sh, False)
    blk.sext(sh[:w // 2], x)
    return [a, b, c, k], [d, e, f, m, sh, x]


def mixed_want(w, a, b, c, k):
    """Integer semantics of record_mixed's outputs, in its order."""
    mask = (1 << w) - 1
    sgn = lambda v, n=w: v - ((v >> (n - 1)) << n)
    d = a + b
    f = int(sgn(d & mask) > sgn(c))
    m = ((b if f else a) * c) & mask
    sh = (m << k) & mask
    return [d, (a - c) % (1 << (w + 1)), f, m, sh, sgn(sh & ((1 << w // 2) - 1), w // 2) & mask]


def mixed_cbs(w):
    """Bootstraps of record_mixed: a, b, c and k once each though a, c and k are read again; then the refreshed d
    (compare), f (select), g (multiply) and m (shift)."""
    return 3 * w + (w - 1).bit_length() + w + 1 + w + w


def test_mixed_block():
    cache = plain_cache()
    blk = cache.block()
    ins, res = record_mixed(blk, W)
    rng = np.random.default_rng(7)
    for vals in [(a, b, c, k) for a in (0, MASK, 8) for b in (1, 7) for c in (0, 9, MASK) for k in (0, 3)] + \
            [tuple(int(x) for x in rng.integers(0, 1 << W, 4) % [16, 16, 16, 4]) for _ in range(20)]:
        o = {r: outs(len(r)) for r in res}
        g = blk.run({r: enc(v, len(r)) for r, v in zip(ins, vals)}, o)
        assert [dec(o[r]) for r in res] == mixed_want(W, *vals), vals
    assert n_cbs(g) == mixed_cbs(W)
    assert cache.misses == 1


def _regs(blk, *widths):
    return [blk.reg(w) for w in widths]


def _run(blk, inputs, outputs, values=None):
    values = values or [0] * len(inputs)
    return blk.run({r: enc(v, len(r)) for r, v in zip(inputs, values)}, {r: outs(len(r)) for r in outputs})


@pytest.mark.parametrize("k", [1, 2, 3, 4])
def test_independent_adds_bootstrap_in_one_stage(k):
    blk = plain_cache().block()
    ins = _regs(blk, *[W] * 2 * k)
    sums = _regs(blk, *[W + 1] * k)
    for i in range(k):
        blk.add(ins[2 * i], ins[2 * i + 1], sums[i])
    g = _run(blk, ins, sums)
    assert n_cbs(g) == 2 * k * W
    level, _ = plan_graph(g.circuit)
    assert len(set(level[g.circuit.ops == OP["CircuitBootstrap"]].tolist())) == 1


def test_a_bit_read_by_two_instructions_is_bootstrapped_once():
    blk = plain_cache().block()
    a, b, c, s, gt = _regs(blk, W, W, W, W + 1, 1)
    blk.add(a, b, s)
    blk.greater_than(a, c, gt[0])
    for x, y, z in ((5, 9, 3), (15, 15, 15), (0, 7, 1)):
        res = {s: outs(W + 1), gt: outs(1)}
        g = blk.run({a: enc(x), b: enc(y), c: enc(z)}, res)
        assert (dec(res[s]), dec(res[gt])) == (x + y, int(x > z))
    assert n_cbs(g) == 3 * W


def test_rewiring_block_has_no_bootstrap():
    blk = plain_cache().block()
    a, b, n, x, sh, ze, se, tr = _regs(blk, W, W, W, W, W, 2 * W, 2 * W, 2)
    blk.not_(a, n)
    blk.xor(n, b, x)
    blk.shift_const(x, 1, sh, True, "arithmetic")
    blk.zext(sh, ze)
    blk.sext(a, se)
    blk.trunc(x[1:], tr)
    for va, vb in ((3, 12), (9, 6), (15, 0)):
        res = {r: outs(len(r)) for r in (x, ze, se, tr)}
        g = blk.run({a: enc(va), b: enc(vb)}, res)
        vx = (~va & MASK) ^ vb
        assert (dec(res[x]), dec(res[ze]), dec(res[se]), dec(res[tr])) == (
            vx, signed(vx) >> 1 & MASK, signed(va) & 0xFF, (vx >> 1) & 3)
    assert n_cbs(g) == 0


def test_sub_then_compare_has_two_cbs_stages():
    blk = plain_cache().block()
    a, b, c, d, lt = _regs(blk, W, W, W, W, 1)
    blk.sub(a, b, d)
    blk.compare(d, c, lt[0], "gt", signed=True)
    g = _run(blk, [a, b, c], [lt])
    level, _ = plan_graph(g.circuit)
    assert len(set(level[g.circuit.ops == OP["CircuitBootstrap"]].tolist())) == 2
    # operand bits of a, b and c, then the w difference bits refreshed for the compare
    assert n_cbs(g) == 4 * W


def _add_cmp(cache, op="gt", with_sum=True):
    blk = cache.block()
    a, b, c, s, f = _regs(blk, W, W, W, W + 1, 1)
    blk.add(a, b, s)
    blk.compare(s[:W], c, f[0], op)
    return blk, [a, b, c], [s, f] if with_sum else [f]


def test_cache_hits_and_misses():
    cache = plain_cache()
    blk, ins, res = _add_cmp(cache)
    g = _run(blk, ins, res, [1, 2, 3])
    assert _run(blk, ins, res, [4, 5, 6]) is g
    assert (cache.misses, cache.hits) == (1, 1)
    blk2, ins2, res2 = _add_cmp(cache)                    # the same block recorded again
    assert _run(blk2, ins2, res2) is g
    assert (cache.misses, cache.hits) == (1, 2)
    blk3, ins3, res3 = _add_cmp(cache, with_sum=False)    # the sum becomes an intermediate
    g3 = _run(blk3, ins3, res3)
    assert g3 is not g and (cache.misses, cache.hits) == (2, 2)
    assert len(g3.circuit) < len(g.circuit)               # no OutputGlwe1 for the sum bits
    _run(*_add_cmp(cache, op="ge"))                       # another flag
    assert (cache.misses, cache.hits) == (3, 2)


def test_bad_blocks_are_rejected_before_anything_is_built():
    cache = plain_cache()

    def double_write():
        blk = cache.block()
        a, b, s = _regs(blk, W, W, W)
        blk.xor(a, b, s)
        blk.not_(a, s)

    def write_after_read():
        blk = cache.block()
        a, b, s, t = _regs(blk, W, W, W, W)
        blk.xor(a, s, t)
        blk.not_(b, s)

    def write_what_it_reads():
        blk = cache.block()
        a, b = _regs(blk, W, W)
        blk.not_(a, a)

    def unbound_input():
        blk = cache.block()
        a, b, s = _regs(blk, W, W, W + 1)
        blk.add(a, b, s)
        _run(blk, [a], [s])

    def output_never_written():
        blk = cache.block()
        a, s, t = _regs(blk, W, W, W)
        blk.not_(a, s)
        _run(blk, [a], [s, t])

    def output_partly_written():
        blk = cache.block()
        a, s = _regs(blk, W, 2 * W)
        blk.not_(a, s[:W])
        _run(blk, [a], [s])

    def written_input():
        blk = cache.block()
        a, s = _regs(blk, W, W)
        blk.not_(a, s)
        _run(blk, [a, s], [s])

    def wrong_length():
        blk = cache.block()
        a, s = _regs(blk, W, W)
        blk.not_(a, s)
        blk.run({a: enc(1, W - 1)}, {s: outs(W)})

    def view_as_key():
        blk = cache.block()
        a, s = _regs(blk, W, W)
        blk.not_(a, s)
        blk.run({a: enc(1)}, {s[:2]: outs(2)})

    def foreign_bit():
        blk, other = cache.block(), cache.block()
        a, s = _regs(blk, W, W)
        blk.not_(other.reg(W), s)

    def shift_too_wide():
        blk = cache.block()
        a, k, s = _regs(blk, 17, 5, 17)
        blk.shift(a, k, s, True)

    def unknown_compare():
        blk = cache.block()
        a, b, f = _regs(blk, W, W, 1)
        blk.compare(a, b, f[0], "eq")

    def register_for_a_bit():
        blk = cache.block()
        a, b, f = _regs(blk, W, W, 1)
        blk.equal(a, b, f)

    bad = [double_write, write_after_read, write_what_it_reads, unbound_input, output_never_written,
           output_partly_written, written_input, wrong_length, view_as_key, foreign_bit, shift_too_wide,
           unknown_compare, register_for_a_bit,
           lambda: cache.block().run({}, {}),                     # an empty block
           lambda: cache.block().reg(0)]
    for call in bad:
        with pytest.raises(ValueError):
            call()
        assert (cache.misses, cache.hits, cache._cache) == (0, 0, {}), call
