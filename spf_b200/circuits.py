"""Program-level circuits.  Two families:
* hand-built ripple MUX chains (ripple_carry_adder, add_then_greater_than): compact adders/comparators
  with the same front end as FheCircuit::insert_mux_circuit_and_connect_inputs (fhe_circuit.rs:473-494):
  per input bit InputGlwe1 -> SampleExtract(0) -> KeyswitchL1toL0 -> CircuitBootstrap, then CMux / Not /
  ZeroGlwe1 / OneGlwe1 nodes and one OutputGlwe1 per result bit; functionally equivalent to, but not
  node-for-node, the reference's BDD-derived trees;
* BDD-derived circuits through spf_b200.mux_circuits (multiply_then_greater_than): the reference's own
  constructions (mux_circuits/src/*.rs), generated natively."""
from __future__ import annotations

import weakref

import numpy as np

from . import FheCircuit


def ripple_carry_adder(a_bits: list[np.ndarray], b_bits: list[np.ndarray], out_bits: list[np.ndarray]) -> FheCircuit:
    """a_bits/b_bits: width L1 GLWE ciphertexts (bit in coefficient 0); out_bits: width+1 output
    buffers (sum bits then carry).  Depth: 2 CMUX levels per bit (notes/leveled_computation.md:34)."""
    w = len(a_bits)
    assert len(b_bits) == w and len(out_bits) == w + 1
    c = FheCircuit()

    def front(ct):
        x = c.add("InputGlwe1", io=ct)
        x = c.add("SampleExtract", x, arg=0)
        x = c.add("KeyswitchL1toL0", x)
        return c.add("CircuitBootstrap", x)

    sa = [front(x) for x in a_bits]
    sb = [front(x) for x in b_bits]
    zero, one = c.add("ZeroGlwe1"), c.add("OneGlwe1")
    carry, ncarry = zero, one
    for i in range(w):
        # sum = a ? (b ? c : !c) : (b ? !c : c)
        s0 = c.add("CMux", sb[i], carry, ncarry)   # a = 0: b ? !c : c
        s1 = c.add("CMux", sb[i], ncarry, carry)   # a = 1: b ? c : !c
        s = c.add("CMux", sa[i], s0, s1)
        c.add("OutputGlwe1", s, io=out_bits[i])
        # carry' = a ? (b ? 1 : c) : (b ? c : 0)
        c0 = c.add("CMux", sb[i], zero, carry)
        c1 = c.add("CMux", sb[i], carry, one)
        carry = c.add("CMux", sa[i], c0, c1)
        if i + 1 < w:
            ncarry = c.add("Not", carry)
    c.add("OutputGlwe1", carry, io=out_bits[w])
    return c


def bdd_adder(a_bits: list[np.ndarray], b_bits: list[np.ndarray], out_bits: list[np.ndarray]) -> FheCircuit:
    """The same add with the reference's own MUX circuit: mux_circuits::add::ripple_carry_adder(w, w, false)
    (add.rs:13-56, inputs interleaved a0 b0 a1 b1 ...) expanded by insert_mux_circuit, behind the front end of
    FheCircuit::insert_mux_circuit_and_connect_inputs (fhe_circuit.rs:473-494) -- what parasol_cpu's Add dispatches."""
    from . import mux_circuits as M

    w = len(a_bits)
    assert len(b_bits) == w and len(out_bits) == w + 1
    c = FheCircuit()
    sa = [_front(c, x) for x in a_bits]
    sb = [_front(c, x) for x in b_bits]
    outs = M.insert_mux_circuit(c, M.ripple_carry_adder(w, w, False), [x for pair in zip(sa, sb) for x in pair])
    for node, buf in zip(outs, out_bits):
        c.add("OutputGlwe1", node, io=buf)
    return c


def _front(c: FheCircuit, ct):
    """InputGlwe1 -> SampleExtract(0) -> KeyswitchL1toL0 -> CircuitBootstrap (fhe_circuit.rs:473-494)."""
    x = c.add("InputGlwe1", io=ct)
    x = c.add("SampleExtract", x, arg=0)
    x = c.add("KeyswitchL1toL0", x)
    return c.add("CircuitBootstrap", x)


_SELECTORS: "weakref.WeakKeyDictionary[FheCircuit, dict[int, int]]" = weakref.WeakKeyDictionary()


def _refresh(c: FheCircuit, glwe_node: int) -> int:
    """Turn a computed GLWE bit back into a selector: SampleExtract(0) -> KeyswitchL1toL0 ->
    CircuitBootstrap, the hop between two dependency levels of a Parasol program.  Memoised per circuit: a GLWE node
    read by several MUX circuits (a register bit read by several instructions of a Block) is bootstrapped once."""
    memo = _SELECTORS.setdefault(c, {})
    if glwe_node not in memo:
        x = c.add("SampleExtract", glwe_node, arg=0)
        x = c.add("KeyswitchL1toL0", x)
        memo[glwe_node] = c.add("CircuitBootstrap", x)
    return memo[glwe_node]


def _adder_nodes(c: FheCircuit, sa: list[int], sb: list[int]) -> list[int]:
    """Ripple-carry MUX tree over selector nodes; returns the GLWE nodes of the w sum bits + carry."""
    zero, one = c.add("ZeroGlwe1"), c.add("OneGlwe1")
    carry, ncarry = zero, one
    outs = []
    for i in range(len(sa)):
        s0 = c.add("CMux", sb[i], carry, ncarry)
        s1 = c.add("CMux", sb[i], ncarry, carry)
        outs.append(c.add("CMux", sa[i], s0, s1))
        c0 = c.add("CMux", sb[i], zero, carry)
        c1 = c.add("CMux", sb[i], carry, one)
        carry = c.add("CMux", sa[i], c0, c1)
        if i + 1 < len(sa):
            ncarry = c.add("Not", carry)
    outs.append(carry)
    return outs


def _greater_than_node(c: FheCircuit, sx: list[int], sy: list[int]) -> int:
    """x > y over selector nodes, LSB first: gt' = (x_i == y_i) ? gt : x_i, one ripple MUX chain
    (the comparison the reference derives from a BDD, parasol_cpu/src/proc/ops/comparisons.rs:62-98)."""
    zero, one = c.add("ZeroGlwe1"), c.add("OneGlwe1")
    gt = zero
    for i in range(len(sx)):
        lo = c.add("CMux", sy[i], gt, zero)   # x_i = 0: y_i ? 0 : gt
        hi = c.add("CMux", sy[i], one, gt)    # x_i = 1: y_i ? gt : 1
        gt = c.add("CMux", sx[i], lo, hi)
    return gt


def add_then_greater_than(a_bits, b_bits, c_bits, out_sum, out_gt, programs: int = 1) -> FheCircuit:
    """`programs` independent two-level Parasol-style programs in ONE graph: s = a + b (w-bit,
    wrapping), then s > c.  Level structure per program: 3w circuit bootstraps of the encrypted
    inputs, w more of the sum bits between the two instructions (the shape of BASELINE config 4's
    multi-instruction programs; the multiplier's BDD generator itself is above the boundary and out
    of scope).  a_bits/b_bits/c_bits: [programs][w] L1 GLWE inputs; out_sum [programs][w],
    out_gt [programs] output buffers."""
    c = FheCircuit()
    for p in range(programs):
        w = len(a_bits[p])
        sa = [_front(c, x) for x in a_bits[p]]
        sb = [_front(c, x) for x in b_bits[p]]
        sc = [_front(c, x) for x in c_bits[p]]
        s = _adder_nodes(c, sa, sb)[:w]
        for i in range(w):
            c.add("OutputGlwe1", s[i], io=out_sum[p][i])
        ss = [_refresh(c, n) for n in s]
        c.add("OutputGlwe1", _greater_than_node(c, ss, sc), io=out_gt[p])
    return c


def multiply_then_greater_than(a_bits, b_bits, c_bits, out_prod, out_gt, programs: int = 1) -> FheCircuit:
    """BASELINE config 4's program: p = a * b (w-bit operands, low w bits of the product, the ISA `Mul`
    of parasol_cpu/src/proc/ops/mul.rs:75-117), then p > c (`CmpGt`, ops/comparisons.rs:62-98 with
    compare_or_maybe_equal(w, greater, !or_equal)).  The MUX circuits are the BDD-derived ones of
    spf_b200.mux_circuits (16x16 multiplier blocks + grade-school reduction for w > 16), the high word is
    pruned as the reference does (mul.rs:106-108).  Dependency levels of circuit bootstraps for w = 32:
    3w inputs | the partial-product bits entering the reduction | w product bits entering the compare.
    a_bits/b_bits/c_bits: [programs][w] L1 GLWE inputs; out_prod [programs][w], out_gt [programs]."""
    from . import mux_circuits as M

    c = FheCircuit()
    keep = []
    for p in range(programs):
        w = len(a_bits[p])
        sa = [_front(c, x) for x in a_bits[p]]
        sb = [_front(c, x) for x in b_bits[p]]
        sc = [_front(c, x) for x in c_bits[p]]
        lo, _hi = M.append_uint_multiply(c, sa, sb)
        for i in range(w):
            keep.append(c.add("OutputGlwe1", lo[i], io=out_prod[p][i]))
        sp = [_refresh(c, n) for n in lo]
        cmp_inputs = [x for pair in zip(sp, sc) for x in pair]  # a0 b0 a1 b1 ... (comparisons.rs:127-141)
        (gt,) = M.insert_mux_circuit(c, M.compare_or_maybe_equal(w, True, False), cmp_inputs)
        keep.append(c.add("OutputGlwe1", gt, io=out_gt[p]))
    return M.prune(c, keep)[0]


class PlainBit:
    """One plaintext bit (`value` 0 or 1): a bit of a Plain operand or of a Block.const register."""

    __slots__ = ("value",)

    def __init__(self, value: int):
        self.value = value

    def __repr__(self) -> str:
        return f"plain({self.value})"


_PLAIN_BITS = (PlainBit(0), PlainBit(1))


class Plain:
    """A plaintext operand: `value` as `width` bits, least significant first like every other operand.  Every instruction
    takes it in place of an operand bit list (a one-bit Plain also as select's cond); its bits enter the graph as
    trivial ZeroGlwe1 / OneGlwe1 and are folded out of the circuit (mux_circuits.fold_constants), so they are never
    bootstrapped and the multiplexers they decide disappear.  value: 0 <= value < 2^width, or a two's-complement
    negative value >= -2^(width - 1)."""

    __slots__ = ("value", "width", "bits")

    def __init__(self, value: int, width: int):
        value, width = int(value), int(width)
        if width < 1:
            raise ValueError(f"Plain: width {width}, expected at least 1")
        if not -(1 << (width - 1)) <= value < 1 << width:
            raise ValueError(f"Plain: value {value} does not fit in {width} bits")
        self.value, self.width = value % (1 << width), width
        self.bits = tuple(_PLAIN_BITS[(self.value >> i) & 1] for i in range(width))

    def __len__(self) -> int:
        return self.width

    def __iter__(self):
        return iter(self.bits)

    def __getitem__(self, i):
        return self.bits[i]

    def __repr__(self) -> str:
        return f"Plain({self.value}, {self.width})"


def _is_plain(bits) -> bool:
    """Whether every bit of an operand is plaintext."""
    return all(isinstance(b, PlainBit) for b in bits)


def _plain_value(bits) -> int:
    return sum(b.value << i for i, b in enumerate(bits))


def _program_graph(inputs, program, outputs) -> tuple[FheCircuit, list[int], list[int]]:
    """A straight-line program as one graph: an InputGlwe1 per input bit, then for every instruction
    `body(c, operand_nodes)` -> the GLWE node behind each of its result bits, an OutputGlwe1 per output bit, pruned to
    what the outputs read (fhe_circuit.rs:516-555).  Bits are any hashable names; a PlainBit operand enters as a
    ZeroGlwe1 / OneGlwe1, and a graph with such bits is constant-folded before it is pruned.  inputs / outputs: (bit,
    buffer) pairs; program: (body, operand bits as a list of lists, result bits).  Returns (graph, input-bit nodes,
    output-bit nodes) in the order of inputs / outputs; an input bit no output reads has node -1."""
    from . import mux_circuits as M

    c = FheCircuit()
    ins = [c.add("InputGlwe1", io=buf) for _, buf in inputs]
    node = {bit: n for (bit, _), n in zip(inputs, ins)}
    plain = False
    for body, operands, results in program:
        for b in (b for op in operands for b in op if isinstance(b, PlainBit) and b not in node):
            node[b], plain = c.add("OneGlwe1" if b.value else "ZeroGlwe1"), True
        res = body(c, [[node[b] for b in op] for op in operands])
        assert len(res) == len(results)
        node.update(zip(results, res))
    outs = [c.add("OutputGlwe1", node[bit], io=buf) for bit, buf in outputs]
    if plain:
        c, ren = M.fold_constants(c)
        ins, outs = [ren[n] for n in ins], [ren[n] for n in outs]
    c, ren = M.prune(c, outs)
    return c, [ren.get(n, -1) for n in ins], [ren[n] for n in outs]


def _instruction_graph(operands, out_bits, body) -> tuple[FheCircuit, list[int], list[int]]:
    """One instruction as a graph: every encrypted operand bit is an input of its own (so the same buffer passed twice
    is read through two InputGlwe1 nodes) and every result bit an output.  operands: lists of bit ciphertexts or
    PlainBits.  Returns (graph, encrypted operand-bit nodes, result-bit nodes), both in the flattened order of operands
    / out_bits."""
    names, inputs = [], []
    for op in operands:
        names.append([])
        for x in op:
            if not isinstance(x, PlainBit):
                inputs.append((len(inputs), x))
            names[-1].append(x if isinstance(x, PlainBit) else len(inputs) - 1)
    results = [("result", i) for i in range(len(out_bits))]
    return _program_graph(inputs, [(body, names, results)], list(zip(results, out_bits)))


def _fronts(c: FheCircuit, inputs: list[list[int]]) -> list[list[int]]:
    """The front end of fhe_circuit.rs:473-494 on every input node: one circuit bootstrap per operand bit."""
    return [[_refresh(c, x) for x in op] for op in inputs]


_COMPARE = {"gt": (True, False), "ge": (True, True), "lt": (False, False), "le": (False, True)}  # (greater, or_equal)
_SHIFT_MODES = ("logical", "rotation", "arithmetic")
# The barrel shifter's BDD orders the value bits above the amount bits (bitshift.rs), so its size grows as 2^w: 16 bits
# is 196 588 multiplexers, 20 bits 3.2 million, 32 bits cannot be built.
SHIFT_MAX_WIDTH = 16
# lookup: a k-bit index reads 2^k table entries, one polynomial of N = 2048 coefficients per 2^11 entries and result
# bit above 11 index bits, so 16 index bits with 16 result bits copy 16 MiB of table per run
LOOKUP_MAX_INDEX_BITS = 16
LOOKUP_MAX_RESULT_BITS = 64
# select_n: one CMux tree of 2^k - 1 multiplexers per result bit over 2^k encrypted entries
SELECT_N_MAX_INDEX_BITS = 8


def _operands(name: str, *ops, equal: bool = True) -> list[list]:
    ops = [list(op) for op in ops]
    if any(not op for op in ops):
        raise ValueError(f"InstructionCache.{name}: empty operand")
    if equal and len({len(op) for op in ops}) > 1:
        raise ValueError(f"InstructionCache.{name}: operand widths differ ({', '.join(str(len(op)) for op in ops)})")
    return ops


def _results(name: str, out_bits, *allowed: int) -> list:
    out = list(out_bits)
    if len(out) not in allowed:
        raise ValueError(f"InstructionCache.{name}: {len(out)} result bits, expected {' or '.join(map(str, allowed))}")
    return out


def _check_results(name: str, out_bits) -> None:
    if any(isinstance(b, (Plain, PlainBit)) for b in out_bits):
        raise ValueError(f"{name}: a plaintext (Plain or a const register) cannot take a result")


def _bit(name: str, bit):
    """A single-bit operand: a ciphertext, a register bit, a PlainBit, or a one-bit Plain."""
    if isinstance(bit, Plain):
        if bit.width != 1:
            raise ValueError(f"InstructionCache.{name}: a {bit.width}-bit Plain where one bit is expected")
        return bit.bits[0]
    return bit


def _plain_key(key, operands):
    """The cache key of a call: with plaintext operand bits, which bits they are and their values are part of it."""
    if not any(isinstance(b, PlainBit) for op in operands for b in op):
        return key
    return key + (tuple(tuple(b.value if isinstance(b, PlainBit) else None for b in op) for op in operands),)


def _table_values(table, m: int) -> np.ndarray:
    """A lookup table's entries as uint64 values mod 2^m; every entry must be an integer in Plain(value, m)'s range."""
    lo, hi = -(1 << (m - 1)), 1 << m
    arr = table if isinstance(table, np.ndarray) else np.asarray(table)
    if arr.ndim != 1:
        raise ValueError(f"InstructionCache.lookup: the table must be a sequence of integers, got shape {arr.shape}")
    if arr.dtype.kind in "iub":   # vectorised: the 2^16 entries of a 16-bit table are checked in well under a millisecond
        if len(arr) and not (lo <= int(arr.min()) and int(arr.max()) < hi):
            bad = next(v for v in arr.tolist() if not lo <= v < hi)
            raise ValueError(f"InstructionCache.lookup: entry {bad} does not fit in {m} bits")
        return arr.astype(np.uint64) & np.uint64((1 << m) - 1)
    if isinstance(table, np.ndarray):
        raise ValueError(f"InstructionCache.lookup: table entries must be integers, got dtype {arr.dtype}")
    values = []
    for v in table:   # entries numpy cannot hold in one integer dtype (2^63 and over next to negative values)
        if not isinstance(v, (int, np.integer)):
            raise ValueError(f"InstructionCache.lookup: table entry {v!r} is not an integer")
        if not lo <= int(v) < hi:
            raise ValueError(f"InstructionCache.lookup: entry {int(v)} does not fit in {m} bits")
        values.append(int(v) % (1 << m))
    return np.array(values, np.uint64)


def _lookup_layout(k: int, m: int, log_n: int) -> tuple[int, int, int]:
    """(stride s, groups, polynomials per group) of a k-bit -> m-bit table in polynomials of 2^log_n coefficients: entry
    i, result bit g * s + r is coefficient i * s + r of group g's polynomial, with s the smallest power of two >= m when
    k + log2(s) <= log_n, else the largest that fits; above log_n index bits s = 1 and each of the m groups (result bits)
    takes 2^(k - log_n) polynomials, polynomial h holding entries [h * 2^log_n, (h + 1) * 2^log_n)."""
    s = 1 << (m - 1).bit_length()
    if k + s.bit_length() - 1 > log_n:
        s = 1 << max(0, log_n - k)
    return s, -(-m // s), 1 << max(0, k - log_n)


def _table_bodies(values: np.ndarray, k: int, m: int, s: int, groups: int, per_group: int) -> np.ndarray:
    """The body coefficients (bits, 0 / 1) of every table polynomial, [groups * per_group, entries per polynomial * s] in
    the order group, then polynomial of the group; entries past len(values) read as 0."""
    padded = np.zeros(1 << k, np.uint64)
    padded[:len(values)] = values
    bits = np.zeros((1 << k, groups * s), np.uint64)
    bits[:, :m] = (padded[:, None] >> np.arange(m, dtype=np.uint64)) & np.uint64(1)
    e = (1 << k) // per_group
    return bits.reshape(per_group, e, groups, s).transpose(2, 0, 1, 3).reshape(groups * per_group, e * s)


_TABLES: "weakref.WeakKeyDictionary[FheCircuit, dict[tuple, list[int]]]" = weakref.WeakKeyDictionary()


def _lookup_nodes(c: FheCircuit, key, values: np.ndarray, sels: list[int], m: int, params, zeros) -> list[int]:
    """Vertical packing of a plaintext table behind the selectors `sels` (index bits, LSB first): the table as trivial
    GLWE polynomials (InputGlwe1 nodes whose buffers, from zeros(shape), the graph owns; memoised per circuit by `key`,
    so two lookups of one table in a block share them), a CMux tree on the index bits above log2 N, then per index bit j
    acc = CMux(x_j, acc, acc * X^(-2^j s)), and every result bit rotated to coefficient 0.  The coefficient read never
    wraps, and at the q/2 bit encoding a negacyclic sign flip is the identity anyway.  Returns the GLWE nodes of the m
    result bits."""
    n, gk = params.glwe_n, params.glwe_k
    log_n, k = n.bit_length() - 1, len(sels)
    s, groups, per_group = _lookup_layout(k, m, log_n)
    memo = _TABLES.setdefault(c, {})
    if key not in memo:
        bodies = _table_bodies(values, k, m, s, groups, per_group)
        polys = zeros((groups * per_group, (gk + 1) * n))
        polys[:, gk * n:gk * n + bodies.shape[1]] = bodies << np.uint64(63)
        memo[key] = [c.add("InputGlwe1", io=p) for p in polys]
    polys = memo[key]
    res = []
    for g in range(groups):
        level = polys[g * per_group:(g + 1) * per_group]
        for sel in sels[log_n:]:   # polynomial h = x >> log_n: index bit log_n at the leaves
            level = [c.add("CMux", sel, level[i], level[i + 1]) for i in range(0, len(level), 2)]
        acc = level[0]
        for j, sel in enumerate(sels[:log_n]):
            acc = c.add("CMux", sel, acc, c.add("MulXN", acc, arg=2 * n - (s << j)))
        res += [acc if r == 0 else c.add("MulXN", acc, arg=2 * n - r) for r in range(min(s, m - g * s))]
    return res


class _Instructions:
    """The Parasol integer instructions, shared by InstructionCache (one graph per call) and Block (one graph per
    block).  Each method checks its arguments (ValueError), then hands `self._run(key, body, operands, out_bits)` the
    cache key of its shape and flags, its body -- body(c, operand_nodes) -> the GLWE node behind every result bit -- and
    its operand and result bits."""

    def _mux_instruction(self, key, mux_builder, operands, out_bits, interleave):
        """One ISA instruction = front end (fhe_circuit.rs:473-494) + one BDD-derived MUX circuit whose first
        len(out_bits) outputs are the results.  MUX inputs: the operands' selectors one operand after the other, or
        interleaved a0 b0 a1 b1 ..."""
        from . import mux_circuits as M

        def body(c, ins):
            sels = _fronts(c, ins)
            order = [x for grp in zip(*sels) for x in grp] if interleave else [x for op in sels for x in op]
            return M.insert_mux_circuit(c, mux_builder(), order)[:len(out_bits)]

        return self._run(key, body, operands, out_bits)

    def add(self, a_bits, b_bits, out_bits):
        """out = a + b (w-bit operands, w + 1 result bits: the last is the carry)."""
        a, b = _operands("add", a_bits, b_bits)
        out = _results("add", out_bits, len(a) + 1)
        return self._run(("add", len(a)), lambda c, ins: _adder_nodes(c, *_fronts(c, ins)), [a, b], out)

    def multiply(self, a_bits, b_bits, out_bits):
        """out = low w bits of a * b, w <= 16 (one multiplier block, parasol_cpu/src/proc/ops/mul.rs:75-117).  With a
        Plain operand, w <= 32 and the circuit is the constant multiplier (mux_circuits.const_multiplier, depth <= w) on
        the other operand."""
        from . import mux_circuits as M

        a_bits, b_bits, out_bits = list(a_bits), list(b_bits), list(out_bits)
        w = len(a_bits)
        plain = _is_plain(a_bits) or _is_plain(b_bits)
        if w > (32 if plain else M.CIRCUIT_CUTOFF) or len(b_bits) != w or len(out_bits) != w:
            raise ValueError("InstructionCache.multiply: equal widths up to 16 bits, 32 with a Plain operand (wider products "
                             "span two bootstrap levels: use circuits.multiply_then_greater_than / mux_circuits.append_uint_multiply)")
        if plain:
            # the constant is b when b is plaintext (a then enters the circuit, and folds if it is plaintext too)
            e, k = (0, _plain_value(b_bits)) if _is_plain(b_bits) else (1, _plain_value(a_bits))
            body = lambda c, ins: M.insert_mux_circuit(c, M.const_multiplier(w, k), _fronts(c, [ins[e]])[0])
            return self._run(("mul", w), body, [a_bits, b_bits], out_bits)
        full = lambda: M.unsigned_multiplier(w, w)
        low = lambda: _keep_outputs(full(), w)
        return self._mux_instruction(("mul", w), low, [a_bits, b_bits], out_bits, interleave=False)

    def greater_than(self, a_bits, b_bits, out_bit):
        """out = (a > b), unsigned (comparisons.rs:62-98 with compare_or_maybe_equal(w, true, false))."""
        from . import mux_circuits as M

        a_bits, b_bits = _operands("greater_than", a_bits, b_bits)
        w = len(a_bits)
        return self._mux_instruction(("gt", w), lambda: M.compare_or_maybe_equal(w, True, False), [a_bits, b_bits], [out_bit], interleave=True)

    # ---- MUX-circuit instructions: one circuit bootstrap per operand bit, then one CMUX level per MUX depth ----
    def sub(self, a_bits, b_bits, out_bits):
        """out = (a - b) mod 2^w; with w + 1 result bits the last one is the borrow (sub.rs:12-49)."""
        from . import mux_circuits as M

        a, b = _operands("sub", a_bits, b_bits)
        w = len(a)
        out = _results("sub", out_bits, w, w + 1)
        return self._mux_instruction(("sub", w, len(out)), lambda: M.full_subtractor(w), [a, b], out, interleave=True)

    def neg(self, a_bits, out_bits):
        """out = -a mod 2^w, two's complement (neg.rs:7-27)."""
        from . import mux_circuits as M

        (a,) = _operands("neg", a_bits)
        w = len(a)
        out = _results("neg", out_bits, w)
        return self._mux_instruction(("neg", w), lambda: M.negator(w), [a], out, interleave=False)

    def compare(self, a_bits, b_bits, out_bit, op: str, signed: bool = False):
        """out = (a op b) for op in "gt" "ge" "lt" "le", unsigned or two's complement (comparisons.rs:79-141)."""
        from . import mux_circuits as M

        if op not in _COMPARE:
            raise ValueError(f"InstructionCache.compare: op {op!r}, expected one of {sorted(_COMPARE)}")
        a, b = _operands("compare", a_bits, b_bits)
        w, signed = len(a), bool(signed)
        gen = M.compare_or_maybe_equal_signed if signed else M.compare_or_maybe_equal
        return self._mux_instruction(("cmp", w, op, signed), lambda: gen(w, *_COMPARE[op]), [a, b], [out_bit], interleave=True)

    def equal(self, a_bits, b_bits, out_bit):
        """out = (a == b) (comparisons.rs, compare_equal)."""
        from . import mux_circuits as M

        a, b = _operands("equal", a_bits, b_bits)
        w = len(a)
        return self._mux_instruction(("eq", w), lambda: M.compare_equal(w), [a, b], [out_bit], interleave=True)

    def not_equal(self, a_bits, b_bits, out_bit):
        """out = (a != b) (comparisons.rs, compare_not_equal)."""
        from . import mux_circuits as M

        a, b = _operands("not_equal", a_bits, b_bits)
        w = len(a)
        return self._mux_instruction(("ne", w), lambda: M.compare_not_equal(w), [a, b], [out_bit], interleave=True)

    def and_(self, a_bits, b_bits, out_bits):
        """out = a & b (make_and_circuit)."""
        from . import mux_circuits as M

        a, b = _operands("and_", a_bits, b_bits)
        w = len(a)
        out = _results("and_", out_bits, w)
        return self._mux_instruction(("and", w), lambda: M.make_and_circuit(w), [a, b], out, interleave=True)

    def or_(self, a_bits, b_bits, out_bits):
        """out = a | b (make_or_circuit)."""
        from . import mux_circuits as M

        a, b = _operands("or_", a_bits, b_bits)
        w = len(a)
        out = _results("or_", out_bits, w)
        return self._mux_instruction(("or", w), lambda: M.make_or_circuit(w), [a, b], out, interleave=True)

    def shift(self, a_bits, amount_bits, out_bits, right: bool, mode: str = "logical"):
        """out = a shifted by the encrypted amount (bitshift.rs:49-157).  mode "logical" clears the bits shifted in (an
        amount >= w gives 0), "rotation" wraps (power-of-two w; the amount counts mod w), "arithmetic" fills a right
        shift with the sign bit.  w <= 16 (SHIFT_MAX_WIDTH); the amount needs at least ceil(log2(w)) bits (at least 1).
        A Plain amount k is shift_const(a, k) -- min(k, w), or k mod w for a rotation -- with shift_const's rules (any
        width) and its cached graph."""
        from . import mux_circuits as M

        a, amt = _operands("shift", a_bits, amount_bits, equal=False)
        w, k, right = len(a), len(amt), bool(right)
        if _is_plain(amt):
            amount = _plain_value(amt)
            return self.shift_const(a, amount % w if mode == "rotation" else min(amount, w), out_bits, right, mode)
        out = _results("shift", out_bits, w)
        if w > SHIFT_MAX_WIDTH:
            raise ValueError(f"InstructionCache.shift: widths up to {SHIFT_MAX_WIDTH} bits, got {w} "
                             "(a constant amount has no such limit: shift_const)")
        if mode not in _SHIFT_MODES:
            raise ValueError(f"InstructionCache.shift: mode {mode!r}, expected one of {_SHIFT_MODES}")
        if mode == "arithmetic" and not right:
            raise ValueError("InstructionCache.shift: an arithmetic shift is a right shift")
        if mode == "rotation" and w & (w - 1):
            raise ValueError(f"InstructionCache.shift: rotation needs a power-of-two width, got {w}")
        if k < max(1, (w - 1).bit_length()):
            raise ValueError(f"InstructionCache.shift: a {w}-bit value needs at least {max(1, (w - 1).bit_length())} amount bits, got {k}")
        # the barrel shifter takes value and amount bits most significant first, and gives its results so
        return self._mux_instruction(("shift", w, k, right, mode), lambda: M.bitshift(w, k, right, mode),
                                     [a[::-1], amt[::-1]], out[::-1], interleave=False)

    def multiply_signed(self, a_bits, b_bits, out_bits):
        """out = low w bits of the two's-complement product a * b, w <= 16 (circuits/mul.rs:19-73: |a|, |b|, one
        multiplier block, conditional negate; three bootstrap levels).  With a Plain operand c, w <= 32: |a| times |c|
        through the constant multiplier, negated by a's sign (mux_circuits.append_int_multiply_const)."""
        from . import mux_circuits as M

        a, b = _operands("multiply_signed", a_bits, b_bits)
        w = len(a)
        plain = _is_plain(a) or _is_plain(b)
        if w > (32 if plain else M.CIRCUIT_CUTOFF):
            raise ValueError(f"InstructionCache.multiply_signed: widths up to {M.CIRCUIT_CUTOFF} bits (32 with a Plain "
                             f"operand), got {w}")
        out = _results("multiply_signed", out_bits, w)
        if plain:
            e, k = (0, _plain_value(b)) if _is_plain(b) else (1, _plain_value(a))
            k -= (k >> (w - 1)) << w   # two's complement
            body = lambda c, ins: M.append_int_multiply_const(c, _fronts(c, [ins[e]])[0], k)
            return self._run(("mul_signed", w), body, [a, b], out)
        return self._run(("mul_signed", w), lambda c, ins: M.append_int_multiply(c, *_fronts(c, ins))[0], [a, b], out)

    # ---- no MUX circuit ----
    def select(self, cond, a_bits, b_bits, out_bits):
        """out = cond ? b : a, for one encrypted bit `cond`: cond is bootstrapped to a selector, then one CMux per bit.
        A plaintext cond (a one-bit Plain) makes out a copy of a or b."""
        a, b = _operands("select", a_bits, b_bits)
        cond = _bit("select", cond)
        out = _results("select", out_bits, len(a))

        def body(c, ins):
            (sel,), a_, b_ = ins
            sel = _refresh(c, sel)
            return [c.add("CMux", sel, lo, hi) for lo, hi in zip(a_, b_)]

        return self._run(("select", len(a)), body, [[cond], a, b], out)

    # ---- table reads: one circuit bootstrap per index bit, then one CMUX level per index bit ----
    def lookup(self, table, index_bits, out_bits):
        """out = table[x] for the encrypted k-bit index x (LSB first) and a plaintext table: a sequence of Python ints
        or a 1-D integer numpy array, 1 <= len(table) <= 2^k, entries in Plain(value, m)'s range for m = len(out_bits)
        (1 <= m <= 64), entries past len(table) reading as 0; k <= 16 (LOOKUP_MAX_INDEX_BITS).  Circuit bootstrapping
        and vertical packing: the table is packed into trivial GLWE polynomials of N = glwe_n coefficients (the
        evaluation's params, DEFAULT_128 without one), m result bits side by side per entry where k + log2(m) <=
        log2(N), otherwise in groups of result bits with a polynomial each; the index bits are bootstrapped to selectors
        and blind-rotate each polynomial by x, one CMux per index bit -- above log2(N) index bits after a CMux tree that
        picks the polynomial holding x.  Whatever the function: k bootstraps, ceil(m / s) * k CMux nodes for k <= 11
        (s the entries' stride), m * (2^(k - 11) - 1 + 11) above.  The graph owns the table polynomials and copies them
        to the device on every run (32 KiB each: 16 MiB for a 16-bit -> 16-bit table); the cache key holds the table,
        so every table builds a graph of its own.  A Plain index makes the results constants (no bootstrap, no table);
        the plaintext bits of a partly Plain index fold into fixed rotations.  Result bits carry their bit in
        coefficient 0, as every instruction reads it, but their other coefficients hold other table bits: refresh them
        (any instruction does) before they go to circuits.pack."""
        (idx,) = _operands("lookup", index_bits)
        out = list(out_bits)
        k, m = len(idx), len(out)
        if k > LOOKUP_MAX_INDEX_BITS:
            raise ValueError(f"InstructionCache.lookup: index widths up to {LOOKUP_MAX_INDEX_BITS} bits, got {k}")
        if not 1 <= m <= LOOKUP_MAX_RESULT_BITS:
            raise ValueError(f"InstructionCache.lookup: {m} result bits, expected 1 .. {LOOKUP_MAX_RESULT_BITS}")
        if not 1 <= len(table) <= 1 << k:
            raise ValueError(f"InstructionCache.lookup: a table of {len(table)} entries for a {k}-bit index (1 .. {1 << k})")
        values = _table_values(table, m)
        key = ("lookup", k, m, values.tobytes())
        if _is_plain(idx):
            x = _plain_value(idx)
            v = int(values[x]) if x < len(values) else 0
            body = lambda c, ins: [c.add("OneGlwe1" if (v >> i) & 1 else "ZeroGlwe1") for i in range(m)]
        else:
            params, zeros = self._params(), self._host_zeros
            body = lambda c, ins: _lookup_nodes(c, key, values, [_refresh(c, x) for x in ins[0]], m, params, zeros)
        return self._run(key, body, [idx], out)

    def select_n(self, entries, index_bits, out_bits):
        """out = entries[x] for the encrypted k-bit index x (LSB first), k <= 8 (SELECT_N_MAX_INDEX_BITS): entries are
        1 .. 2^k operands of len(out_bits) bits each -- bit lists, registers, Plain values or const registers -- and an
        index past the last entry reads 0.  The index bits are bootstrapped to selectors, the entries are not: one CMux
        tree per result bit with index bit 0 at the leaves (2^k - 1 CMux nodes, k levels).  Missing and Plain entries
        are constants and fold out of the tree."""
        (idx,) = _operands("select_n", index_bits)
        out = list(out_bits)
        k, m = len(idx), len(out)
        if k > SELECT_N_MAX_INDEX_BITS:
            raise ValueError(f"InstructionCache.select_n: index widths up to {SELECT_N_MAX_INDEX_BITS} bits, got {k}")
        if m < 1:
            raise ValueError("InstructionCache.select_n: no result bits")
        entries = [list(e) for e in entries]
        if not 1 <= len(entries) <= 1 << k:
            raise ValueError(f"InstructionCache.select_n: {len(entries)} entries for a {k}-bit index (1 .. {1 << k})")
        if any(len(e) != m for e in entries):
            raise ValueError(f"InstructionCache.select_n: entry widths {[len(e) for e in entries]}, expected {m}")
        missing = [[_PLAIN_BITS[0]] * m] * ((1 << k) - len(entries))

        def body(c, ins):
            sels, res = [_refresh(c, x) for x in ins[0]], []
            for b in range(m):
                level = [e[b] for e in ins[1:]]
                for sel in sels:
                    level = [c.add("CMux", sel, level[i], level[i + 1]) for i in range(0, len(level), 2)]
                res.append(level[0])
            return res

        return self._run(("select_n", k, m), body, [idx] + entries + missing, out)

    def xor(self, a_bits, b_bits, out_bits):
        """out = a ^ b: one GlweAdd per bit (KeylessEvaluation::xor), no bootstrap."""
        a, b = _operands("xor", a_bits, b_bits)
        out = _results("xor", out_bits, len(a))
        return self._run(("xor", len(a)), lambda c, ins: [c.add("GlweAdd", x, y) for x, y in zip(*ins)], [a, b], out)

    def not_(self, a_bits, out_bits):
        """out = ~a: one Not per bit (KeylessEvaluation::not), no bootstrap."""
        (a,) = _operands("not_", a_bits)
        out = _results("not_", out_bits, len(a))
        return self._run(("not", len(a)), lambda c, ins: [c.add("Not", x) for x in ins[0]], [a], out)

    def shift_const(self, a_bits, k: int, out_bits, right: bool, mode: str = "logical"):
        """out = a shifted by the plaintext amount k, 0 <= k <= w: pure rewiring, no bootstrap.  Vacated bits are an
        encrypted-constant zero ("logical"), the sign bit ("arithmetic", right shifts only), or the bits shifted out
        ("rotation")."""
        (a,) = _operands("shift_const", a_bits)
        w, k, right = len(a), int(k), bool(right)
        out = _results("shift_const", out_bits, w)
        if mode not in _SHIFT_MODES:
            raise ValueError(f"InstructionCache.shift_const: mode {mode!r}, expected one of {_SHIFT_MODES}")
        if mode == "arithmetic" and not right:
            raise ValueError("InstructionCache.shift_const: an arithmetic shift is a right shift")
        if not 0 <= k <= w:
            raise ValueError(f"InstructionCache.shift_const: amount {k} outside 0 .. {w}")

        def body(c, ins):
            x, zero = ins[0], None
            res = []
            for i in range(w):
                src = i + k if right else i - k
                if mode == "rotation":
                    res.append(x[src % w])
                elif 0 <= src < w:
                    res.append(x[src])
                elif mode == "arithmetic":
                    res.append(x[w - 1])
                else:
                    zero = zero if zero is not None else c.add("ZeroGlwe1")
                    res.append(zero)
            return res

        return self._run(("shift_const", w, k, right, mode), body, [a], out)

    def zext(self, a_bits, out_bits):
        """out = a zero-extended to len(out_bits) >= w bits: copies and encrypted-constant zeros, no bootstrap."""
        return self._extend("zext", a_bits, out_bits)

    def sext(self, a_bits, out_bits):
        """out = a sign-extended to len(out_bits) >= w bits: copies of the bits and of the sign bit, no bootstrap."""
        return self._extend("sext", a_bits, out_bits)

    def trunc(self, a_bits, out_bits):
        """out = the low len(out_bits) <= w bits of a: copies, no bootstrap."""
        return self._extend("trunc", a_bits, out_bits)

    def _extend(self, name, a_bits, out_bits):
        (a,) = _operands(name, a_bits)
        w = len(a)
        out = list(out_bits)
        if not (1 <= len(out) <= w if name == "trunc" else len(out) >= w):
            raise ValueError(f"InstructionCache.{name}: {len(out)} result bits from a {w}-bit operand")

        def body(c, ins):
            x = ins[0]
            fill = x[w - 1] if name == "sext" else c.add("ZeroGlwe1") if len(out) > w else None
            return [x[i] if i < w else fill for i in range(len(out))]

        return self._run((name, w, len(out)), body, [a], out)


class InstructionCache(_Instructions):
    """Graph-generation cache (SURVEY.md 8(f).3): one compiled, levelised, device-resident graph per
    (instruction, widths, flags), re-bound to the operands of each invocation with CompiledGraph.set_io
    instead of rebuilding the MUX circuit and re-levelising it per dispatch as
    FheCircuit::insert_mux_circuit_and_connect_inputs (fhe_circuit.rs:473-494) does.

    Operands and results are lists of L1 GLWE bit ciphertexts, least significant bit first: host arrays, or
    BoxCiphertext handles on a BoxEvaluation.  Any operand may be a Plain instead: its bits are constants of the graph,
    folded out of the circuit.  The cache key then records which operand bits are plaintext and their values, so every
    distinct constant builds (and caches) a graph of its own, and a call with the same constants in the same places
    hits.  Every method checks its widths before anything is built (ValueError), runs blocking and returns the graph it
    ran.  block() records several instructions and runs them as one graph."""

    def __init__(self, evaluation):
        from . import BoxEvaluation, BoxGraph, CompiledGraph

        self._compile = BoxGraph if isinstance(evaluation, BoxEvaluation) else CompiledGraph
        self._ev, self._cache = evaluation, {}
        self.hits = self.misses = 0

    def block(self) -> "Block":
        """An empty Block whose graphs are cached here."""
        return Block(self)

    def _params(self):
        """The evaluation's params (DEFAULT_128 without an evaluation)."""
        from . import default_128

        return self._ev.params if self._ev is not None else default_128()

    def _host_zeros(self, shape) -> np.ndarray:
        """Zeroed uint64 host memory for buffers a graph owns (lookup tables): one page-locked slab when there is an
        evaluation, so that their copies are DMAs without a registration per buffer."""
        from . import pinned_zeros

        return pinned_zeros(shape) if self._ev is not None else np.zeros(shape, np.uint64)

    def _run(self, key, body, operands, out_bits):
        _check_results(f"InstructionCache.{key[0]}", out_bits)
        return self._cached(_plain_key(key, operands), lambda: _instruction_graph(operands, out_bits, body),
                            [x for op in operands for x in op if not isinstance(x, PlainBit)] + list(out_bits))

    def _cached(self, key, build, bufs):
        """Build (on a miss) the graph of `key` with build() -> (graph, input-bit nodes, output-bit nodes), bind it to
        `bufs` (input bits then output bits) and run it.  Binding goes through the node maps recorded at build time:
        pruning may have removed input bits, and a rewired output may read an input bit directly."""
        if key not in self._cache:
            self.misses += 1
            c, ins, outs = build()
            self._cache[key] = (self._compile(self._ev, c), ins, outs)
        else:
            self.hits += 1
        g, ins, outs = self._cache[key]
        for node, buf in zip(ins + outs, bufs):
            if node >= 0:
                g.set_io(node, buf)
        g.run()
        return g


class Bit:
    """One bit of a Block register (`reg[i]`): pass it where an instruction takes `out_bit` or `cond`."""

    __slots__ = ("block", "reg", "index")

    def __init__(self, block: "Block", reg: int, index: int):
        self.block, self.reg, self.index = block, reg, index

    def __repr__(self) -> str:
        return f"r{self.reg}[{self.index}]"


class Reg:
    """A Block register: an ordered list of bits, least significant first.  Slicing gives a view over the same bits (an
    operand or result of an instruction, not a key of Block.run), indexing gives a Bit."""

    __slots__ = ("bits", "index")

    def __init__(self, bits, index: int | None = None):
        self.bits, self.index = tuple(bits), index   # index: creation order; None for a view

    def __len__(self) -> int:
        return len(self.bits)

    def __iter__(self):
        return iter(self.bits)

    def __getitem__(self, i):
        return Reg(self.bits[i]) if isinstance(i, slice) else self.bits[i]

    def __repr__(self) -> str:
        return f"Reg({list(self.bits)})"


class Block(_Instructions):
    """A straight-line sequence of instructions over registers, run as ONE graph (InstructionCache.block()).

    The instruction methods are InstructionCache's -- same names, argument order, flags and checks -- with registers or
    register views in place of buffer lists; they record the instruction and return nothing.  Every bit is written at
    most once, and an instruction may not write a bit that it or an earlier instruction reads: program order is the
    only order.  run() lowers the whole block into one graph, so the planner batches the bootstraps of independent
    instructions into one launch per stage, intermediates stay in device memory, and a bit read by several
    instructions is bootstrapped once.  A result read by a later instruction goes through the same SampleExtract ->
    KeyswitchL1toL0 -> CircuitBootstrap refresh it would after a round trip through the host.  Operands may also be
    const registers (const()) or Plain values: the block's graph is then constant-folded as a whole, so a result that
    depends on constants only is a constant for the instructions after it; the cache key records the constants."""

    def __init__(self, cache: InstructionCache):
        self._icache, self._regs, self._program = cache, [], []
        self._read, self._written = set(), set()

    def reg(self, width: int) -> Reg:
        """A new register of `width` >= 1 bits."""
        width = int(width)
        if width < 1:
            raise ValueError(f"Block.reg: width {width}, expected at least 1")
        r = len(self._regs)
        self._regs.append(Reg([Bit(self, r, i) for i in range(width)], index=r))
        return self._regs[-1]

    def const(self, width: int, value: int) -> Reg:
        """A read-only register of plaintext bits holding `value` (the range of Plain(value, width)): instructions read
        it like Plain(value, width); writing it, or binding it in run(), raises ValueError."""
        return Reg(Plain(value, width).bits)

    def _params(self):
        return self._icache._params()

    def _host_zeros(self, shape) -> np.ndarray:
        return self._icache._host_zeros(shape)

    def _run(self, key, body, operands, out_bits):
        reads, out = [b for op in operands for b in op], list(out_bits)
        _check_results(f"Block {key[0]}", out)
        for b in reads + out:
            if not isinstance(b, PlainBit) and (not isinstance(b, Bit) or b.block is not self):
                raise ValueError(f"Block {key[0]}: {b!r} is not a bit of this block's registers")
        if len(set(out)) < len(out) or self._written.intersection(out):
            raise ValueError(f"Block {key[0]}: writes a bit a second time")
        if self._read.intersection(out) or set(reads).intersection(out):
            raise ValueError(f"Block {key[0]}: writes a bit that this or an earlier instruction reads")
        self._program.append((key, body, operands, out))
        self._read.update(b for b in reads if isinstance(b, Bit))
        self._written.update(out)

    def _binding(self, name: str, regs) -> list:
        """{Reg: buffers} -> [(register, buffer list)] in register creation order."""
        bound = []
        for r, bufs in dict(regs).items():
            if isinstance(r, Reg) and r.bits and isinstance(r.bits[0], PlainBit):
                raise ValueError(f"Block.run: a const register is plaintext, it cannot be bound in {name}")
            if not isinstance(r, Reg) or r.index is None or r.bits[0].block is not self:
                raise ValueError(f"Block.run: {name} keys must be registers of this block (from reg(), not views)")
            bufs = list(bufs)
            if len(bufs) != len(r):
                raise ValueError(f"Block.run: {name} register r{r.index} has {len(r)} bits, bound to {len(bufs)} buffers")
            bound.append((r, bufs))
        return sorted(bound, key=lambda rb: rb[0].index)

    def run(self, inputs, outputs):
        """Run the block: inputs / outputs are {register: list of L1 GLWE bit ciphertexts} -- host arrays, or
        BoxCiphertext handles on a BoxEvaluation.  Every register read and never written must be an input, every output
        register must be written in full; written registers that are not outputs are intermediates.  The graph is
        built on the cache's first sight of this block's structure and rebound afterwards; returns it."""
        if not self._program:
            raise ValueError("Block.run: empty block")
        ins, outs = self._binding("inputs", inputs), self._binding("outputs", outputs)
        in_regs = {r.index for r, _ in ins}
        for r, _ in ins:
            if self._written.intersection(r):
                raise ValueError(f"Block.run: input register r{r.index} is written by an instruction")
        unbound = sorted({b.reg for b in self._read - self._written} - in_regs)
        if unbound:
            raise ValueError(f"Block.run: registers {['r%d' % r for r in unbound]} are read and never written: bind them in inputs")
        for r, _ in outs:
            if not self._written.issuperset(r):
                raise ValueError(f"Block.run: output register r{r.index} is not written in full")
        name = lambda b: ("plain", b.value) if isinstance(b, PlainBit) else (b.reg, b.index)
        key = ("block",
               tuple((k, tuple(tuple(map(name, op)) for op in operands), tuple(map(name, res))) for k, _, operands, res in self._program),
               tuple(len(r) for r in self._regs), tuple(r.index for r, _ in ins), tuple(r.index for r, _ in outs))
        in_bits = [(b, buf) for r, bufs in ins for b, buf in zip(r, bufs)]
        out_bits = [(b, buf) for r, bufs in outs for b, buf in zip(r, bufs)]
        program = [(body, operands, res) for _, body, operands, res in self._program]
        return self._icache._cached(key, lambda: _program_graph(in_bits, program, out_bits),
                                    [buf for _, buf in in_bits + out_bits])


def _keep_outputs(mux, n_outputs: int):
    """The first n_outputs outputs of a MUX circuit (the unreferenced multiplexers are pruned after expansion)."""
    from . import mux_circuits as M

    keep = mux.op != M.OUTPUT
    keep[mux.outputs[:n_outputs]] = True
    idx = np.flatnonzero(keep)
    new = np.full(len(mux.op), -1, np.int32)
    new[idx] = np.arange(len(idx), dtype=np.int32)
    ren = lambda x: np.where(x[idx] >= 0, new[np.maximum(x[idx], 0)], -1)
    return M.MuxCircuit(mux.op[idx], mux.arg[idx], ren(mux.sel), ren(mux.low), ren(mux.high))


# ---- packing front end (SURVEY.md 8(f).4) --------------------------------------------------------
def pack(c: FheCircuit, bit_nodes: list[int]) -> int:
    """DynamicGenericIntGraphNodes::pack (parasol_runtime/src/fluent/dynamic_generic_int_graph_nodes.rs:
    139-205): bit i (an L1 GLWE with the bit in coefficient 0) is multiplied by X^i (MulXN) and the shifted
    ciphertexts are summed by a GlweAdd tree, so bit i ends up in coefficient i of ONE GLWE."""
    assert len(bit_nodes) > 0
    level = [n if i == 0 else c.add("MulXN", n, arg=i) for i, n in enumerate(bit_nodes)]
    while len(level) > 1:
        nxt = [c.add("GlweAdd", level[i], level[i + 1]) if i + 1 < len(level) else level[i] for i in range(0, len(level), 2)]
        level = nxt
    return level[0]


def unpack(c: FheCircuit, packed_node: int, bit_len: int) -> list[int]:
    """PackedDynamicGenericIntGraphNode::unpack (fluent/packed_dynamic_generic_int_graph_node.rs:24-38):
    SampleExtract(i) of the packed GLWE gives bit i as an L1 LWE."""
    return [c.add("SampleExtract", packed_node, arg=i) for i in range(bit_len)]
