"""Program-level circuits.  Two families:
* hand-built ripple MUX chains (ripple_carry_adder, add_then_greater_than): compact adders/comparators
  with the same front end as FheCircuit::insert_mux_circuit_and_connect_inputs (fhe_circuit.rs:473-494):
  per input bit InputGlwe1 -> SampleExtract(0) -> KeyswitchL1toL0 -> CircuitBootstrap, then CMux / Not /
  ZeroGlwe1 / OneGlwe1 nodes and one OutputGlwe1 per result bit; functionally equivalent to, but not
  node-for-node, the reference's BDD-derived trees;
* BDD-derived circuits through spf_b200.mux_circuits (multiply_then_greater_than): the reference's own
  constructions (mux_circuits/src/*.rs), generated natively."""
from __future__ import annotations

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


def _refresh(c: FheCircuit, glwe_node: int) -> int:
    """Turn a computed GLWE bit back into a selector: SampleExtract(0) -> KeyswitchL1toL0 ->
    CircuitBootstrap, the hop between two dependency levels of a Parasol program."""
    x = c.add("SampleExtract", glwe_node, arg=0)
    x = c.add("KeyswitchL1toL0", x)
    return c.add("CircuitBootstrap", x)


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


class InstructionCache:
    """Graph-generation cache (SURVEY.md 8(f).3): one compiled, levelised, device-resident graph per
    (instruction, width), re-bound to the operands of each invocation with CompiledGraph.set_io
    instead of rebuilding the MUX circuit and re-levelising it per dispatch as
    FheCircuit::insert_mux_circuit_and_connect_inputs (fhe_circuit.rs:473-494) does."""

    def __init__(self, evaluation):
        from . import BoxEvaluation, BoxGraph, CompiledGraph

        self._compile = BoxGraph if isinstance(evaluation, BoxEvaluation) else CompiledGraph
        self._ev, self._cache = evaluation, {}
        self.hits = self.misses = 0

    def _run(self, key, build, in_bufs, out_bufs):
        if key not in self._cache:
            self.misses += 1
            c = build()
            ins = [i for i, n in enumerate(c.nodes) if n[0] == 2]    # InputGlwe1, in operand order
            outs = [i for i, n in enumerate(c.nodes) if n[0] == 7]   # OutputGlwe1, in result-bit order
            assert len(ins) == len(in_bufs) and len(outs) == len(out_bufs)
            self._cache[key] = (self._compile(self._ev, c), ins, outs)
        else:
            self.hits += 1
        g, ins, outs = self._cache[key]
        for node, buf in zip(ins + outs, list(in_bufs) + list(out_bufs)):
            g.set_io(node, buf)
        g.run()
        return g

    def add(self, a_bits, b_bits, out_bits):
        """out = a + b (w-bit operands as L1 GLWE bit ciphertexts, w + 1 result bits), blocking."""
        a_bits, b_bits, out_bits = list(a_bits), list(b_bits), list(out_bits)
        return self._run(("add", len(a_bits)), lambda: ripple_carry_adder(a_bits, b_bits, out_bits), a_bits + b_bits, out_bits)

    def _mux_instruction(self, key, mux_builder, operands, out_bits, interleave):
        """One ISA instruction = front end (fhe_circuit.rs:473-494) + one BDD-derived MUX circuit + outputs."""
        from . import mux_circuits as M

        def build():
            c = FheCircuit()
            sels = [[_front(c, x) for x in op] for op in operands]
            order = [x for grp in zip(*sels) for x in grp] if interleave else [x for op in sels for x in op]
            for node, buf in zip(M.insert_mux_circuit(c, mux_builder(), order), out_bits):
                c.add("OutputGlwe1", node, io=buf)
            return M.prune(c, [i for i, n in enumerate(c.nodes) if n[0] == 7])[0]

        return self._run(key, build, [x for op in operands for x in op], out_bits)

    def multiply(self, a_bits, b_bits, out_bits):
        """out = low w bits of a * b, w <= 16 (one multiplier block, parasol_cpu/src/proc/ops/mul.rs:75-117)."""
        from . import mux_circuits as M

        a_bits, b_bits, out_bits = list(a_bits), list(b_bits), list(out_bits)
        w = len(a_bits)
        if w > M.CIRCUIT_CUTOFF or len(b_bits) != w or len(out_bits) != w:
            raise ValueError("InstructionCache.multiply: equal widths up to 16 bits (wider products span two bootstrap levels: "
                             "use circuits.multiply_then_greater_than / mux_circuits.append_uint_multiply)")
        full = lambda: M.unsigned_multiplier(w, w)
        low = lambda: _keep_outputs(full(), w)
        return self._mux_instruction(("mul", w), low, [a_bits, b_bits], out_bits, interleave=False)

    def greater_than(self, a_bits, b_bits, out_bit):
        """out = (a > b), unsigned (comparisons.rs:62-98 with compare_or_maybe_equal(w, true, false))."""
        from . import mux_circuits as M

        a_bits, b_bits = list(a_bits), list(b_bits)
        w = len(a_bits)
        return self._mux_instruction(("gt", w), lambda: M.compare_or_maybe_equal(w, True, False), [a_bits, b_bits], [out_bit], interleave=True)


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
