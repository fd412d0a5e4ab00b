"""Table lookups (InstructionCache.lookup, select_n) checked without a GPU: the cache's compile step is replaced by a
plaintext interpreter of the graph that keeps a whole polynomial of bits per GLWE value, so the vertical packing is
checked coefficient by coefficient through the shipped builder and the cache's own rebinding, against Python indexing.
A bound input carries its bit in coefficient 0; a table input is read from the buffer the graph was built with (body
coefficient >> 63); MulXN(e) is the cyclic rotation out[(t + e) mod N] = in[t] (the negacyclic signs vanish at the q/2
bit encoding); CMux, GlweAdd and Not act per coefficient (Not on coefficient 0); the SampleExtract / keyswitch /
circuit-bootstrap chain passes coefficient 0 through."""
import numpy as np
import pytest

from spf_b200 import OP, OPS, default_128, plan_graph
from spf_b200.circuits import InstructionCache, Plain

P = default_128()
N, GK = P.glwe_n, P.glwe_k
LOG_N = N.bit_length() - 1
_PASS = {OP[n] for n in ("SampleExtract", "KeyswitchL1toL0", "CircuitBootstrap")}
_ZERO = {OP[n] for n in OPS if n.startswith("Zero")}
_ONE = {OP[n] for n in OPS if n.startswith("One")}


def _bit0(b):
    v = np.zeros(N, np.uint8)
    v[0] = b
    return v


class PolyGraph:
    """Stands in for CompiledGraph: set_io binds buffers to Input/Output nodes; an unbound InputGlwe1 is a table the
    graph owns and is read from its build-time buffer."""

    def __init__(self, ev, circuit):
        self.circuit = circuit
        self.nodes = list(circuit.nodes)
        self.io = {}

    def set_io(self, node, buf):
        assert OPS[self.nodes[node][0]].startswith(("Input", "Output")), node
        self.io[node] = buf

    def run(self):
        v = [None] * len(self.nodes)
        for i, (op, arg, ins, io) in enumerate(self.nodes):
            if op == OP["InputGlwe1"]:
                v[i] = _bit0(int(self.io[i][0])) if i in self.io else (io[GK * N:(GK + 1) * N] >> np.uint64(63)).astype(np.uint8)
            elif op == OP["OutputGlwe1"]:
                self.io[i][0] = v[ins[0]][0]
            elif op in _PASS:
                assert op != OP["SampleExtract"] or arg == 0
                v[i] = _bit0(v[ins[0]][0])
            elif op == OP["CMux"]:
                v[i] = v[ins[2]] if v[ins[0]][0] else v[ins[1]]
            elif op == OP["MulXN"]:
                v[i] = np.roll(v[ins[0]], arg % N)
            elif op == OP["Not"]:
                v[i] = v[ins[0]].copy()
                v[i][0] ^= 1
            elif op == OP["GlweAdd"]:
                v[i] = v[ins[0]] ^ v[ins[1]]
            elif op in _ZERO:
                v[i] = _bit0(0)
            elif op in _ONE:
                v[i] = _bit0(1)
            else:
                raise AssertionError(f"unexpected node {OPS[op]}")


def poly_cache():
    cache = InstructionCache(None)
    cache._compile = PolyGraph
    return cache


def enc(v, w):
    bufs = [np.zeros(4096, np.uint64) for _ in range(w)]
    for i, b in enumerate(bufs):
        b[0] = (v >> i) & 1
    return bufs


def outs(n):
    return [np.zeros(4096, np.uint64) for _ in range(n)]


def dec(bufs):
    return sum(int(b[0]) << i for i, b in enumerate(bufs))


def count(g, op):
    return int((g.circuit.ops == OP[op]).sum())


def tables(g):
    """The table inputs of a graph: InputGlwe1 nodes never bound through set_io."""
    return [i for i, (op, *_rest) in enumerate(g.nodes) if op == OP["InputGlwe1"] and i not in g.io]


def layout(k, m):
    """(stride, groups, polynomials per group), as the lookup packs a k-bit -> m-bit table."""
    s = 1 << (m - 1).bit_length()
    if k + s.bit_length() - 1 > LOG_N:
        s = 1 << max(0, LOG_N - k)
    return s, -(-m // s), 1 << max(0, k - LOG_N)


def expected_cmux(k, m):
    s, groups, _ = layout(k, m)
    return groups * k if k <= LOG_N else m * ((1 << (k - LOG_N)) - 1 + LOG_N)


def check_lookup_graph(cache, g, k, m, encrypted=None):
    assert any(entry[0] is g for entry in cache._cache.values())
    assert count(g, "CircuitBootstrap") == (k if encrypted is None else encrypted)
    if encrypted is None:
        assert count(g, "CMux") == expected_cmux(k, m)
        s, groups, per_group = layout(k, m)
        assert len(tables(g)) == groups * per_group
    plan_graph(g.circuit)


def random_table(rng, k, m, n=None):
    return [int(v) for v in rng.integers(0, 1 << m, n or (1 << k), dtype=np.uint64)]


@pytest.mark.parametrize("m", [1, 3, 4, 5, 8])
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6])
def test_lookup_exhaustive(k, m):
    cache = poly_cache()
    table = random_table(np.random.default_rng(16 * k + m), k, m)
    for x in range(1 << k):
        o = outs(m)
        g = cache.lookup(table, enc(x, k), o)
        assert dec(o) == table[x], (x, table[x])
    check_lookup_graph(cache, g, k, m)
    assert layout(k, m)[1] == 1   # one polynomial holds every result bit
    assert (cache.misses, cache.hits) == (1, (1 << k) - 1)


@pytest.mark.parametrize("k,m", [(8, 16), (10, 5), (11, 3), (7, 33), (1, 64)])
def test_lookup_split_into_groups(k, m):
    s, groups, _ = layout(k, m)
    assert groups > 1 or s == 64
    cache = poly_cache()
    rng = np.random.default_rng(k * m)
    table = random_table(rng, k, min(m, 63)) if m < 64 else [(1 << 64) - 1, -(1 << 63)]
    xs = range(1 << k) if k <= 8 else [0, (1 << k) - 1] + [int(x) for x in rng.integers(0, 1 << k, 40)]
    for x in xs:
        o = outs(m)
        g = cache.lookup(table, enc(x, k), o)
        assert dec(o) == table[x] % (1 << m), x
    check_lookup_graph(cache, g, k, m)


@pytest.mark.parametrize("k,m", [(12, 1), (12, 3), (16, 16)])
def test_lookup_above_one_polynomial(k, m):
    """More than N entries: a CMux tree on the index bits above log2 N picks the polynomial, then the rotation."""
    cache = poly_cache()
    rng = np.random.default_rng(k + m)
    table = np.asarray(random_table(rng, k, m), np.uint64)
    corners = [0, N - 1, N, 2 * N - 1, (1 << k) - 1]
    for x in corners + [int(x) for x in rng.integers(0, 1 << k, 6)]:
        o = outs(m)
        g = cache.lookup(table, enc(x, k), o)
        assert dec(o) == int(table[x]), x
    check_lookup_graph(cache, g, k, m)
    assert (cache.misses, cache.hits) == (1, len(corners) + 5)


def test_short_tables_read_zero_past_the_end():
    cache = poly_cache()
    rng = np.random.default_rng(7)
    for k, m, n, xs in [(5, 4, 7, range(32)), (3, 8, 1, range(8)), (12, 2, 3000, [0, 2999, 3000, 4095, 2047, 2048])]:
        table = random_table(rng, k, m, n)
        for x in xs:
            o = outs(m)
            g = cache.lookup(table, enc(x, k), o)
            assert dec(o) == (table[x] if x < n else 0), (k, x)
        check_lookup_graph(cache, g, k, m)


def test_signed_entries_are_stored_mod_2_to_the_m():
    cache = poly_cache()
    table = [-8, -1, 7, 0, 3]
    for x in range(8):
        o = outs(4)
        cache.lookup(table, enc(x, 3), o)
        assert dec(o) == (table[x] % 16 if x < len(table) else 0)


def test_plain_index_gives_constants():
    cache = poly_cache()
    table = random_table(np.random.default_rng(3), 4, 5)
    for x in range(16):
        o = outs(5)
        g = cache.lookup(table, Plain(x, 4), o)
        assert dec(o) == table[x]
        ops = {OPS[op] for op in g.circuit.ops}
        assert ops <= {"ZeroGlwe1", "OneGlwe1", "OutputGlwe1"}, ops   # no table input, no bootstrap
    assert cache.misses == 16


@pytest.mark.parametrize("k,m,plain_bits", [(5, 3, (1, 3)), (4, 8, (0,)), (12, 2, (11,)), (12, 1, (0, 11))])
def test_partly_plain_index(k, m, plain_bits):
    """The plaintext index bits fold into fixed rotations (and pick the polynomial above log2 N): one bootstrap and
    one CMux per encrypted index bit and group, and only the polynomials the plaintext bits leave."""
    cache = poly_cache()
    rng = np.random.default_rng(k * 10 + m)
    table = random_table(rng, k, m)
    enc_bits = [j for j in range(k) if j not in plain_bits]
    for fixed in range(1 << len(plain_bits)):
        pv = sum(((fixed >> t) & 1) << j for t, j in enumerate(plain_bits))
        xs = range(1 << k) if k <= 6 else [int(x) for x in rng.integers(0, 1 << k, 12)]
        for x in {(x & ~sum(1 << j for j in plain_bits)) | pv for x in xs}:
            ct = enc(x, k)
            idx = [Plain(pv, k).bits[j] if j in plain_bits else ct[j] for j in range(k)]
            o = outs(m)
            g = cache.lookup(table, idx, o)
            assert dec(o) == table[x], (x, pv)
        _, groups, per_group = layout(k, m)
        low = sum(j < LOG_N for j in enc_bits)
        high = len(enc_bits) - low
        check_lookup_graph(cache, g, k, m, encrypted=len(enc_bits))
        assert count(g, "CMux") == groups * (low + (1 << high) - 1)
        assert len(tables(g)) == groups * (1 << high)
    assert cache.misses == 1 << len(plain_bits)


@pytest.mark.parametrize("n_entries", [8, 5, 1])
def test_select_n_exhaustive(n_entries):
    cache = poly_cache()
    k, m = 3, 4
    rng = np.random.default_rng(n_entries)
    for _ in range(3):
        vals = [int(v) for v in rng.integers(0, 1 << m, n_entries)]
        for x in range(1 << k):
            o = outs(m)
            g = cache.select_n([enc(v, m) for v in vals], enc(x, k), o)
            assert dec(o) == (vals[x] if x < n_entries else 0), (vals, x)
    assert count(g, "CircuitBootstrap") == k
    assert count(g, "CMux") <= m * ((1 << k) - 1)
    if n_entries == 8:
        assert count(g, "CMux") == m * ((1 << k) - 1)
    plan_graph(g.circuit)
    assert (cache.misses, cache.hits) == (1, 3 * (1 << k) - 1)


def test_select_n_with_plain_entries_and_plain_index_bits():
    cache = poly_cache()
    k, m = 3, 5
    rng = np.random.default_rng(11)
    for trial in range(4):
        vals = [int(v) for v in rng.integers(0, 1 << m, 6)]
        plain_at = {1, 4} if trial % 2 else {0, 2, 3, 5}
        entries_for = lambda: [Plain(v, m) if i in plain_at else enc(v, m) for i, v in enumerate(vals)]
        for x in range(1 << k):
            o = outs(m)
            cache.select_n(entries_for(), enc(x, k), o)
            assert dec(o) == (vals[x] if x < 6 else 0), (trial, x)
            # index bit 1 plaintext: the tree folds to the half it picks
            ct = enc(x, k)
            o = outs(m)
            g = cache.select_n(entries_for(), [ct[0], Plain(x, k).bits[1], ct[2]], o)
            assert dec(o) == (vals[x] if x < 6 else 0), (trial, x)
            assert count(g, "CircuitBootstrap") == 2
    # every entry plaintext and a plaintext index: constants only
    o = outs(m)
    g = cache.select_n([Plain(v, m) for v in vals], Plain(4, k), o)
    assert dec(o) == vals[4] and count(g, "CMux") == count(g, "CircuitBootstrap") == 0


def test_block_lookup_add_compare():
    """t = table[x]; s = t + y; f = s[:4] > y -- a lookup result is refreshed like any other result bit."""
    cache = poly_cache()
    table = random_table(np.random.default_rng(5), 4, 4)
    for x in range(16):
        for y in range(16):
            blk = cache.block()
            rx, ry, t, s, f, u = blk.reg(4), blk.reg(4), blk.reg(4), blk.reg(5), blk.reg(1), blk.reg(4)
            blk.lookup(table, rx, t)
            blk.add(t, ry, s)
            blk.compare(s[:4], ry, f[0], "gt")
            blk.lookup(table, ry, u)          # the same table: one set of table inputs
            o = {s: outs(5), f: outs(1), t: outs(4), u: outs(4)}
            g = blk.run({rx: enc(x, 4), ry: enc(y, 4)}, o)
            want_s = table[x] + y
            assert (dec(o[t]), dec(o[s]), dec(o[f]), dec(o[u])) == (table[x], want_s, int(want_s % 16 > y), table[y])
    assert len(tables(g)) == 1
    # x, y and the 4 sum bits the compare reads
    assert count(g, "CircuitBootstrap") == 4 + 4 + 4 + 4
    plan_graph(g.circuit)
    assert (cache.misses, cache.hits) == (1, 255)


def test_block_folds_a_lookup_of_a_const_register():
    cache = poly_cache()
    table = [9, 4, 12, 1]
    blk = cache.block()
    y, t, s = blk.reg(4), blk.reg(4), blk.reg(5)
    blk.lookup(table, blk.const(2, 2), t)
    blk.add(t, y, s)
    for v in (0, 3, 15):
        o = {s: outs(5)}
        g = blk.run({y: enc(v, 4)}, o)
        assert dec(o[s]) == 12 + v
    assert count(g, "CircuitBootstrap") == 4 and not tables(g)


def test_cache_keys():
    cache = poly_cache()
    t1, t2 = [3, 1, 4, 1, 5, 9, 2, 6], [3, 1, 4, 1, 5, 9, 2, 7]
    cache.lookup(t1, enc(2, 3), outs(4))
    cache.lookup(list(t1), enc(5, 3), outs(4))
    cache.lookup(np.asarray(t1, np.int64), enc(1, 3), outs(4))
    assert (cache.misses, cache.hits) == (1, 2)
    cache.lookup(t2, enc(2, 3), outs(4))
    cache.lookup(t1, enc(2, 3), outs(5))
    assert (cache.misses, cache.hits) == (3, 2)
    assert ("lookup", 3, 4, np.asarray(t1, np.uint64).tobytes()) in cache._cache
    # a negative entry is keyed by its value mod 2^m
    cache.lookup([-1, 0], enc(1, 1), outs(4))
    cache.lookup([15, 0], enc(0, 1), outs(4))
    assert (cache.misses, cache.hits) == (4, 3)
    cache.select_n([enc(1, 4)] * 4, enc(1, 2), outs(4))
    cache.select_n([enc(2, 4)] * 4, enc(3, 2), outs(4))
    assert ("select_n", 2, 4) in cache._cache and (cache.misses, cache.hits) == (5, 4)
    cache.select_n([enc(2, 4)] * 3, enc(3, 2), outs(4))   # a missing entry is a constant: a graph of its own
    assert cache.misses == 6
    # blocks: the table is part of the block's key
    for table, miss in ((t1, 7), (t1, 7), (t2, 8)):
        blk = cache.block()
        x, r = blk.reg(3), blk.reg(4)
        blk.lookup(table, x, r)
        blk.run({x: enc(1, 3)}, {r: outs(4)})
        assert cache.misses == miss


def test_bad_arguments_are_rejected_before_anything_is_built():
    cache = poly_cache()
    a3, o4 = enc(1, 3), outs(4)
    bad = [
        lambda: cache.lookup([1], [], o4),                              # empty index
        lambda: cache.lookup([1], enc(1, 17), o4),                      # index wider than 16 bits
        lambda: cache.lookup([1], a3, []),                              # no result bits
        lambda: cache.lookup([1], a3, outs(65)),                        # more than 64 result bits
        lambda: cache.lookup([], a3, o4),                               # empty table
        lambda: cache.lookup([0] * 9, a3, o4),                          # longer than 2^k
        lambda: cache.lookup([16], a3, o4),                             # does not fit 4 bits
        lambda: cache.lookup([-9], a3, o4),                             # below -2^(m - 1)
        lambda: cache.lookup(np.asarray([0, 16]), a3, o4),
        lambda: cache.lookup([0, 1 << 64], enc(1, 1), outs(64)),
        lambda: cache.lookup([0.5], a3, o4),                            # not an integer
        lambda: cache.lookup(np.asarray([0.0]), a3, o4),
        lambda: cache.lookup(np.zeros((2, 2), np.int64), a3, o4),
        lambda: cache.lookup([1], a3, Plain(0, 4)),                     # plaintext result
        lambda: cache.select_n([enc(1, 4)], [], o4),
        lambda: cache.select_n([enc(1, 4)], enc(1, 9), o4),             # index wider than 8 bits
        lambda: cache.select_n([], a3, o4),
        lambda: cache.select_n([enc(1, 4)] * 9, a3, o4),
        lambda: cache.select_n([enc(1, 4), enc(1, 3)], a3, o4),         # unequal widths
        lambda: cache.select_n([enc(1, 3)], a3, o4),
        lambda: cache.select_n([enc(1, 4)], a3, []),
        lambda: cache.select_n([enc(1, 4)], a3, Plain(1, 4)),
    ]
    for i, call in enumerate(bad):
        with pytest.raises(ValueError):
            call()
        assert (cache.misses, cache.hits, cache._cache) == (0, 0, {}), i
    blk = cache.block()
    x, r = blk.reg(3), blk.reg(4)
    blk.lookup([1, 2], x, r)
    for call in (lambda: blk.lookup([1], x, r),                        # writes r a second time
                 lambda: blk.lookup([1], r[:3], [x[0]]),               # writes what an earlier instruction reads
                 lambda: blk.lookup([1], x, blk.const(4, 0)),
                 lambda: blk.select_n([x], r[:2], x)):
        with pytest.raises(ValueError):
            call()
    assert len(blk._program) == 1
