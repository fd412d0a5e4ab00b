"""InstructionCache's integer instructions on the GPU: every method at w = 8 on encrypted operands (seeded random values
plus the corners 0, 2^w - 1, 2^(w-1), 2^(w-1) - 1), decrypted and compared with integer semantics; one compiled graph
per instruction shape, rebound on every later call; 32-bit sub and signed less-than; and sub then compare on a box
(two ranks on cuda:0) chained through box ciphertext handles."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W = 8
MASK = (1 << W) - 1
CORNERS = [0, MASK, 1 << (W - 1), (1 << (W - 1)) - 1]
_rng = np.random.default_rng(0x15A)
VALUES = CORNERS + [int(x) for x in _rng.integers(0, 1 << W, 3)]
PAIRS = [(a, b) for a in CORNERS for b in CORNERS] + [(int(a), int(b)) for a, b in _rng.integers(0, 1 << W, (4, 2))]


@pytest.fixture(scope="module")
def box2(keys):
    import spf_b200

    b = spf_b200.BoxEvaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft, devices=[0, 0])
    yield b
    b.close()


@pytest.fixture(scope="module")
def enc(client):
    memo = {}

    def f(v, w=W):
        if (v, w) not in memo:
            memo[v, w] = [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]
        return memo[v, w]

    return f


def _outs(n):
    return [np.zeros(4096, np.uint64) for _ in range(n)]


def _dec(client, bufs):
    return sum(int(client.decrypt_glwe_l1(np.asarray(b))[0]) << i for i, b in enumerate(bufs))


def _signed(v, w=W):
    return v - ((v >> (w - 1)) << w)


def _check_one_graph(cache, graphs, calls):
    """Every call ran the one graph compiled by the first."""
    assert (cache.misses, cache.hits) == (1, calls - 1)
    assert all(g is graphs[0] for g in graphs)


BINARY = {
    "sub": (lambda c, a, b, o: c.sub(a, b, o), W + 1, lambda a, b: (a - b) % (1 << (W + 1))),  # borrow = bit W
    "and_": (lambda c, a, b, o: c.and_(a, b, o), W, lambda a, b: a & b),
    "or_": (lambda c, a, b, o: c.or_(a, b, o), W, lambda a, b: a | b),
    "xor": (lambda c, a, b, o: c.xor(a, b, o), W, lambda a, b: a ^ b),
    "equal": (lambda c, a, b, o: c.equal(a, b, o[0]), 1, lambda a, b: int(a == b)),
    "not_equal": (lambda c, a, b, o: c.not_equal(a, b, o[0]), 1, lambda a, b: int(a != b)),
    "multiply_signed": (lambda c, a, b, o: c.multiply_signed(a, b, o), W, lambda a, b: (_signed(a) * _signed(b)) & MASK),
}
for _op, _rel in (("gt", lambda x, y: x > y), ("ge", lambda x, y: x >= y), ("lt", lambda x, y: x < y), ("le", lambda x, y: x <= y)):
    for _s in (False, True):
        BINARY[f"compare_{_op}{'_signed' if _s else ''}"] = (
            lambda c, a, b, o, op=_op, s=_s: c.compare(a, b, o[0], op, signed=s), 1,
            lambda a, b, rel=_rel, s=_s: int(rel(_signed(a), _signed(b)) if s else rel(a, b)))


@pytest.mark.parametrize("name", sorted(BINARY))
def test_binary_instruction(client, evaluation, enc, name):
    from spf_b200.circuits import InstructionCache

    call, n_out, want = BINARY[name]
    cache = InstructionCache(evaluation)
    graphs = []
    for a, b in PAIRS:
        o = _outs(n_out)
        graphs.append(call(cache, enc(a), enc(b), o))
        assert _dec(client, o) == want(a, b), (name, a, b)
    _check_one_graph(cache, graphs, len(PAIRS))


def test_unary_instructions_and_casts(client, evaluation, enc):
    from spf_b200.circuits import InstructionCache

    cases = {
        "neg": (lambda c, a, o: c.neg(a, o), W, lambda v: (-v) & MASK),
        "not_": (lambda c, a, o: c.not_(a, o), W, lambda v: ~v & MASK),
        "zext": (lambda c, a, o: c.zext(a, o), 2 * W, lambda v: v),
        "sext": (lambda c, a, o: c.sext(a, o), 2 * W, lambda v: _signed(v) & ((1 << 2 * W) - 1)),
        "trunc": (lambda c, a, o: c.trunc(a, o), 3, lambda v: v & 7),
    }
    for name, (call, n_out, want) in cases.items():
        cache = InstructionCache(evaluation)
        graphs = []
        for v in VALUES:
            o = _outs(n_out)
            graphs.append(call(cache, enc(v), o))
            assert _dec(client, o) == want(v), (name, v)
        _check_one_graph(cache, graphs, len(VALUES))


SHIFTS = [(False, "logical"), (True, "logical"), (True, "arithmetic"), (False, "rotation"), (True, "rotation")]


def _shifted(v, k, right, mode):
    if mode == "rotation":
        k %= W
        return ((v >> k) | (v << (W - k))) & MASK if right else ((v << k) | (v >> (W - k))) & MASK
    if mode == "arithmetic":
        return (_signed(v) >> min(k, W)) & MASK
    return ((v >> k) if right else (v << k)) & MASK if k < W else 0


@pytest.mark.parametrize("right,mode", SHIFTS)
def test_shift_by_encrypted_amount(client, evaluation, enc, right, mode):
    from spf_b200.circuits import InstructionCache

    cache = InstructionCache(evaluation)
    graphs = []
    cases = [(v, k) for v in VALUES[:5] for k in (0, 1, 5, 7, 8, 13)]
    for v, k in cases:
        o = _outs(W)
        graphs.append(cache.shift(enc(v), enc(k, 4), o, right, mode))
        assert _dec(client, o) == _shifted(v, k, right, mode), (v, k)
    _check_one_graph(cache, graphs, len(cases))


@pytest.mark.parametrize("right,mode", SHIFTS)
def test_shift_by_constant(client, evaluation, enc, right, mode):
    """Rewiring only: k = W under a logical shift leaves a graph with no operand bit at all."""
    from spf_b200.circuits import InstructionCache

    for k in (0, 3, W):
        cache = InstructionCache(evaluation)
        graphs = []
        for v in VALUES:
            o = _outs(W)
            graphs.append(cache.shift_const(enc(v), k, o, right, mode))
            assert _dec(client, o) == _shifted(v, k, right, mode), (v, k)
        _check_one_graph(cache, graphs, len(VALUES))


def test_select(client, evaluation, enc):
    from spf_b200.circuits import InstructionCache

    cache = InstructionCache(evaluation)
    graphs = []
    cases = [(c, a, b) for c in (0, 1) for a, b in PAIRS[::3]]
    for c, a, b in cases:
        o = _outs(W)
        graphs.append(cache.select(enc(c, 1)[0], enc(a), enc(b), o))
        assert _dec(client, o) == (b if c else a), (c, a, b)
    _check_one_graph(cache, graphs, len(cases))


def test_32_bit_sub_and_signed_less_than(client, evaluation, enc):
    from spf_b200.circuits import InstructionCache

    cache = InstructionCache(evaluation)
    for a, b in ((0x1234ABCD, 0xF00DBEEF), (0xF00DBEEF, 0x1234ABCD)):
        o = _outs(32)
        cache.sub(enc(a, 32), enc(b, 32), o)
        assert _dec(client, o) == (a - b) % (1 << 32)
        lt = _outs(1)
        cache.compare(enc(a, 32), enc(b, 32), lt[0], "lt", signed=True)
        assert _dec(client, lt) == int(_signed(a, 32) < _signed(b, 32)), (a, b)
    assert (cache.misses, cache.hits) == (2, 2)


def test_box_sub_then_compare_through_handles(client, evaluation, box2, enc):
    """d = a - b on the box into box ciphertext handles, then d < c (signed) reading those handles: the decryptions
    match the same two instructions on the single context through host buffers."""
    import spf_b200
    from spf_b200.circuits import InstructionCache

    single, box = InstructionCache(evaluation), InstructionCache(box2)
    for a, b, c in ((200, 100, 50), (3, 130, 1), (77, 77, 0)):
        handles = lambda n: [spf_b200.BoxCiphertext.alloc(box2, "Glwe1") for _ in range(n)]
        ha, hb, hc = handles(W), handles(W), handles(W)
        for hs, v in ((ha, a), (hb, b), (hc, c)):
            for h, ct in zip(hs, enc(v)):
                h.write(ct)
        d, lt = handles(W), handles(1)
        box.sub(ha, hb, d)
        box.compare(d, hc, lt[0], "lt", signed=True)
        d_ref, lt_ref = _outs(W), _outs(1)
        single.sub(enc(a), enc(b), d_ref)
        single.compare(d_ref, enc(c), lt_ref[0], "lt", signed=True)
        want_d = (a - b) & MASK
        for r in range(box2.size):
            assert _dec(client, [h.read(r) for h in d]) == _dec(client, d_ref) == want_d, (a, b, r)
            assert _dec(client, [h.read(r) for h in lt]) == _dec(client, lt_ref) == int(_signed(want_d) < _signed(c))
    assert (box.misses, box.hits) == (single.misses, single.hits) == (2, 4)
