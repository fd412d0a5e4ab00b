"""Plaintext operands on the GPU: every instruction at 8 bits with a Plain operand (in either place, and as select's
condition and the shift amount) on encrypted values, add / compare / multiply by a constant at 32 bits, a graph of
constants only, and a block with const registers on a two-rank box (both ranks on cuda:0) whose inputs and outputs are
BoxCiphertext handles -- including outputs that fold to constants.  Decrypted and compared with integer semantics."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W = 8
MASK = (1 << W) - 1


def _sg(v, w=W):
    return v - ((v >> (w - 1)) << w)


def _enc(client, v, w):
    return [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]


def _outs(n):
    return [np.zeros(4096, np.uint64) for _ in range(n)]


def _dec(client, bufs):
    return sum(int(client.decrypt_glwe_l1(np.asarray(b))[0]) << i for i, b in enumerate(bufs))


def _run(call, r):
    call(r)
    return r


def _calls(P):
    """(name, call(cache, x, y, out_factory) -> result bits, semantics(x, y)): x is encrypted, y the constant."""
    yield "add", lambda c, x, y, o: _run(lambda r: c.add(x, P(y), r), o(W + 1)), lambda x, y: x + y
    yield "add_plain_first", lambda c, x, y, o: _run(lambda r: c.add(P(y), x, r), o(W + 1)), lambda x, y: x + y
    yield "sub", lambda c, x, y, o: _run(lambda r: c.sub(x, P(y), r), o(W)), lambda x, y: (x - y) & MASK
    yield "sub_plain_first", lambda c, x, y, o: _run(lambda r: c.sub(P(y), x, r), o(W + 1)), lambda x, y: (y - x) % (1 << W + 1)
    yield "compare_gt", lambda c, x, y, o: _run(lambda r: c.compare(x, P(y), r[0], "gt"), o(1)), lambda x, y: int(x > y)
    yield "compare_le_signed", lambda c, x, y, o: _run(lambda r: c.compare(P(y), x, r[0], "le", signed=True), o(1)), \
        lambda x, y: int(_sg(y) <= _sg(x))
    yield "equal", lambda c, x, y, o: _run(lambda r: c.equal(x, P(y), r[0]), o(1)), lambda x, y: int(x == y)
    yield "not_equal", lambda c, x, y, o: _run(lambda r: c.not_equal(x, P(y), r[0]), o(1)), lambda x, y: int(x != y)
    yield "and_", lambda c, x, y, o: _run(lambda r: c.and_(x, P(y), r), o(W)), lambda x, y: x & y
    yield "or_", lambda c, x, y, o: _run(lambda r: c.or_(P(y), x, r), o(W)), lambda x, y: x | y
    yield "xor", lambda c, x, y, o: _run(lambda r: c.xor(x, P(y), r), o(W)), lambda x, y: x ^ y
    yield "multiply", lambda c, x, y, o: _run(lambda r: c.multiply(x, P(y), r), o(W)), lambda x, y: x * y & MASK
    yield "multiply_signed", lambda c, x, y, o: _run(lambda r: c.multiply_signed(P(y), x, r), o(W)), lambda x, y: _sg(x) * _sg(y) & MASK
    yield "select_plain_cond", lambda c, x, y, o: _run(lambda r: c.select(P(y & 1, 1), x, P(y), r), o(W)), \
        lambda x, y: y if y & 1 else x
    yield "shift_plain_amount", lambda c, x, y, o: _run(lambda r: c.shift(x, P(y % 11, 4), r, True, "arithmetic"), o(W)), \
        lambda x, y: (_sg(x) >> min(y % 11, W)) & MASK
    yield "shift_plain_value", lambda c, x, y, o: _run(lambda r: c.shift(P(y), [b for b in x[:3]], r, False), o(W)), \
        lambda x, y: (y << (x & 7)) & MASK


@pytest.mark.parametrize("case", range(16))
def test_every_instruction_with_a_plaintext_operand(client, evaluation, case):
    from spf_b200.circuits import InstructionCache, Plain

    name, call, want = list(_calls(lambda v, w=W: Plain(v, w)))[case]
    cache = InstructionCache(evaluation)
    rng = np.random.default_rng(case)
    for x, y in [(0x5A, 0xC3), (MASK, 1)] + [tuple(int(v) for v in rng.integers(0, 1 << W, 2))]:
        xs = _enc(client, x, W)
        r = call(cache, xs, y, _outs)
        assert _dec(client, r) == want(x, y), (name, x, y)


def test_32_bit_add_compare_and_multiply_by_a_constant(client, evaluation):
    from spf_b200.circuits import InstructionCache, Plain

    cache = InstructionCache(evaluation)
    rng = np.random.default_rng(32)
    for x, k in [(0xFFFFFFFF, 1), (int(rng.integers(0, 1 << 32)), 77), (int(rng.integers(0, 1 << 32)), 0xDEADBEEF)]:
        xs = _enc(client, x, 32)
        s, gt, m, sm = _outs(33), _outs(1), _outs(32), _outs(32)
        cache.add(xs, Plain(k, 32), s)
        cache.compare(xs, Plain(k, 32), gt[0], "gt", signed=True)
        assert (_dec(client, s), _dec(client, gt)) == (x + k, int(_sg(x, 32) > _sg(k, 32))), (x, k)
        if k < 1 << 16:   # a full-width constant's multiplier is ~600 k multiplexers: tools/plain_latency.py times one
            cache.multiply(xs, Plain(k, 32), m)
            cache.multiply_signed(xs, Plain(-k, 32), sm)
            assert (_dec(client, m), _dec(client, sm)) == (x * k % (1 << 32), _sg(x, 32) * -k % (1 << 32)), (x, k)


def test_a_graph_of_constants_only(client, evaluation):
    from spf_b200.circuits import InstructionCache, Plain

    cache = InstructionCache(evaluation)
    s, p = _outs(W + 1), _outs(W)
    g = cache.add(Plain(200, W), Plain(100, W), s)
    cache.multiply(Plain(13, W), Plain(11, W), p)
    assert (_dec(client, s), _dec(client, p)) == (300, 143)
    assert g.levels >= 1


def _const_block(blk):
    """s = a + 100, f = s > -3 signed, m = a * 7, z = a & 0 (constant), t = 9 + 4 (constants only), g = f ? m : 37."""
    from spf_b200.circuits import Plain

    a = blk.reg(W)
    s, f, m, z, t, g = blk.reg(W + 1), blk.reg(1), blk.reg(W), blk.reg(W), blk.reg(W + 1), blk.reg(W)
    blk.add(a, blk.const(W, 100), s)
    blk.compare(s[:W], blk.const(W, -3), f[0], "gt", signed=True)
    blk.multiply(a, blk.const(W, 7), m)
    blk.and_(a, Plain(0, W), z)
    blk.add(blk.const(W, 9), Plain(4, W), t)
    blk.select(f[0], blk.const(W, 37), m, g)
    return a, [s, f, m, z, t, g]


def _const_block_want(a):
    s = a + 100
    f = int(_sg(s & MASK) > -3)
    m = a * 7 & MASK
    return [s, f, m, 0, 13, m if f else 37]


def test_box_const_block_through_handles(client, evaluation, box2):
    import spf_b200
    from spf_b200.circuits import InstructionCache

    box, single = InstructionCache(box2), InstructionCache(evaluation)
    bblk, sblk = box.block(), single.block()
    (ba, bres), (sa, sres) = _const_block(bblk), _const_block(sblk)
    hin = [spf_b200.BoxCiphertext.alloc(box2, "Glwe1") for _ in range(W)]
    hout = {r: [spf_b200.BoxCiphertext.alloc(box2, "Glwe1") for _ in range(len(r))] for r in bres}
    for a in (0x7F, 0xA0):
        for h, ct in zip(hin, _enc(client, a, W)):
            h.write(ct)
        bblk.run({ba: hin}, hout)
        o = {r: _outs(len(r)) for r in sres}
        sblk.run({sa: _enc(client, a, W)}, o)
        want = _const_block_want(a)
        assert [_dec(client, o[r]) for r in sres] == want, a
        for rank in range(box2.size):
            assert [_dec(client, [h.read(rank) for h in hout[r]]) for r in bres] == want, (a, rank)
    assert (box.misses, box.hits) == (single.misses, single.hits) == (1, 1)


@pytest.fixture(scope="module")
def box2(keys):
    import spf_b200

    b = spf_b200.BoxEvaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft, devices=[0, 0])
    yield b
    b.close()
