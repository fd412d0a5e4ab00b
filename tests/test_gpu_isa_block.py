"""InstructionCache.block() on the GPU: a mixed 8-bit block (add, sub with borrow, signed compare, select, multiply,
encrypted shift, sign extension) on encrypted corners and seeded random values, decrypted and compared with integer
semantics; four independent 32-bit adds fused into one graph with one circuit-bootstrap stage; and the mixed block on a
box (two ranks on cuda:0) with box ciphertext handles as inputs and outputs, rebound on a second run."""
import numpy as np
import pytest

from test_isa_block import mixed_cbs, mixed_want, record_mixed

pytestmark = pytest.mark.gpu

W = 8
MASK = (1 << W) - 1
CORNERS = [0, MASK, 1 << (W - 1), (1 << (W - 1)) - 1]
_rng = np.random.default_rng(0xB10C)
VALUES = [(a, b, c, k) for a, b, c, k in zip(CORNERS, CORNERS[::-1], CORNERS[1:] + CORNERS[:1], (0, 7, 1, 3))] + \
    [tuple(int(x) for x in _rng.integers(0, 1 << W, 4) % [256, 256, 256, 8]) for _ in range(3)]


@pytest.fixture(scope="module")
def box2(keys):
    import spf_b200

    b = spf_b200.BoxEvaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft, devices=[0, 0])
    yield b
    b.close()


def _enc(client, v, w):
    return [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]


def _outs(n):
    return [np.zeros(4096, np.uint64) for _ in range(n)]


def _dec(client, bufs):
    return sum(int(client.decrypt_glwe_l1(np.asarray(b))[0]) << i for i, b in enumerate(bufs))


def _cbs(g):
    from spf_b200 import OP

    return int((g._keep.ops == OP["CircuitBootstrap"]).sum())


def test_mixed_block(client, evaluation):
    from spf_b200.circuits import InstructionCache

    cache = InstructionCache(evaluation)
    blk = cache.block()
    ins, res = record_mixed(blk, W)
    for vals in VALUES:
        o = {r: _outs(len(r)) for r in res}
        g = blk.run({r: _enc(client, v, len(r)) for r, v in zip(ins, vals)}, o)
        assert [_dec(client, o[r]) for r in res] == mixed_want(W, *vals), vals
    assert _cbs(g) == mixed_cbs(W)
    assert (cache.misses, cache.hits) == (1, len(VALUES) - 1)


def test_independent_32_bit_adds_share_one_cbs_stage(client, evaluation):
    from spf_b200 import OP, plan_graph
    from spf_b200.circuits import InstructionCache

    cache = InstructionCache(evaluation)
    blk = cache.block()
    ops = [blk.reg(32) for _ in range(8)]
    sums = [blk.reg(33) for _ in range(4)]
    for i, s in enumerate(sums):
        blk.add(ops[2 * i], ops[2 * i + 1], s)
    for seed in (1, 2):
        vals = [int(x) for x in np.random.default_rng(seed).integers(0, 1 << 32, 8, dtype=np.uint64)]
        o = {s: _outs(33) for s in sums}
        g = blk.run({r: _enc(client, v, 32) for r, v in zip(ops, vals)}, o)
        assert [_dec(client, o[s]) for s in sums] == [vals[2 * i] + vals[2 * i + 1] for i in range(4)], seed
    level, _ = plan_graph(g._keep)
    assert len(set(level[g._keep.ops == OP["CircuitBootstrap"]].tolist())) == 1
    assert _cbs(g) == 4 * 2 * 32


def test_box_mixed_block_through_handles(client, evaluation, box2):
    """The same block on the box, every input and output a BoxCiphertext handle: each rank's replica decrypts as the
    single-context run does; the second run writes new values into the same handles and rebinds them (a cache hit)."""
    import spf_b200
    from spf_b200.circuits import InstructionCache

    box, single = InstructionCache(box2), InstructionCache(evaluation)
    bblk, sblk = box.block(), single.block()
    (bins, bres), (sins, sres) = record_mixed(bblk, W), record_mixed(sblk, W)
    handles = lambda n: [spf_b200.BoxCiphertext.alloc(box2, "Glwe1") for _ in range(n)]
    hin, hout = {r: handles(len(r)) for r in bins}, {r: handles(len(r)) for r in bres}
    for vals in VALUES[1:3]:
        for r, v in zip(bins, vals):
            for h, ct in zip(hin[r], _enc(client, v, len(r))):
                h.write(ct)
        bblk.run(hin, hout)
        o = {r: _outs(len(r)) for r in sres}
        sblk.run({r: _enc(client, v, len(r)) for r, v in zip(sins, vals)}, o)
        want = mixed_want(W, *vals)
        assert [_dec(client, o[r]) for r in sres] == want, vals
        for rank in range(box2.size):
            assert [_dec(client, [h.read(rank) for h in hout[r]]) for r in bres] == want, (vals, rank)
    assert (box.misses, box.hits) == (single.misses, single.hits) == (1, 1)
