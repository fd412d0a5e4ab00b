"""Table lookups on the GPU: the AES S-box at every index, a 5 -> 3-bit table behind a partly plaintext index, 12 -> 1 and
16 -> 16-bit tables (the CMux tree above one polynomial), an 8-bit product read from a 16-bit table against
InstructionCache.multiply, select_n over encrypted entries, and a lookup -> add -> compare block on one context and on a
two-rank box (both ranks on cuda:0) through BoxCiphertext handles.  Decrypted and compared with Python indexing; the
worst noise of the S-box and 16-bit results is printed and bounded."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def aes_sbox() -> list[int]:
    """The AES S-box (FIPS-197 5.1.1): the inverse in GF(2^8) mod x^8 + x^4 + x^3 + x + 1, then the affine map."""
    def mul(a, b):
        p = 0
        while b:
            p, a, b = p ^ (a if b & 1 else 0), ((a << 1) ^ 0x11B) if a & 0x80 else a << 1, b >> 1
        return p

    inv = [0] + [next(b for b in range(1, 256) if mul(a, b) == 1) for a in range(1, 256)]
    rot = lambda x, i: ((x << i) | (x >> (8 - i))) & 0xFF
    return [inv[a] ^ rot(inv[a], 1) ^ rot(inv[a], 2) ^ rot(inv[a], 3) ^ rot(inv[a], 4) ^ 0x63 for a in range(256)]


SBOX = aes_sbox()


def _enc(client, v, w):
    return [client.encrypt_glwe_l1([(v >> i) & 1]) for i in range(w)]


def _outs(n):
    return [np.zeros(4096, np.uint64) for _ in range(n)]


def _dec(client, bufs):
    return sum(int(client.decrypt_glwe_l1(np.asarray(b))[0]) << i for i, b in enumerate(bufs))


def _noise(client, bufs, value):
    """Worst torus distance of coefficient 0 of each result bit from its encoded bit (bit * q/2)."""
    worst = 0.0
    for i, b in enumerate(bufs):
        d = (int(client.decrypt_glwe_l1_raw(np.asarray(b))[0]) - (((value >> i) & 1) << 63)) % (1 << 64)
        worst = max(worst, min(d, (1 << 64) - d) / 2.0 ** 64)
    return worst


def _check_noise(name, worst):
    """Decryption fails at a torus distance of 1/4; the lookup results stay far below it."""
    print(f"{name}: worst noise of a lookup result bit {worst:.3e} (2^{np.log2(max(worst, 2.0 ** -64)):.1f})")
    assert worst < 1 / 16


def test_aes_sbox_at_every_index(client, evaluation):
    from spf_b200.circuits import InstructionCache

    assert (SBOX[0x00], SBOX[0x01], SBOX[0x53], SBOX[0xFF]) == (0x63, 0x7C, 0xED, 0x16)
    cache, worst = InstructionCache(evaluation), 0.0
    for x in range(256):
        o = _outs(8)
        cache.lookup(SBOX, _enc(client, x, 8), o)
        assert _dec(client, o) == SBOX[x], x
        worst = max(worst, _noise(client, o, SBOX[x]))
    assert (cache.misses, cache.hits) == (1, 255)
    _check_noise("S-box", worst)


def test_partly_plain_index(client, evaluation):
    from spf_b200.circuits import InstructionCache, Plain

    cache = InstructionCache(evaluation)
    table = [int(v) for v in np.random.default_rng(53).integers(0, 8, 32)]
    for x in range(32):
        ct = _enc(client, x, 5)
        idx = [Plain(x, 5).bits[j] if j in (1, 3) else ct[j] for j in range(5)]
        o = _outs(3)
        cache.lookup(table, idx, o)
        assert _dec(client, o) == table[x], x
    assert cache.misses == 4


def test_12_bit_table(client, evaluation):
    from spf_b200.circuits import InstructionCache

    rng = np.random.default_rng(12)
    table = rng.integers(0, 2, 1 << 12)
    cache = InstructionCache(evaluation)
    for x in [0, 2047, 2048, 4095] + [int(v) for v in rng.integers(0, 1 << 12, 4)]:
        o = _outs(1)
        cache.lookup(table, _enc(client, x, 12), o)
        assert _dec(client, o) == table[x], x


def test_16_bit_table(client, evaluation):
    from spf_b200.circuits import InstructionCache

    rng = np.random.default_rng(16)
    table = rng.integers(0, 1 << 16, 1 << 16)
    cache, worst = InstructionCache(evaluation), 0.0
    for x in [0, (1 << 16) - 1] + [int(v) for v in rng.integers(0, 1 << 16, 4)]:
        o = _outs(16)
        cache.lookup(table, _enc(client, x, 16), o)
        assert _dec(client, o) == table[x], x
        worst = max(worst, _noise(client, o, int(table[x])))
    _check_noise("16-bit table", worst)


def test_product_table_against_multiply(client, evaluation):
    from spf_b200.circuits import InstructionCache

    i = np.arange(1 << 16)
    table = (i & 0xFF) * (i >> 8) & 0xFF
    cache = InstructionCache(evaluation)
    rng = np.random.default_rng(88)
    for x, y in [(0xFF, 0xFF), (3, 0x55)] + [tuple(int(v) for v in rng.integers(0, 256, 2)) for _ in range(2)]:
        a, b = _enc(client, x, 8), _enc(client, y, 8)
        lo, mu = _outs(8), _outs(8)
        cache.lookup(table, a + b, lo)
        cache.multiply(a, b, mu)
        assert _dec(client, lo) == _dec(client, mu) == x * y & 0xFF, (x, y)


def test_select_n(client, evaluation):
    from spf_b200.circuits import InstructionCache

    rng = np.random.default_rng(8)
    vals = [int(v) for v in rng.integers(0, 256, 8)]
    entries = [_enc(client, v, 8) for v in vals]
    cache = InstructionCache(evaluation)
    for x in range(8):
        o = _outs(8)
        cache.select_n(entries, _enc(client, x, 3), o)
        assert _dec(client, o) == vals[x], x
        o = _outs(8)
        cache.select_n(entries[:5], _enc(client, x, 3), o)
        assert _dec(client, o) == (vals[x] if x < 5 else 0), x
    assert (cache.misses, cache.hits) == (2, 14)


def _lookup_block(blk):
    """t = SBOX[x]; s = t + y; f = s[:8] > y."""
    x, y, t, s, f = blk.reg(8), blk.reg(8), blk.reg(8), blk.reg(9), blk.reg(1)
    blk.lookup(SBOX, x, t)
    blk.add(t, y, s)
    blk.compare(s[:8], y, f[0], "gt")
    return (x, y), [t, s, f]


def _lookup_block_want(x, y):
    s = SBOX[x] + y
    return [SBOX[x], s, int(s & 0xFF > y)]


def test_block_on_one_context_and_on_a_box_through_handles(client, evaluation, box2):
    import spf_b200
    from spf_b200.circuits import InstructionCache

    box, single = InstructionCache(box2), InstructionCache(evaluation)
    bblk, sblk = box.block(), single.block()
    (bx, by), bres = _lookup_block(bblk)
    (sx, sy), sres = _lookup_block(sblk)
    hx, hy = ([spf_b200.BoxCiphertext.alloc(box2, "Glwe1") for _ in range(8)] for _ in range(2))
    hout = {r: [spf_b200.BoxCiphertext.alloc(box2, "Glwe1") for _ in range(len(r))] for r in bres}
    for x, y in [(0x00, 0x9C), (0x53, 0x12)]:
        cx, cy = _enc(client, x, 8), _enc(client, y, 8)
        for h, ct in zip(hx + hy, cx + cy):
            h.write(ct)
        bblk.run({bx: hx, by: hy}, hout)
        o = {r: _outs(len(r)) for r in sres}
        sblk.run({sx: cx, sy: cy}, o)
        want = _lookup_block_want(x, y)
        assert [_dec(client, o[r]) for r in sres] == want, (x, y)
        for rank in range(box2.size):
            assert [_dec(client, [h.read(rank) for h in hout[r]]) for r in bres] == want, (x, y, rank)
    assert (box.misses, box.hits) == (single.misses, single.hits) == (1, 1)


@pytest.fixture(scope="module")
def box2(keys):
    import spf_b200

    b = spf_b200.BoxEvaluation(keys.bsk_fft, keys.ksk, keys.ssk_fft, keys.ak_fft, devices=[0, 0])
    yield b
    b.close()
