"""GPU parity tests proper: the CUDA path through the C ABI (spf_b200.Evaluation over
libspf_b200.so) against the CPU oracle on the same seeded keys and inputs.

Bars (DESIGN.md "Parity contract"):
  * integer / index ops (keyswitch, sample extract, not, xor, mul_xn): bit-exact;
  * single-pass FFT ops on exact inputs (cmux, external product, scheme switch): max torus
    distance <= 2^-30 (f64 rounding of ~2^88-sized IFFT outputs), FFT-domain rel. error <= 1e-12;
  * multi-step ops whose later steps decompose values carrying FFT rounding noise (PBS, trace,
    CBS): decryptions bit-exact, phase (b - a.s) distance <= 4 x the measured maximum (PBS 3.8e-6, CBS 2.4e-6,
    trace 1.9e-7 of the torus; tests/test_gpu_distances.py) -- ciphertext bytes are not comparable between any
    two FFT implementations (see test_emu.test_pbs_first_steps...); against the host emulator, which
    rounds identically, every kernel is BIT-EXACT (tests/test_gpu_bitexact.py);
  * exact regime (integer-polynomial keys, tests/exact_keys.py): PBS, trace, CMUX and the CBS stages BIT-EXACT against
    the oracle on arbitrary u64 inputs, every item; CBS and scheme-switch outputs FFT-domain <= 1e-14 relative
    (tests/test_gpu_exact.py).
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TIGHT = 2.0 ** -30


def test_library_is_the_cuda_path(evaluation):
    import spf_b200

    assert spf_b200.LIB_PATH.endswith("libspf_b200.so")
    assert evaluation.kernel_launches >= 3  # key rescale kernels ran on the device


def test_keyswitch_bit_exact(oracle, keys, client, evaluation):
    bits = [1, 0, 1, 1, 0, 0, 1]
    l1 = np.stack([client.encrypt_lwe_l1(b) for b in bits])
    got = evaluation.keyswitch_lwe_l1_lwe_l0(l1)
    want = np.stack([oracle.keyswitch_lwe(keys, x) for x in l1])
    assert np.array_equal(got, want)
    assert [client.decrypt_lwe_l0(x) for x in got] == bits


@pytest.mark.parametrize("batch", [1, 15, 16, 17, 33, 129, 300])
def test_keyswitch_ragged_batches(oracle, keys, evaluation, batch):
    rng = np.random.default_rng(batch)
    l1 = rng.integers(0, 1 << 64, (batch, keys.lwe1_len), dtype=np.uint64)
    got = evaluation.keyswitch_lwe_l1_lwe_l0(l1)
    want = np.zeros_like(got)
    oracle.lib().orc_keyswitch_lwe_batch(want, l1, batch, keys.ksk, C.byref(keys.params), oracle.hw_threads())
    bad = [i for i in range(batch) if not np.array_equal(got[i], want[i])]
    assert not bad, bad


def test_sample_extract_bit_exact(oracle, keys, evaluation):
    rng = np.random.default_rng(3)
    g = rng.integers(0, 1 << 64, (6, keys.glwe_len), dtype=np.uint64)
    idx = np.array([0, 1, 2, 1000, 2046, 2047], dtype=np.uint32)
    got = evaluation.sample_extract_l1(g, idx)
    for i, h in enumerate(idx):
        assert np.array_equal(got[i], oracle.sample_extract(keys, g[i], int(h)))
    got0 = evaluation.sample_extract_l1(g, 0)
    for i in range(len(g)):
        assert np.array_equal(got0[i], oracle.sample_extract(keys, g[i], 0)), i
    # every index once, one per item
    g = rng.integers(0, 1 << 64, (2048, keys.glwe_len), dtype=np.uint64)
    got = evaluation.sample_extract_l1(g, np.arange(2048, dtype=np.uint32))
    bad = [h for h in range(2048) if not np.array_equal(got[h], oracle.sample_extract(keys, g[h], h))]
    assert not bad, bad


def test_not_xor_mul_xn_bit_exact(oracle, keys, evaluation):
    rng = np.random.default_rng(4)
    a = rng.integers(0, 1 << 64, (5, keys.glwe_len), dtype=np.uint64)
    b = rng.integers(0, 1 << 64, (5, keys.glwe_len), dtype=np.uint64)
    assert np.array_equal(evaluation.not_(a)[2], oracle.glwe_not(keys, a[2]))
    assert np.array_equal(evaluation.xor(a, b), a + b)
    for n in (0, 1, 7, 2047, 2048, 2049, 4095):
        assert np.array_equal(evaluation.mul_xn(a, n)[1], oracle.glwe_mul_xn(keys, a[1], n)), n


def test_cmux_matches_oracle(oracle, keys, client, evaluation):
    a = client.encrypt_glwe_l1([0, 1, 1, 0])
    b = client.encrypt_glwe_l1([1, 0, 1, 0])
    sels = [0, 1, 1, 0, 1]
    ggsw = np.stack([client.encrypt_ggsw_l1(s) for s in sels])
    out = evaluation.cmux(ggsw, np.stack([a] * 5), np.stack([b] * 5))
    for i, s in enumerate(sels):
        ref = oracle.cmux(keys, a, b, ggsw[i])
        assert oracle.torus_distance(ref, out[i]).max() <= TIGHT
        assert client.decrypt_glwe_l1(out[i])[:4].tolist() == ([1, 0, 1, 0] if s else [0, 1, 1, 0])


def test_multiply_glwe_ggsw_and_glev_cmux(oracle, keys, client, evaluation):
    g = client.encrypt_glwe_l1([1, 1, 0, 1])
    for bit in (0, 1):
        ggsw = client.encrypt_ggsw_l1(bit)
        out = evaluation.multiply_glwe_ggsw(g, ggsw)[0]
        assert oracle.torus_distance(oracle.multiply_glwe_ggsw(keys, g, ggsw), out).max() <= TIGHT
        assert client.decrypt_glwe_l1(out)[:4].tolist() == ([1, 1, 0, 1] if bit else [0, 0, 0, 0])
        d0 = client.encrypt_glev_l1([0, 1])
        d1 = client.encrypt_glev_l1([1, 1])
        out = evaluation.glev_cmux(ggsw, d0, d1)[0]
        assert oracle.torus_distance(oracle.glev_cmux(keys, d0, d1, ggsw), out).max() <= TIGHT


def test_scheme_switch_matches_oracle(oracle, keys, client, evaluation):
    glevs = np.stack([client.encrypt_glev_l1([b]) for b in (0, 1, 1)])
    out = evaluation.scheme_switch(glevs)
    for i, bit in enumerate((0, 1, 1)):
        ref = oracle.scheme_switch(keys, glevs[i])
        assert np.abs(out[i] - ref).max() <= 1e-12 * np.abs(ref).max()
        assert np.array_equal(client.ggsw_level_messages(out[i]), client.ggsw_expected_messages(bit))


def test_trace_decrypts_like_oracle(oracle, keys, client, evaluation):
    n = keys.params.glwe_n
    msg = np.zeros(n, dtype=np.uint64)
    msg[:8] = np.arange(1, 9, dtype=np.uint64) << np.uint64(64 - 4 - 11)
    ct = np.zeros(keys.glwe_len, dtype=np.uint64)
    oracle.lib().orc_encrypt_glwe(C.byref(client.rng), ct, msg, keys.glwe1_sk, C.byref(keys.params))
    out = evaluation.trace(ct)[0]
    ref = oracle.trace(keys, ct)
    dec = client.decrypt_glwe_l1(out, 4)
    assert dec[0] == 1 and not dec[1:].any()
    ph = oracle.torus_distance(client.decrypt_glwe_l1_raw(ref), client.decrypt_glwe_l1_raw(out))
    assert ph.max() <= 1.9e-7  # 4 x the measured maximum (tests/test_gpu_distances.py)


def test_single_pbs_config2(oracle, keys, client, evaluation):
    """BASELINE config 2: programmable_bootstrap_univariate with identity and (x+3)%8 LUTs at
    3 plaintext bits + 1 padding bit (programmable_bootstrapping.rs:709-789), all 8 messages,
    GPU vs CPU: decrypt equality and max phase distance."""
    p = keys.params
    worst = 0.0
    for fn in (lambda x: x, lambda x: (x + 3) % 8):
        lut = oracle.generate_lut(p, [fn], 3)
        cts = np.zeros((8, keys.lwe0_len), dtype=np.uint64)
        for m in range(8):
            oracle.lib().orc_encrypt_lwe(C.byref(client.rng), cts[m], keys.lwe0_sk, p.lwe_n, p.lwe_std, m << 60)
        out = evaluation.programmable_bootstrap(cts, lut)
        for m in range(8):
            l1 = evaluation.sample_extract_l1(out[m], 0)[0]
            assert client.decrypt_lwe_l1(l1, 3) == fn(m)
            ref = oracle.pbs_generalized(keys, cts[m], lut)
            assert int(oracle.decode(client.decrypt_glwe_l1_raw(ref)[:1], 3)[0]) == fn(m)
            d = oracle.torus_distance(client.decrypt_glwe_l1_raw(ref)[:1], client.decrypt_glwe_l1_raw(out[m])[:1]).max()
            worst = max(worst, d)
    assert worst <= 3.8e-6, worst  # 4 x the measured maximum 9.5e-7 (tests/test_gpu_distances.py, profiles/r2_measured_distances.json)


def test_multifunction_pbs_cbs_stage(oracle, keys, client, evaluation):
    """The CBS-internal multi-function PBS (log_v = 2): coefficient i of the output phase is
    +/- B^-(i+1)/2 (circuit_bootstrapping.rs:430-482; pattern test programmable_bootstrapping.rs:963-983)."""
    lut = np.zeros(keys.glwe_len, dtype=np.uint64)
    oracle.lib().orc_cbs_lut(lut, C.byref(keys.params))
    for bit in (0, 1):
        ct = client.encrypt_lwe_l0(bit)
        rot = ct.copy()
        rot[-1] = np.uint64((int(rot[-1]) + (1 << 62)) & ((1 << 64) - 1))
        out = evaluation.programmable_bootstrap(rot, lut, 0, 2)[0]
        ref = oracle.cbs_pbs_stage(keys, ct)
        pg, pr = client.decrypt_glwe_l1_raw(out), client.decrypt_glwe_l1_raw(ref)
        for i in range(4):
            mag = 1 << (64 - (4 * (i + 1) + 1))
            want = mag if bit else -mag
            assert abs(int(np.int64(pg[i])) - want) < mag // 8
            assert abs(int(np.int64(pr[i])) - want) < mag // 8


def _cbs_preprocess(glwe: np.ndarray, level: int, params) -> np.ndarray:
    """mod_switch_trace_and_rotate up to (not including) the trace, for cbs level `level` (circuit_bootstrapping.rs:
    260-298): b[i'] += encode(1, 4 (i' + 1) + 1) for i' <= level (the reference adds them cumulatively on one buffer),
    every polynomial times X^-level (entities/polynomial.rs:211-236), then glwe_mod_switch_and_expand_pow_2 by log2 N
    (glwe_ciphertext_ops.rs:268-281, vector_shr_round scalar.rs:134-143).  Exact integer arithmetic in numpy."""
    n, k = params.glwe_n, params.glwe_k
    x = glwe.astype(np.uint64).reshape(k + 1, n).copy()
    for i in range(level + 1):
        x[k, i] += np.uint64(1 << (64 - (params.cbs.radix_log * (i + 1) + 1)))
    j = np.arange(n) + level
    y = np.where(j < n, x[:, j % n], (~x[:, j % n]) + np.uint64(1))      # (p X^-level)[j] = p[j + level], negated past N
    shift = n.bit_length() - 1
    return ((y >> np.uint64(shift)) + ((y >> np.uint64(shift - 1)) & np.uint64(1))).reshape(-1)


def test_cbs_preprocessing_stage_bit_exact(oracle, keys, client, evaluation):
    """SURVEY 8(a) row a10 on its own: the integer pre-processing that trace_ss_kernel fuses in front of the trace (level
    offsets on b, X^-level, rounded shift by log2 N) against an exact numpy restatement -- blind rotation on the GPU,
    pre-processing on the CPU, trace and scheme switch through their own entry points, and the result must equal the
    one-call circuit bootstrap BIT FOR BIT (the floating-point stages are the same device code on the same inputs)."""
    p = keys.params
    bits = [0, 1, 1]
    cts = client.encrypt_lwe_l0_batch(bits)
    rot = cts.copy()
    rot[:, -1] += np.uint64(1 << 62)                                     # lwe_rotate by encode(1, 2 bits), :403-408
    lut = np.zeros(keys.glwe_len, dtype=np.uint64)
    oracle.lib().orc_cbs_lut(lut, C.byref(p))
    x = evaluation.programmable_bootstrap(rot, lut, 0, 2)                # hi_noise_lwe_to_lo_noise_glwe
    # the numpy pre-processing agrees with the oracle's C restatement of the whole stage (trace included) on level 0 ..
    pre = np.stack([[_cbs_preprocess(x[c], i, p) for i in range(p.cbs.count)] for c in range(len(bits))])
    ref0 = oracle.cbs_trace_stage(keys, x[0]).reshape(p.cbs.count, -1)
    assert np.array_equal(oracle.trace(keys, pre[0, 0]), ref0[0]) and np.array_equal(oracle.trace(keys, pre[0, 3]), ref0[3])
    # .. and the GPU's fused form equals trace + scheme switch applied to it
    glev = evaluation.trace(pre.reshape(-1, keys.glwe_len)).reshape(len(bits), -1)
    staged = evaluation.scheme_switch(glev)
    fused = evaluation.circuit_bootstrap(cts)
    assert np.array_equal(staged.view(np.uint64), fused.view(np.uint64))
    for i, bit in enumerate(bits):
        assert np.array_equal(client.ggsw_level_messages(fused[i]), client.ggsw_expected_messages(bit))


def test_circuit_bootstrap_all_levels(oracle, keys, client, evaluation):
    """can_circuit_bootstrap_via_trace_ss (circuit_bootstrapping.rs:721-805) through the C ABI:
    every (row, level) GLWE of the output GGSW decrypts like a fresh GGSW encryption."""
    bits = [0, 1, 1, 0, 1]
    cts = client.encrypt_lwe_l0_batch(bits)
    out = evaluation.circuit_bootstrap(cts)
    for i, bit in enumerate(bits):
        assert np.array_equal(client.ggsw_level_messages(out[i]), client.ggsw_expected_messages(bit)), i
        assert client.decrypt_ggsw_l1(out[i]) == bit
    # trivial inputs, as Evaluation::new does for l1ggsw_zero/one (evaluation.rs:161-197)
    triv = np.stack([client.trivial_lwe_l0(0), client.trivial_lwe_l0(1)])
    out = evaluation.circuit_bootstrap(triv)
    assert [client.decrypt_ggsw_l1(g) for g in out] == [0, 1]


def test_cbs_then_cmux_chain(oracle, keys, client, evaluation):
    """circuit_processor/tests/mod.rs:53-193 'CBS + CMux': bootstrap the selector on the GPU, mux
    on the GPU, sample-extract + keyswitch back to L0, decrypt."""
    a = client.encrypt_glwe_l1([0])
    b = client.encrypt_glwe_l1([1])
    sels = [0, 1, 1, 0]
    ggsw = evaluation.circuit_bootstrap(client.encrypt_lwe_l0_batch(sels))
    out = evaluation.cmux(ggsw, np.stack([a] * 4), np.stack([b] * 4))
    l1 = evaluation.sample_extract_l1(out, 0)
    l0 = evaluation.keyswitch_lwe_l1_lwe_l0(l1)
    assert [client.decrypt_lwe_l0(x) for x in l0] == sels
    # and around the loop once more: the L0 outputs are valid CBS inputs
    ggsw2 = evaluation.circuit_bootstrap(l0)
    assert [client.decrypt_ggsw_l1(g) for g in ggsw2] == sels


def test_batch_invariance_and_ragged_sizes(oracle, keys, client, evaluation):
    """Size-independent property for the big configs: item i of a batch is bit-identical to the
    same input bootstrapped alone (deterministic kernels, no cross-item state), across batch
    sizes that are not multiples of the 4-per-CTA / 3-per-CTA team counts."""
    rng = np.random.default_rng(11)
    bits = rng.integers(0, 2, 11).tolist()
    cts = client.encrypt_lwe_l0_batch(bits)
    full = evaluation.circuit_bootstrap(cts)
    for n in (1, 2, 3, 5):
        part = evaluation.circuit_bootstrap(cts[:n])
        assert np.array_equal(part, full[:n])
    alone = evaluation.circuit_bootstrap(cts[7])
    assert np.array_equal(alone[0], full[7])
    assert [client.decrypt_ggsw_l1(g) for g in full] == bits


def test_empty_batches_and_errors(keys, evaluation):
    import spf_b200

    assert evaluation.circuit_bootstrap(np.zeros((0, keys.lwe0_len), dtype=np.uint64)).shape == (0, keys.ggsw_fft_len)
    assert evaluation.keyswitch_lwe_l1_lwe_l0(np.zeros((0, keys.lwe1_len), dtype=np.uint64)).shape == (0, keys.lwe0_len)
    with pytest.raises(spf_b200.SpfError):
        evaluation.circuit_bootstrap(np.zeros((2, keys.lwe0_len + 1), dtype=np.uint64))
    with pytest.raises(spf_b200.SpfError):
        evaluation.sample_extract_l1(np.zeros((1, keys.glwe_len), dtype=np.uint64), 2048)
    with pytest.raises(spf_b200.SpfError):
        evaluation.programmable_bootstrap(np.zeros((1, keys.lwe0_len), dtype=np.uint64),
                                          np.zeros(keys.glwe_len, dtype=np.uint64), 0, 12)


def test_large_batch_cbs_sampled(oracle, keys, client, evaluation):
    """BASELINE config 3 shape at reduced size for the test suite (the full 4096 runs in
    bench.py --check): 600 inputs > one wave of 148 SMs x 4; decrypt a sample of outputs."""
    rng = np.random.default_rng(12)
    bits = rng.integers(0, 2, 600)
    cts = client.encrypt_lwe_l0_batch(bits.tolist())
    out = evaluation.circuit_bootstrap(cts)
    for i in rng.choice(600, 24, replace=False):
        assert client.decrypt_ggsw_l1(out[i]) == bits[i], i
    i = 599
    assert np.array_equal(client.ggsw_level_messages(out[i]), client.ggsw_expected_messages(int(bits[i])))


def test_kernel_selection_thresholds(oracle, keys, client, evaluation):
    """launch_pbs switches kernels at one ciphertext per SM (148), launch_cmux at two outputs per SM (296): the
    latency kernels (pbs_quad_kernel, cmux_wide_kernel) below, the throughput kernels (pair teams, one team per
    CMUX) above.  Both sides must decrypt correctly; within a kernel, results do not depend on the batch."""
    rng = np.random.default_rng(21)
    bits = rng.integers(0, 2, 300)
    cts = client.encrypt_lwe_l0_batch(bits.tolist())
    quad = evaluation.circuit_bootstrap(cts[:148])     # one ciphertext per SM on four teams
    pair = evaluation.circuit_bootstrap(cts[:150])     # pair teams, two per SM
    pair2 = evaluation.circuit_bootstrap(cts)          # pair teams, three per SM
    assert np.array_equal(pair, pair2[:150])
    for i in (0, 77, 147):
        assert client.decrypt_ggsw_l1(quad[i]) == bits[i] == client.decrypt_ggsw_l1(pair[i])
    assert client.decrypt_ggsw_l1(pair2[299]) == bits[299]
    # CMUX: 297 ops through the bulk kernel, the first 148 and the first 296 through the wide kernel
    a, b = client.encrypt_glwe_l1([0, 1]), client.encrypt_glwe_l1([1, 1])
    sel = np.stack([quad[i % 148] for i in range(297)])
    A, B = np.stack([a] * 297), np.stack([b] * 297)
    bulk = evaluation.cmux(sel, A, B)
    wide = evaluation.cmux(sel[:148], A[:148], B[:148])
    wide2 = evaluation.cmux(sel[:296], A[:296], B[:296])
    assert np.array_equal(wide2[:148], wide)
    for i in (0, 5, 100, 147):
        want = oracle.cmux(keys, a, b, sel[i])
        assert oracle.torus_distance(want, bulk[i]).max() <= 2.0 ** -30
        assert oracle.torus_distance(want, wide[i]).max() <= 2.0 ** -30
        assert client.decrypt_glwe_l1(wide[i])[:2].tolist() == ([1, 1] if bits[i] else [0, 1])


@pytest.mark.parametrize("batch", [149, 297, 445, 494, 593, 889])
def test_pbs_wave_and_tail_shapes(oracle, keys, client, evaluation, batch):
    """Every way launch_pbs lays a batch out: 2 or 3 pairs per CTA sharing one BSK ring, a ragged last round (pairs with
    fewer ciphertexts count themselves off the ring), full waves followed by the quad-kernel tail (445 = 444 + 1,
    494 = 444 + 50, 889 = 2 x 444 + 1), and a remainder too large for the tail kernel (593 = 444 + 149).  Items at every
    boundary must decrypt."""
    p = keys.params
    lut = oracle.generate_lut(p, [lambda x: (x + 1) % 8], 3)
    rng = np.random.default_rng(batch)
    msgs = rng.integers(0, 8, batch)
    cts = np.zeros((batch, keys.lwe0_len), dtype=np.uint64)
    for m in range(batch):
        oracle.lib().orc_encrypt_lwe(C.byref(client.rng), cts[m], keys.lwe0_sk, p.lwe_n, p.lwe_std, int(msgs[m]) << 60)
    out = evaluation.programmable_bootstrap(cts, lut)
    idx = sorted({0, 1, 147, 148, 149, 295, 296, 443, 444, 445, 591, 592, 887, 888, batch - 2, batch - 1} & set(range(batch)))
    for i in idx:
        assert int(oracle.decode(client.decrypt_glwe_l1_raw(out[i])[:1], 3)[0]) == (msgs[i] + 1) % 8, (batch, i)


def test_short_lwe_through_every_kernel():
    """tools/sanitizer_probe.py: DEFAULT_128 rings with a 16-step blind rotation through every kernel
    (quad and pair-team PBS, trace / scheme switch, wide and bulk CMUX, tensor-core and IMAD keyswitch);
    also exercises a non-default l0 dimension end to end."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "sanitizer_probe.py")], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and "sanitizer probe: ok" in r.stdout, r.stdout + r.stderr


def test_rlwe_encrypt_public_bit_exact(oracle, keys, evaluation):
    """spf_b200_rlwe_encrypt_public vs the oracle's rlwe_encrypt_public_impl (rlwe_encryption.rs:125-160): integer work,
    bit-exact, for the reference's binary u and for arbitrary u64 multipliers; ragged batches; decrypts like
    can_rlwe_public_key_encrypt (:188-211)."""
    c = oracle.Client(keys, seed=0xC0FFEE)
    p = keys.params
    n = p.glwe_n
    pk = c.generate_public_key()
    rng = np.random.default_rng(9)
    for batch in (1, 3, 301):
        bits = rng.integers(0, 2, (batch, n), dtype=np.uint64)
        msg = bits << np.uint64(63)
        rnd = [c.rlwe_randomness() for _ in range(batch)]
        u, e0, e1 = (np.stack([r[i] for r in rnd]) for i in range(3))
        got = evaluation.rlwe_encrypt_public(pk, msg, u, e0, e1)
        for i in sorted({0, batch // 2, batch - 1}):
            assert np.array_equal(got[i], oracle.rlwe_encrypt_public(p, msg[i], pk, u[i], e0[i], e1[i])), (batch, i)
            assert np.array_equal(c.decrypt_glwe_l1(got[i]), bits[i])
    # any u64 multiplier, any key material
    pk2 = rng.integers(0, 1 << 64, 2 * n, dtype=np.uint64)
    m, u, e0, e1 = (rng.integers(0, 1 << 64, (2, n), dtype=np.uint64) for _ in range(4))
    got = evaluation.rlwe_encrypt_public(pk2, m, u, e0, e1)
    for i in range(2):
        assert np.array_equal(got[i], oracle.rlwe_encrypt_public(p, m[i], pk2, u[i], e0[i], e1[i]))
    # empty batch and bad shapes
    assert evaluation.rlwe_encrypt_public(pk, np.zeros((0, n), np.uint64), np.zeros((0, n), np.uint64),
                                          np.zeros((0, n), np.uint64), np.zeros((0, n), np.uint64)).shape == (0, 2 * n)
    import spf_b200
    with pytest.raises(spf_b200.SpfError):
        evaluation.rlwe_encrypt_public(pk[:n], m, u, e0, e1)
