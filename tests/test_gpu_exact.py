"""GPU kernels against the oracle BIT FOR BIT, in the exact regime (tests/exact_keys.py: integer-polynomial keys, NOT
secure).  With such keys every inverse transform is an integer far below 2^53, so the device's FFT and the oracle's
independent C code round to the same values and whole blind rotations, traces and CMUXes of ARBITRARY u64 inputs are
comparable byte for byte (tests/test_exact_regime.py guards that premise on the CPU).  What is checked here is the device
machinery the host emulator does not model -- the BSK ring of pbs_kernel, the staged-row prefetch of pbs_quad_kernel,
the wave / tail split of launch_pbs, the packed CBS remainder on the side stream, the per-CTA layouts of trace_ss_kernel
and of the CMUX kernels -- on every item of every batch unless stated.

Batch sizes name launch layouts of a 148-SM B200 (capi.cu launch_pbs / launch_cbs / launch_trace_ss / launch_cmux):
  * PBS, batch <= 148: pbs_quad_kernel, CTA c = item c.
  * PBS, 149 <= batch <= 444: pbs_kernel, per = 2 pairs per CTA up to 296 items, 3 above; grid = min(ceil(batch / per),
    148); pair p of CTA b takes items p * grid + b, p * grid + b + grid * per, ...  (slots numbered pair-major, so a
    ragged last round leaves pairs with fewer items, which count themselves off the BSK ring).
  * PBS, batch > 444 = one wave (148 CTAs x 3 pairs): remainder r = batch % 444; 0 < r <= 148: the full waves on
    pbs_kernel, the r-item tail on pbs_quad_kernel (445 = 444 + 1, 494 = 444 + 50, 889 = 2 x 444 + 1); r > 148 (593 =
    444 + 149): the whole batch on pbs_kernel, ragged last round.
  * CBS of 4096 = 9 x 444 + 100 through the device entry point: full waves on the compute stream, the 100-item remainder
    packed three to an SM on the side stream, concurrently with the full waves' trace kernels.
  * Trace: one team per item, up to 4 per CTA (fewer for small batches).
  * CMUX: cmux_wide_kernel (one CTA per output) up to 296 outputs, cmux_kernel (one team per output) above.
The host-pointer entry points cut batches into chunks of one PBS wave, so the multi-wave PBS and CBS layouts are reached
through the device-pointer entry points.
"""
import ctypes as C

import numpy as np
import pytest

from exact_keys import exact_ggsw, exact_keys, interleaved_masks, par_map, random_u64

pytestmark = pytest.mark.gpu

N = 2048
GLWE = 2 * N
WAVE = 444


@pytest.fixture(scope="module")
def xk(oracle):
    return exact_keys(0xE0AC7 + 1)


@pytest.fixture(scope="module")
def xev(xk):
    import spf_b200

    ev = spf_b200.Evaluation(xk.bsk_fft, xk.ksk, xk.ssk_fft, xk.ak_fft)
    yield ev
    ev.close()


def _to_dev(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8)).to("cuda")


def _dev_empty(nbytes):
    import torch

    return torch.empty(nbytes, dtype=torch.uint8, device="cuda")


def _dev_pbs(ev, lwe, lut, log_chi=0, log_v=0):
    """spf_b200_dev_programmable_bootstrap: the whole batch is one launch_pbs (no host-side chunking)."""
    import torch

    d_in, d_lut, d_out = _to_dev(lwe), _to_dev(lut), _dev_empty(lwe.shape[0] * GLWE * 8)
    torch.cuda.synchronize()
    ev.dev_programmable_bootstrap(d_out.data_ptr(), d_in.data_ptr(), d_lut.data_ptr(), log_chi, log_v, lwe.shape[0])
    ev.synchronize()
    return d_out.cpu().numpy().view(np.uint64).reshape(-1, GLWE)


def _assert_items_equal(got, want, items, what):
    bad = [int(c) for c, w in zip(items, want) if not np.array_equal(got[c], w)]
    assert not bad, f"{what}: {len(bad)} of {len(want)} items differ, first {bad[:12]}"


# ---- 1. PBS at every launch layout, skipped steps interleaved ----------------------------------------------------------

@pytest.fixture(scope="module")
def pbs_case(oracle, xk):
    """889 LWEs cycling through the mask patterns of exact_keys.MASK_KINDS (random, all-zero, every 2nd / 3rd / 7th step
    zero, first / last step zero, long zero runs, 2^64 - 1, half-way values), a random u64 LUT, and the oracle's PBS of
    each; batch b of the layout tests is the first b items."""
    lwe, _ = interleaved_masks(889, 0xB5)
    lut = random_u64(np.random.default_rng(0xB6), GLWE)
    return lwe, lut, np.stack(par_map(lambda x: oracle.pbs_generalized(xk, x, lut), lwe))


@pytest.mark.parametrize("batch", [
    pytest.param(1, id="1-quad"), pytest.param(3, id="3-quad"), pytest.param(148, id="148-quad-full"),
    pytest.param(149, id="149-pair-2perCTA"), pytest.param(297, id="297-pair-3perCTA"),
    pytest.param(445, id="445-wave-quad-tail1"), pytest.param(494, id="494-wave-quad-tail50"),
    pytest.param(593, id="593-pair-remainder-too-large-for-tail"), pytest.param(889, id="889-2waves-quad-tail1")])
def test_pbs_every_layout_bit_exact(xev, pbs_case, batch):
    lwe, lut, ref = pbs_case
    got = _dev_pbs(xev, lwe[:batch], lut)
    _assert_items_equal(got, ref[:batch], range(batch), f"PBS batch {batch}")


# ---- 2. log_chi / log_v ------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def sweep_inputs():
    lwe, _ = interleaved_masks(300, 0xC1)
    return lwe, random_u64(np.random.default_rng(0xC2), GLWE)


@pytest.mark.parametrize("log_chi,log_v", [(0, 1), (0, 3), (2, 0), (3, 2), (5, 6), (0, 11), (11, 0), (4, 7)])
def test_pbs_log_chi_log_v_bit_exact(oracle, xk, xev, sweep_inputs, log_chi, log_v):
    """generalized_programmable_bootstrap's (log_chi, log_v) on the quad kernel (batch 40) and the pair kernel (batch
    300), up to log_chi + log_v = 11."""
    lwe, lut = sweep_inputs
    ref = np.stack(par_map(lambda x: oracle.pbs_generalized(xk, x, lut, log_chi, log_v), lwe))
    _assert_items_equal(_dev_pbs(xev, lwe[:40], lut, log_chi, log_v), ref[:40], range(40), "quad")
    _assert_items_equal(_dev_pbs(xev, lwe, lut, log_chi, log_v), ref, range(300), "pair")


def test_pbs_log_chi_log_v_out_of_range(xk, xev):
    import spf_b200

    lwe = np.zeros((1, xk.lwe0_len), dtype=np.uint64)
    lut = np.zeros(GLWE, dtype=np.uint64)
    for lc, lv in ((0, 12), (12, 0), (6, 6)):
        with pytest.raises(spf_b200.SpfError) as e:
            xev.programmable_bootstrap(lwe, lut, lc, lv)
        assert e.value.code == -1
        with pytest.raises(spf_b200.SpfError):
            _dev_pbs(xev, lwe, lut, lc, lv)


# ---- 3. initial rotation LUT X^-b~, oracle-free --------------------------------------------------------------------------

def _rotate(lut, d):
    """LUT * X^-d for both polynomials, numpy (negacyclic: X^N = -1)."""
    j = (np.arange(N) + d) % (2 * N)
    out = lut.reshape(2, N)[:, j % N].copy()
    out[:, j >= N] = np.uint64(0) - out[:, j >= N]
    return out.reshape(-1)


@pytest.mark.parametrize("batch", [pytest.param(4096, id="4096-waves-quad-tail"), pytest.param(148, id="148-quad")])
def test_initial_rotation_sweep(xk, xev, batch):
    """Zero masks: every blind-rotation step is skipped and the output is LUT X^-b~ exactly.  b = k 2^52 for every
    k = 0 .. 4095 (4096 items: nine full pbs_kernel waves and a 100-item pbs_quad_kernel tail), checked against numpy
    rotations of a random LUT; then half-way values k 2^52 + 2^51 (round up to k + 1) and k 2^52 + 2^51 - 1 (round
    down to k)."""
    rng = np.random.default_rng(batch)
    lut = random_u64(rng, GLWE)
    k = np.arange(4096, dtype=np.uint64) if batch == 4096 else rng.choice(4096, batch, replace=False).astype(np.uint64)
    for extra, up in ((0, 0), (1 << 51, 1), ((1 << 51) - 1, 0)):
        lwe = np.zeros((batch, xk.lwe0_len), dtype=np.uint64)
        lwe[:, -1] = (k << np.uint64(52)) + np.uint64(extra)
        got = _dev_pbs(xev, lwe, lut)
        bad = [c for c in range(batch) if not np.array_equal(got[c], _rotate(lut, (int(k[c]) + up) % 4096))]
        assert not bad, f"b = k 2^52 + {extra}: {len(bad)} items wrong, k = {[int(k[c]) for c in bad[:8]]}"


# ---- 4. trace ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("batch", [1, 4, 5, 150, 600, 601, 1199])
def test_trace_bit_exact(oracle, xk, xev, batch):
    """Random u64 GLWEs: 1 / 4 / 5 items (one per CTA), 150 (two per CTA), 600 (four per CTA, exactly 150 CTAs: a second
    wave of 2), 601 (ragged last CTA), 1199 (many waves, ragged)."""
    g = random_u64(np.random.default_rng(batch), batch, GLWE)
    _assert_items_equal(xev.trace(g), par_map(lambda x: oracle.trace(xk, x), g), range(batch), f"trace batch {batch}")


# ---- 5. circuit bootstrap --------------------------------------------------------------------------------------------------

CBS_REL_BAR = 1e-14  # ~100 x the f64 rounding measured between the oracle and the emulator (8.8e-17)


def _cbs_rel_err(got, ref):
    return float((np.abs(got - ref).max(axis=1) / np.abs(ref).max(axis=1)).max())


def _record_cbs(key, value):
    from test_gpu_distances import _record

    _record(key, value)
    print(f"{key} = {value:.3g}")


@pytest.mark.parametrize("batch", [pytest.param(2, id="2-quad"), pytest.param(300, id="300-pair")])
def test_cbs_fft_domain(oracle, xk, xev, batch):
    """Random u64 L0 LWEs: the output GGSWs are FFT-domain transforms of full-size torus values, equal to the oracle's
    up to f64 rounding only; every item."""
    lwe = random_u64(np.random.default_rng(batch), batch, xk.lwe0_len)
    got = xev.circuit_bootstrap(lwe)
    err = _cbs_rel_err(got, oracle.circuit_bootstrap_batch(xk, lwe))
    _record_cbs(f"exact_cbs_rel_err_b{batch}", err)
    assert err <= CBS_REL_BAR, err


def test_cbs_4096_packed_remainder(oracle, xk, xev):
    """4096 = 9 x 444 + 100 through spf_b200_dev_circuit_bootstrap: the 100-item remainder runs packed on the side
    stream.  Checked: all 100 remainder items, and one item on every CTA of the full waves (item r 444 + p 148 + b on
    CTA b, pair p, round r, with p and r cycling over b)."""
    import torch

    B = 4096
    lwe = random_u64(np.random.default_rng(0xCB5), B, xk.lwe0_len)
    d_in, d_out = _to_dev(lwe), _dev_empty(B * xk.ggsw_fft_len * 16)
    torch.cuda.synchronize()
    xev.dev_circuit_bootstrap(d_out.data_ptr(), d_in.data_ptr(), B, reference_scale=True)
    xev.synchronize()
    got = d_out.cpu().numpy().view(np.complex128).reshape(B, -1)
    items = sorted({(b % 9) * WAVE + (b % 3) * 148 + b for b in range(148)} | set(range(9 * WAVE, B)))
    ref = oracle.circuit_bootstrap_batch(xk, lwe[items])
    err = _cbs_rel_err(got[items], ref)
    _record_cbs("exact_cbs_rel_err_b4096", err)
    assert err <= CBS_REL_BAR, err
    # the batch is all one computation: items outside the sample equal the same inputs bootstrapped in a small batch
    again = xev.circuit_bootstrap(lwe[[5, 2000, 3995]])
    assert np.array_equal(again.view(np.uint64), got[[5, 2000, 3995]].view(np.uint64))


def test_cbs_stages_bit_exact(oracle, xk, xev):
    """The staged circuit bootstrap in the exact regime: the multi-function blind rotation (b + q/4, CBS LUT, log_v = 2)
    equals oracle.cbs_pbs_stage, and the trace of the pre-processed levels equals oracle.cbs_trace_stage, bit for bit."""
    from test_gpu_parity import _cbs_preprocess

    p = xk.params
    lwe = random_u64(np.random.default_rng(0xC5), 6, xk.lwe0_len)
    rot = lwe.copy()
    rot[:, -1] += np.uint64(1 << 62)
    lut = np.zeros(GLWE, dtype=np.uint64)
    oracle.lib().orc_cbs_lut(lut, C.byref(p))
    x = xev.programmable_bootstrap(rot, lut, 0, 2)
    _assert_items_equal(x, [oracle.cbs_pbs_stage(xk, c) for c in lwe], range(6), "cbs_pbs_stage")
    pre = np.stack([_cbs_preprocess(x[c], lv, p) for c in range(6) for lv in range(p.cbs.count)])
    glev = xev.trace(pre).reshape(6, -1)
    _assert_items_equal(glev, [oracle.cbs_trace_stage(xk, g) for g in x], range(6), "cbs_trace_stage")


# ---- 6. CMUX family ----------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cmux_case(oracle, xk):
    """600 (selector, a, b): distinct exact GGSWs, random u64 GLWEs, and the oracle's CMUX of each."""
    rng = np.random.default_rng(0xC3)
    sel = np.stack([exact_ggsw(rng, xk) for _ in range(600)])
    a, b = random_u64(rng, 600, GLWE), random_u64(rng, 600, GLWE)
    return sel, a, b, np.stack(par_map(lambda i: oracle.cmux(xk, a[i], b[i], sel[i]), range(600)))


@pytest.mark.parametrize("batch", [pytest.param(1, id="1-wide"), pytest.param(148, id="148-wide"),
                                   pytest.param(296, id="296-wide"), pytest.param(297, id="297-bulk"),
                                   pytest.param(600, id="600-bulk")])
def test_cmux_bit_exact(xev, cmux_case, batch):
    sel, a, b, ref = cmux_case
    _assert_items_equal(xev.cmux(sel[:batch], a[:batch], b[:batch]), ref[:batch], range(batch), f"cmux batch {batch}")


@pytest.mark.parametrize("batch", [pytest.param(5, id="5-wide"), pytest.param(297, id="297-bulk")])
def test_multiply_glwe_ggsw_bit_exact(oracle, xk, xev, cmux_case, batch):
    sel, _, b, _ = cmux_case
    want = par_map(lambda i: oracle.multiply_glwe_ggsw(xk, b[i], sel[i]), range(batch))
    _assert_items_equal(xev.multiply_glwe_ggsw(b[:batch], sel[:batch]), want, range(batch), "multiply_glwe_ggsw")


@pytest.mark.parametrize("batch", [pytest.param(3, id="3-wide"), pytest.param(80, id="80-bulk")])
def test_glev_cmux_bit_exact(oracle, xk, xev, cmux_case, batch):
    """glev_cmux: the l_cbs = 4 GLWEs of an item share its selector (12 outputs: wide kernel, 320: bulk kernel)."""
    sel = cmux_case[0]
    rng = np.random.default_rng(batch)
    d0, d1 = random_u64(rng, batch, xk.glev_len), random_u64(rng, batch, xk.glev_len)
    want = par_map(lambda i: oracle.glev_cmux(xk, d0[i], d1[i], sel[i]), range(batch))
    _assert_items_equal(xev.glev_cmux(sel[:batch], d0, d1), want, range(batch), "glev_cmux")


@pytest.mark.parametrize("stride,batch", [pytest.param(0, 5, id="ggsw_stride0-5-wide"),
                                          pytest.param(0, 300, id="ggsw_stride0-300-bulk"),
                                          pytest.param(1, 300, id="full_stride-300-bulk")])
def test_dev_cmux_bit_exact(oracle, xk, xev, cmux_case, stride, batch):
    """spf_b200_dev_cmux with one selector shared by the whole batch (ggsw_stride = 0) and with one per item."""
    import torch

    sel, a, b, ref = cmux_case
    s = sel[:1] if stride == 0 else sel[:batch]
    d_sel, d_a, d_b = _to_dev(s / 1024.0), _to_dev(a[:batch]), _to_dev(b[:batch])  # device scale: x 2^-10, exact
    d_out = _dev_empty(batch * GLWE * 8)
    torch.cuda.synchronize()
    xev.dev_cmux(d_out.data_ptr(), d_sel.data_ptr(), stride * xk.ggsw_fft_len, d_a.data_ptr(), d_b.data_ptr(), batch)
    xev.synchronize()
    got = d_out.cpu().numpy().view(np.uint64).reshape(batch, GLWE)
    want = ref[:batch] if stride else par_map(lambda i: oracle.cmux(xk, a[i], b[i], sel[0]), range(batch))
    _assert_items_equal(got, want, range(batch), f"dev_cmux stride {stride}")


# ---- 7. graph: MUX tree -> sample extract -> keyswitch ------------------------------------------------------------------

def test_graph_mux_tree_then_keyswitch_bit_exact(oracle, xk, xev):
    """A depth-3 MUX tree over 8 random u64 GLWE leaves with exact selectors (InputGgsw1), then SampleExtract ->
    KeyswitchL1toL0 at several indices, through the graph executor.  A CMUX of a CMUX output stays exact (its digits are
    bounded whatever the GLWE), so every output equals the oracle's composition bit for bit."""
    import spf_b200

    rng = np.random.default_rng(0x6A)
    leaves = random_u64(rng, 8, GLWE)
    sels = [exact_ggsw(rng, xk) for _ in range(7)]
    idx = [0, 1, 1000, 2047]
    root = np.zeros(GLWE, dtype=np.uint64)
    l0s = [np.zeros(xk.lwe0_len, dtype=np.uint64) for _ in idx]
    c = spf_b200.FheCircuit()
    level = [c.add("InputGlwe1", io=x) for x in leaves]
    want = list(leaves)
    s = 0
    while len(level) > 1:
        nxt, wnxt = [], []
        for j in range(0, len(level), 2):
            ns = c.add("InputGgsw1", io=sels[s])
            nxt.append(c.add("CMux", ns, level[j], level[j + 1]))
            wnxt.append(oracle.cmux(xk, want[j], want[j + 1], sels[s]))
            s += 1
        level, want = nxt, wnxt
    c.add("OutputGlwe1", level[0], io=root)
    for h, out in zip(idx, l0s):
        c.add("OutputLwe0", c.add("KeyswitchL1toL0", c.add("SampleExtract", level[0], arg=h)), io=out)
    spf_b200.CircuitProcessor(xev).run_graph_blocking(c)
    assert np.array_equal(root, want[0])
    for h, out in zip(idx, l0s):
        assert np.array_equal(out, oracle.keyswitch_lwe(xk, oracle.sample_extract(xk, want[0], h))), h
