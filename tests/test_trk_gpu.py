"""GPU parity tests for the tracking correlator, all through the C ABI (libb200gnss.so).

Oracles: the reference's own Cpu_Multicorrelator_Real_Codes / volk_gnsssdr kernels
(oracle.ref, prebuilt oracle/_ref/liboracle_ref.so) when present, else the pinned C port
(oracle.port); plus the float64 truth.  Tolerances:
  * integer-exact configurations: EXACT equality (this is what pins the chip indices);
  * float data: |gpu - avx_oracle| / |avx_oracle| < 1e-3  (the reference's own SIMD-vs-generic
    bound, VG lib/kernel_tests.h:41,87-89) and |gpu - f64 truth| < 1e-5 * |prompt|.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from gnss_synth import make_iq, trk_params_for  # noqa: E402


@pytest.fixture(scope="module")
def capi():
    import gnss_sdr_b200.capi as c
    return c


@pytest.fixture(scope="module")
def engine(capi):
    e = capi.Engine(0)
    yield e
    e.close()


def int_oracle(x_int, code_int, idx):
    """exact integer correlation given chip indices (taps x n)."""
    return np.array([np.sum(x_int * code_int[idx[t]]) for t in range(idx.shape[0])], dtype=np.int64)


SHAPES = [
    # n, L, shifts, rem, step
    (25000, 1023, [-0.5, 0.0, 0.5], 0.37, 1.023e6 * (1 + 3000 / 1575.42e6) / 25e6),
    (25001, 1023, [-0.5, 0.0, 0.5], 0.93, 1.023e6 * (1 - 4500 / 1575.42e6) / 25e6),
    (200000, 8184, [-1.2, -0.3, 0.0, 0.3, 1.2], 1.71, 2 * 1.023e6 / 50e6),
    (4000, 1023, [-0.5, 0.0, 0.5], -0.25, 1.023e6 / 4e6),
    (8111, 2046, [-0.1, 0.0, 0.1], -0.234, (2046 + 0.1) / 8111),
    (511, 1023, [-0.5, 0.0, 0.5], 0.1, 1.9),
    (512, 1023, [-0.5, 0.0, 0.5], 0.1, 1.9),
    (513, 1023, [-0.5, 0.0, 0.5], 0.1, 1.9),
    (1031, 1023, [0.0], 0.6, 0.99),
    (7, 11, [-0.5, 0.0], 0.2, 1.9),
    (1, 1023, [-0.5, 0.0, 0.5], 0.0, 0.04),
    (100000, 1023, [-0.5, 0.0, 0.5], 0.37, 0.0409),        # 4 code periods: general (modulo) path
    (6000, 1023, [-700.25, 0.0, 1500.5], 3.3, 0.7),         # far-apart taps: general path
    (3000, 1023, [-0.5, -0.25, -0.1, 0.0, 0.1, 0.25, 0.5, 0.75], 0.3, 0.341),  # 8 taps
    (3000, 1023, [-0.5, 0.5], 0.3, 0.341),
    (3000, 1023, [-0.5, -0.2, 0.2, 0.5], 0.3, 0.341),
]


@pytest.mark.parametrize("n,L,shifts,rem,step", SHAPES)
def test_single_correlator_integer_exact(capi, engine, oracle, n, L, shifts, rem, step):
    """Small-integer samples and code values, zero carrier: every partial sum is an exactly
    representable integer, so the GPU result must EQUAL the integer oracle built from the
    AVX-association chip indices.  One wrong index changes the sum."""
    rng = np.random.default_rng(n + L)
    x_int = rng.integers(-7, 8, n)
    x_int[x_int == 0] = 1
    code_int = ((np.arange(L) * 7919) % 31) - 15
    code_int[code_int == 0] = 16
    _, idx = oracle.port.resampler(1, code_int.astype(np.float32), rem, step, shifts, n, return_idx=True)
    want = int_oracle(x_int, code_int, idx)
    mc = capi.Multicorrelator(engine, n, len(shifts))
    mc.set_high_dynamics_resampler(False)
    mc.set_local_code_and_taps(code_int.astype(np.float32), shifts)
    got = mc.Carrier_wipeoff_multicorrelator_resampler(x_int.astype(np.complex64), 0.0, 0.0, 0.0, rem, step, 0.0)
    mc.free()
    assert np.array_equal(got.real.astype(np.int64), want)
    assert np.all(got.imag == 0)


@pytest.mark.parametrize("first,offset", [(0, 0), (0, 1), (0, 2), (0, 3), (0, 255), (0, 511), (0, 513),
                                          (1000000, 0), (1000000, 1), (1000000, 2047), (5000, 7)])
def test_batch_sample_offsets_integer_exact(capi, engine, oracle, first, offset):
    """Epochs starting at odd/even absolute sample indices of a shared ring band (alignment
    peel), including epochs that wrap around the end of the ring."""
    n, L, shifts, rem, step = 5003, 1023, [-0.5, 0.0, 0.5], 0.37, 0.2051
    rng = np.random.default_rng(first + offset)
    total = 8192
    x_int = rng.integers(-7, 8, total)
    code_int = ((np.arange(L) * 7919) % 31) - 15
    e = engine
    band = 3
    e.iq_create(band, total)
    # advance the ring so absolute indices are large and the data wraps around the ring end
    pad = np.zeros(total, np.complex64)
    done = 0
    while done < first:
        k = min(total, first - done)
        e.iq_push(band, pad[:k])
        done += k
    f0 = e.iq_push(band, x_int.astype(np.complex64))
    assert f0 == first
    cid = e.channel_create(band, 3)
    e.channel_set_code(cid, code_int.astype(np.float32), shifts)
    s_idx = first + offset
    items = np.zeros(1, capi.TRK_ITEM_DTYPE)
    items["channel"] = cid
    items["n"] = n
    items["sample_index"] = s_idx
    items["rem_code_phase_chips"] = rem
    items["code_phase_step_chips"] = step
    got = e.trk_batch(items, 3)[0]
    xs = x_int[offset: offset + n]
    _, idx = oracle.port.resampler(1, code_int.astype(np.float32), rem, step, shifts, n, return_idx=True)
    want = int_oracle(xs, code_int, idx)
    assert np.array_equal(got.real.astype(np.int64), want)
    assert np.all(got.imag == 0)


def _ref_or_port_avx(oracle, iq, code, shifts, rem_carr, dphi, rem_code, step):
    if oracle.ref is not None:
        oracle.ref.select_arch("a_avx")
        h = oracle.ref.mc_create(len(iq), len(shifts), high_dyn=False)
        oracle.ref.mc_set_code(h, code, shifts)
        out = oracle.ref.mc_correlate(h, iq, len(shifts), rem_carr, dphi, 0.0, rem_code, step, 0.0)
        oracle.ref.mc_destroy(h)
        return out
    return oracle.port.multicorrelator(1, iq, code, shifts, rem_carr, dphi, rem_code, step)


@pytest.mark.parametrize("fs,n,prn,doppler,shifts", [
    (25e6, 25000, 7, 3217.0, [-0.5, 0.0, 0.5]),
    (25e6, 25000, 19, -4711.0, [-0.5, 0.0, 0.5]),
    (4e6, 4000, 1, 1680.0, [-0.5, 0.0, 0.5]),
    (4e6, 8000, 3, -2500.0, [-0.25, 0.0, 0.25]),
])
def test_single_correlator_signal_parity(capi, engine, oracle, fs, n, prn, doppler, shifts):
    code = oracle.port.gps_ca_code(prn)
    sv = dict(prn=prn, doppler=doppler, code_phase_chips=417.3, cn0=45.0, phase0=0.9)
    iq = make_iq({prn: code}, fs, n, [sv], seed=prn)
    _, rem_carr, dphi, rem_code, step = trk_params_for(sv, fs, n, 1)
    args = (float(rem_carr[0]), float(dphi[0]), float(rem_code[0]), float(step[0]))
    want = _ref_or_port_avx(oracle, iq, code, shifts, *args)
    truth = oracle.port.multicorrelator_f64(1, iq, code, shifts, *args)
    mc = capi.Multicorrelator(engine, n, len(shifts))
    mc.set_high_dynamics_resampler(False)
    mc.set_local_code_and_taps(code, shifts)
    got = mc.Carrier_wipeoff_multicorrelator_resampler(iq, args[0], args[1], 0.0, args[2], args[3], 0.0)
    mc.free()
    # the prompt must be a real peak for the test to mean anything
    assert np.abs(truth[1]) > 5 * np.sqrt(n)
    assert np.all(np.abs(got - want) / np.abs(want) < 1e-3)            # the reference's own bound
    assert np.max(np.abs(got - truth)) / np.abs(truth[1]) < 1e-5         # vs float64 truth
    # and we must be at least as close to the truth as the reference's SIMD path is
    assert np.max(np.abs(got - truth)) <= np.max(np.abs(want - truth)) * 1.5 + 1e-6 * np.abs(truth[1])


def test_galileo_e1_five_taps_parity(capi, engine, oracle):
    """C3 shape: N=200000 @ 50 Msps, sinBOC(1,1) table of 8184 values, VE/E/P/L/VL."""
    rng = np.random.default_rng(33)
    primary = rng.choice([-1, 1], 4092)
    code = oracle.port.sinboc11(primary)
    fs, n = 50e6, 200000
    shifts = np.array([-0.6, -0.15, 0.0, 0.15, 0.6], np.float32) * 2
    sv = dict(prn=1, doppler=-1234.5, code_phase_chips=1000.25, cn0=42.0, phase0=2.1)
    iq = make_iq({1: code}, fs, n, [sv], seed=33, chips_per_table_chip=2.0)
    _, rem_carr, dphi, rem_code, step = trk_params_for(sv, fs, n, 1, table_chips_per_chip=2.0, L=8184)
    args = (float(rem_carr[0]), float(dphi[0]), float(rem_code[0]), float(step[0]))
    want = _ref_or_port_avx(oracle, iq, code, shifts, *args)
    truth = oracle.port.multicorrelator_f64(1, iq, code, shifts, *args)
    mc = capi.Multicorrelator(engine, n, 5)
    mc.set_high_dynamics_resampler(False)
    mc.set_local_code_and_taps(code, shifts)
    got = mc.Carrier_wipeoff_multicorrelator_resampler(iq, args[0], args[1], 0.0, args[2], args[3], 0.0)
    mc.free()
    assert np.abs(truth[2]) > 5 * np.sqrt(n)
    assert np.all(np.abs(got - want) / np.abs(want) < 1e-3)
    assert np.max(np.abs(got - truth)) / np.abs(truth[2]) < 1e-5


def test_batch_c2_slice_of_baseline_config(capi, engine, oracle):
    """C2 (32 channels x 25 Msps) on a 40-epoch slice: batched launch == per-epoch oracle."""
    fs, n, nch, nep = 25e6, 25000, 32, 40
    rng = np.random.default_rng(2)
    codes = {p: oracle.port.gps_ca_code(p) for p in range(1, nch + 1)}
    svs = [dict(prn=p, doppler=float(rng.uniform(-5000, 5000)), code_phase_chips=float(rng.uniform(0, 1023)),
                cn0=45.0, phase0=float(rng.uniform(0, 6.28))) for p in range(1, nch + 1)]
    iq = make_iq(codes, fs, n * nep + 64, svs, seed=2)
    e = engine
    band = 1
    e.iq_create(band, len(iq))
    first = e.iq_push(band, iq)
    shifts = [-0.5, 0.0, 0.5]
    items = np.zeros(nch * nep, capi.TRK_ITEM_DTYPE)
    cids = []
    for sv in svs:
        cid = e.channel_create(band, 3)
        e.channel_set_code(cid, codes[sv["prn"]], shifts)
        cids.append(cid)
    params = []
    for c, sv in enumerate(svs):
        s, rc, dp, rcode, st = trk_params_for(sv, fs, n, nep)
        for k in range(nep):
            it = items[k * nch + c]   # epoch-major order: channels of one epoch are neighbours
            it["channel"] = cids[c]
            it["n"] = n
            it["sample_index"] = first + int(s[k])
            it["rem_carrier_phase_rad"] = rc[k]
            it["phase_step_rad"] = dp[k]
            it["rem_code_phase_chips"] = rcode[k]
            it["code_phase_step_chips"] = st[k]
    got = e.trk_batch(items, 3)
    # oracle on a subset of items (every 7th) to keep the CPU side quick
    worst_ref, worst_truth = 0.0, 0.0
    for i in range(0, len(items), 7):
        it = items[i]
        sv = svs[i % nch]
        seg = iq[int(it["sample_index"]) - first: int(it["sample_index"]) - first + n]
        a = (float(it["rem_carrier_phase_rad"]), float(it["phase_step_rad"]), float(it["rem_code_phase_chips"]),
             float(it["code_phase_step_chips"]))
        want = _ref_or_port_avx(oracle, seg, codes[sv["prn"]], shifts, *a)
        truth = oracle.port.multicorrelator_f64(1, seg, codes[sv["prn"]], shifts, *a)
        worst_ref = max(worst_ref, float(np.max(np.abs(got[i] - want) / np.abs(want))))
        worst_truth = max(worst_truth, float(np.max(np.abs(got[i] - truth)) / np.abs(truth[1])))
        assert np.abs(truth[1]) > 3 * np.sqrt(n)
    assert worst_ref < 1e-3
    assert worst_truth < 1e-5


def test_batch_slices_agree_and_are_deterministic(capi, engine, oracle):
    """Splitting an epoch over 1..64 CTAs changes only the float summation order (tiny) and
    repeated launches are bitwise identical (deterministic cross-CTA combine)."""
    import torch
    n, L = 25000, 1023
    rng = np.random.default_rng(5)
    iq = (rng.standard_normal(n + 8) + 1j * rng.standard_normal(n + 8)).astype(np.complex64)
    code = oracle.port.gps_ca_code(5)
    e = engine
    band = 2
    iq_t = torch.from_numpy(iq.view(np.float32)).cuda()
    e.iq_attach_dev(band, iq_t.data_ptr(), n + 8, 0)
    cid = e.channel_create(band, 3)
    e.channel_set_code(cid, code, [-0.5, 0.0, 0.5])
    items = np.zeros(1, capi.TRK_ITEM_DTYPE)
    items["channel"] = cid
    items["n"] = n
    items["sample_index"] = 3
    items["rem_carrier_phase_rad"] = 0.3
    items["phase_step_rad"] = 1e-3
    items["rem_code_phase_chips"] = 0.2
    items["code_phase_step_chips"] = 0.04092
    items_t = torch.from_numpy(items.view(np.uint8)).cuda()
    outs = {}
    for slices in (1, 2, 7, 16, 64):
        reps = []
        for _ in range(3):
            out_t = torch.zeros(8, 2, dtype=torch.float32, device="cuda")
            e.trk_batch_dev(items_t.data_ptr(), 1, out_t.data_ptr(), 8, slices)
            e.sync()
            reps.append(out_t.cpu().numpy().copy())
        assert np.array_equal(reps[0], reps[1]) and np.array_equal(reps[0], reps[2])
        outs[slices] = reps[0][:3, 0] + 1j * reps[0][:3, 1]
    for s, v in outs.items():
        assert np.max(np.abs(v - outs[1])) / np.max(np.abs(outs[1])) < 2e-5, s


def test_mixed_tap_counts_in_one_batch(capi, engine, oracle):
    """Galileo-style: a 5-tap pilot channel and a 1-tap data channel in the same launch
    (dll_pll_veml_tracking.cc:1246-1256)."""
    n, L = 6000, 2046
    rng = np.random.default_rng(8)
    x_int = rng.integers(-7, 8, n)
    code_a = ((np.arange(L) * 7919) % 31) - 15
    code_b = ((np.arange(L) * 104729) % 29) - 14
    e = engine
    band = 4
    e.iq_create(band, 8192)
    first = e.iq_push(band, x_int.astype(np.complex64))
    sh5 = [-1.2, -0.3, 0.0, 0.3, 1.2]
    ca = e.channel_create(band, 5)
    cb = e.channel_create(band, 1)
    e.channel_set_code(ca, code_a.astype(np.float32), sh5)
    e.channel_set_code(cb, code_b.astype(np.float32), [0.0])
    items = np.zeros(2, capi.TRK_ITEM_DTYPE)
    items["channel"] = [ca, cb]
    items["n"] = n
    items["sample_index"] = first
    items["rem_code_phase_chips"] = 0.41
    items["code_phase_step_chips"] = 0.3411
    got = e.trk_batch(items, 5)
    _, ia = oracle.port.resampler(1, code_a.astype(np.float32), 0.41, 0.3411, sh5, n, return_idx=True)
    _, ib = oracle.port.resampler(1, code_b.astype(np.float32), 0.41, 0.3411, [0.0], n, return_idx=True)
    assert np.array_equal(got[0].real.astype(np.int64), int_oracle(x_int, code_a, ia))
    assert np.array_equal(got[1, :1].real.astype(np.int64), int_oracle(x_int, code_b, ib))


def test_error_paths(capi, engine):
    with pytest.raises(capi.B200Error):
        capi.Multicorrelator(engine, 1000, 9)         # too many taps
    mc = capi.Multicorrelator(engine, 1000, 3)
    with pytest.raises(capi.B200Error):               # correlate before set_local_code
        mc.Carrier_wipeoff_multicorrelator_resampler(np.zeros(10, np.complex64), 0, 0, 0, 0, 0.1, 0)
    mc.set_local_code_and_taps(np.ones(1023, np.float32), [-0.5, 0, 0.5])
    with pytest.raises(capi.B200Error):               # longer than init() allowed
        mc.Carrier_wipeoff_multicorrelator_resampler(np.zeros(2000, np.complex64), 0, 0, 0, 0, 0.1, 0)
    out = mc.Carrier_wipeoff_multicorrelator_resampler(np.zeros(0, np.complex64), 0, 0, 0, 0, 0.1, 0, 0)
    assert np.all(out == 0)
    mc.free()


# ---- high-dynamics variants (a4) ----------------------------------------------------------------------
@pytest.mark.parametrize("n,L,shifts,step,rate", [
    (25000, 1023, [-0.5, 0.0, 0.5], 0.04092, 3e-12),
    (25003, 1023, [-0.5, 0.0, 0.5], 0.04092, -3e-12),
    (8111, 2046, [-0.1, 0.0, 0.1], (2046 + 0.1) / 8111, 1e-9),
    (4000, 1023, [-0.5, 0.0, 0.5], 0.25575, 2e-10),
    (200000, 8184, [-1.2, -0.3, 0.0, 0.3, 1.2], 0.04092, 1e-13),
])
def test_high_dynamics_resampler_integer_exact(capi, engine, oracle, n, L, shifts, step, rate):
    """high_dyn=true: quadratic code phase on tap 0 with the a_avx association, other taps are
    circular sample shifts of tap 0 (VG ..._high_dynamics_resampler_32f_xn.h:433-513).  Integer data
    and zero carrier make the expected taps exact integers."""
    rng = np.random.default_rng(n)
    x_int = rng.integers(-7, 8, n)
    x_int[x_int == 0] = 1
    code_int = ((np.arange(L) * 7919) % 31) - 15
    code_int[code_int == 0] = 16
    rem = 0.37
    resampled = oracle.port.hd_resampler_avx(code_int.astype(np.float32), rem, step, rate, shifts, n)
    want = (resampled.astype(np.int64) * x_int[None, :]).sum(axis=1)
    mc = capi.Multicorrelator(engine, n, len(shifts))
    mc.set_high_dynamics_resampler(True)
    mc.set_local_code_and_taps(code_int.astype(np.float32), shifts)
    got = mc.Carrier_wipeoff_multicorrelator_resampler(x_int.astype(np.complex64), 0.0, 0.0, 0.0, rem, step, rate)
    mc.free()
    assert np.array_equal(got.real.astype(np.int64), want)
    assert np.all(got.imag == 0)


def test_high_dynamics_rotator_parity(capi, engine, oracle):
    """high_dyn=true with a carrier phase rate: against the reference class
    (HD resampler + volk_gnsssdr_32fc_32f_high_dynamic_rotator_dot_prod_32fc_xn_generic, whose
    cpowf-based phase is itself only float-accurate) within 1e-3, and against a float64 evaluation of
    the same phase law (rate term lagging one sample, ..._high_dynamic_rotator...h:92-103) within 2e-5."""
    n, L = 25000, 1023
    rng = np.random.default_rng(77)
    code = oracle.port.gps_ca_code(9)
    shifts = np.array([-0.5, 0.0, 0.5], np.float32)
    step, crate = np.float32(0.04092), np.float32(2e-12)
    rem_code, rem_carr, dphi, drate = np.float32(0.3), np.float32(0.7), np.float32(1.1e-3), np.float32(2e-9)
    k = np.arange(n)
    resampled = oracle.port.hd_resampler_avx(code, float(rem_code), float(step), float(crate), shifts, n)
    e = np.where(k >= 1, (k - 1.0) ** 2, 0.0)
    ph = -(float(rem_carr) + k * float(dphi) + e * float(drate))
    iq = (0.05 * resampled[1] * np.exp(-1j * ph) + rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    truth = (resampled.astype(np.float64) * (iq.astype(np.complex128) * np.exp(1j * ph))[None, :]).sum(axis=1)
    mc = capi.Multicorrelator(engine, n, 3)
    mc.set_high_dynamics_resampler(True)
    mc.set_local_code_and_taps(code, shifts)
    got = mc.Carrier_wipeoff_multicorrelator_resampler(iq, float(rem_carr), float(dphi), float(drate), float(rem_code),
                                                       float(step), float(crate))
    mc.free()
    assert np.abs(truth[1]) > 5 * np.sqrt(n)
    assert np.max(np.abs(got - truth)) / np.abs(truth[1]) < 2e-5
    if oracle.ref is not None:
        oracle.ref.select_arch("a_avx")
        h = oracle.ref.mc_create(n, 3, high_dyn=True)
        oracle.ref.mc_set_code(h, code, shifts)
        want = oracle.ref.mc_correlate(h, iq, 3, float(rem_carr), float(dphi), float(drate), float(rem_code), float(step), float(crate))
        oracle.ref.mc_destroy(h)
        assert np.all(np.abs(got - want) / np.abs(want) < 1e-3)


def test_submit_wait_overlapped_batches(capi, engine, oracle):
    """b200_trk_submit / b200_trk_wait: several batches in flight, waited out of order, equal the
    synchronous b200_trk_batch results bit for bit."""
    n, L = 4000, 1023
    rng = np.random.default_rng(21)
    iq = (rng.standard_normal(n * 6 + 8) + 1j * rng.standard_normal(n * 6 + 8)).astype(np.complex64)
    e = engine
    band = 5
    e.iq_create(band, len(iq))
    first = e.iq_push(band, iq)
    cid = e.channel_create(band, 3)
    e.channel_set_code(cid, oracle.port.gps_ca_code(4), [-0.5, 0.0, 0.5])
    items = np.zeros(6, capi.TRK_ITEM_DTYPE)
    items["channel"] = cid
    items["n"] = n
    items["sample_index"] = first + np.arange(6) * n + 1
    items["rem_carrier_phase_rad"] = 0.2
    items["phase_step_rad"] = 2e-3
    items["rem_code_phase_chips"] = 0.1
    items["code_phase_step_chips"] = 0.25575
    want = e.trk_batch(items, 3)
    t = [e.trk_submit(items[k:k + 2], 3) for k in (0, 2, 4)]
    got = {k: e.trk_wait(t[k]) for k in (2, 0, 1)}
    assert np.array_equal(np.concatenate([got[0], got[1], got[2]]), want)
    with pytest.raises(capi.B200Error):
        e.trk_wait(t[0])      # ticket already consumed


@pytest.mark.parametrize("dtype", [np.int16, np.int8])
def test_integer_sample_ingestion_bitexact(capi, engine, oracle, dtype):
    """b200_iq_push_i16 / _i8: raw integer I/Q over PCIe, converted on the device
    (volk_gnsssdr_16ic_convert_32fc semantics: plain int -> float), must give exactly the taps
    of pushing the same samples as complex64, including across the ring wrap."""
    n, L = 4000, 1023
    rng = np.random.default_rng(31)
    hi = 2000 if dtype == np.int16 else 100
    raw = rng.integers(-hi, hi + 1, 2 * (n * 5 + 11)).astype(dtype)
    as_c64 = (raw[0::2].astype(np.float32) + 1j * raw[1::2].astype(np.float32)).astype(np.complex64)
    e = engine
    res = {}
    for name, band in (("float", 6), ("int", 7)):
        e.iq_create(band, 32768)
        # misalign the write position so that the data wraps around the ring end
        e.iq_push(band, np.zeros(20001, np.complex64))
        first = e.iq_push(band, as_c64) if name == "float" else e.iq_push_int(band, raw)
        assert first == 20001
        cid = e.channel_create(band, 3)
        e.channel_set_code(cid, oracle.port.gps_ca_code(6), [-0.5, 0.0, 0.5])
        items = np.zeros(5, capi.TRK_ITEM_DTYPE)
        items["channel"] = cid
        items["n"] = n
        items["sample_index"] = first + np.arange(5) * n + 3
        items["rem_carrier_phase_rad"] = 0.2
        items["phase_step_rad"] = 2e-3
        items["rem_code_phase_chips"] = 0.1
        items["code_phase_step_chips"] = 0.25575
        res[name] = e.trk_batch(items, 3)
    assert np.array_equal(res["float"], res["int"])
    assert np.all(np.abs(res["int"]) > 0)


@pytest.mark.parametrize("L,taps_shifts,step,n", [
    (1023, [-0.5, 0.0, 0.5], 0.04092, 25000),
    (8184, [-1.2, -0.3, 0.0, 0.3, 1.2], 0.08184, 20000),      # Galileo E1 sinBOC table, 5 taps
    (10230, [-0.5, 0.0, 0.5], 0.2046, 12000),                   # L5-sized table
    (1023, [0.0], 0.2557, 4001),                                # 1 tap, ragged length
])
def test_shared_window_groups_staggered_integer_exact(capi, oracle, L, taps_shifts, step, n):
    """The shared-window kernel (groups of 8 items served from one TMA-staged copy of the samples):
    epochs of different channels start at different, odd/even sample offsets (as in a real receiver,
    where every channel is aligned to its own code period), item count not a multiple of 8, different
    code tables and code phases per channel.  Integer data => results must be EXACT.  Run with the
    shared kernel forced on and forced off: both must equal the integer oracle."""
    import os
    rng = np.random.default_rng(L + n)
    n_ch, n_ep = 11, 3
    total = n * (n_ep + 1) + 4096
    x_int = rng.integers(-7, 8, total)
    starts = np.sort(rng.integers(0, n, n_ch))                  # per-channel epoch alignment
    codes = [(((np.arange(L) * (7919 + 2 * c)) % 31) - 15) for c in range(n_ch)]
    rems = rng.uniform(-3, 3, n_ch).astype(np.float32)
    want = {}
    for c in range(n_ch):
        _, idx = oracle.port.resampler(1, codes[c].astype(np.float32), float(rems[c]), step, taps_shifts, n, return_idx=True)
        for k in range(n_ep):
            s0 = int(starts[c]) + k * n
            want[(k, c)] = int_oracle(x_int[s0:s0 + n], codes[c], idx)
    results = {}
    for mode in ("1", "0"):
        os.environ["B200_TRK_SHARED"] = mode
        e = capi.Engine(0)
        e.iq_create(0, total)
        first = e.iq_push(0, x_int.astype(np.complex64))
        cids = []
        for c in range(n_ch):
            cid = e.channel_create(0, len(taps_shifts))
            e.channel_set_code(cid, codes[c].astype(np.float32), taps_shifts)
            cids.append(cid)
        items = np.zeros(n_ch * n_ep, capi.TRK_ITEM_DTYPE)
        order = []
        for k in range(n_ep):
            for c in range(n_ch):
                it = items[len(order)]
                it["channel"] = cids[c]
                it["n"] = n
                it["sample_index"] = first + int(starts[c]) + k * n
                it["rem_code_phase_chips"] = rems[c]
                it["code_phase_step_chips"] = step
                order.append((k, c))
        # device-pointer entry point with slices = 1 is where the engine picks the shared kernel
        import torch
        items_t = torch.from_numpy(items.view(np.uint8)).cuda()
        out_t = torch.zeros(len(order), len(taps_shifts), 2, dtype=torch.float32, device="cuda")
        e.trk_batch_dev(items_t.data_ptr(), len(order), out_t.data_ptr(), len(taps_shifts), 1)
        e.sync()
        got = out_t.cpu().numpy()
        results[mode] = got
        for i, key in enumerate(order):
            assert np.array_equal(got[i, :, 0].astype(np.int64), want[key]), (mode, key)
            assert np.all(got[i, :, 1] == 0)
        e.close()
    os.environ.pop("B200_TRK_SHARED", None)
    assert np.array_equal(results["0"], results["1"])


def test_shared_kernel_groups_that_cannot_share(capi, oracle):
    """Groups of 8 items whose sample ranges are far apart (channel-major order: 8 consecutive epochs of one
    channel) or that sit on different bands cannot share a window; each warp then streams its own samples
    with the same arithmetic.  Integer-exact."""
    import os
    import torch
    n, L, shifts, step = 6000, 1023, [-0.5, 0.0, 0.5], 0.1705
    rng = np.random.default_rng(4242)
    n_ch, n_ep = 4, 9
    total = n * n_ep + 1001
    xs = [rng.integers(-7, 8, total) for _ in range(2)]           # two bands
    codes = [(((np.arange(L) * (7919 + 2 * c)) % 31) - 15) for c in range(n_ch)]
    os.environ["B200_TRK_SHARED"] = "1"
    e = capi.Engine(0)
    firsts = []
    for b in range(2):
        e.iq_create(b, total)
        firsts.append(e.iq_push(b, xs[b].astype(np.complex64)))
    cids = []
    for c in range(n_ch):
        cid = e.channel_create(c % 2, 3)                          # channels alternate between the bands
        e.channel_set_code(cid, codes[c].astype(np.float32), shifts)
        cids.append(cid)
    items = np.zeros(n_ch * n_ep, capi.TRK_ITEM_DTYPE)
    order = []
    for c in range(n_ch):                                         # channel-major: consecutive epochs of one channel
        for k in range(n_ep):
            it = items[len(order)]
            it["channel"] = cids[c]
            it["n"] = n
            it["sample_index"] = firsts[c % 2] + 37 * c + k * n + (k % 2)
            it["rem_code_phase_chips"] = 0.3 + c
            it["code_phase_step_chips"] = step
            order.append((c, k))
    items_t = torch.from_numpy(items.view(np.uint8)).cuda()
    out_t = torch.zeros(len(order), 3, 2, dtype=torch.float32, device="cuda")
    e.trk_batch_dev(items_t.data_ptr(), len(order), out_t.data_ptr(), 3, 1)
    e.sync()
    got = out_t.cpu().numpy()
    e.close()
    os.environ.pop("B200_TRK_SHARED", None)
    for i, (c, k) in enumerate(order):
        _, idx = oracle.port.resampler(1, codes[c].astype(np.float32), 0.3 + c, step, shifts, n, return_idx=True)
        s0 = 37 * c + k * n + (k % 2)
        want = int_oracle(xs[c % 2][s0:s0 + n], codes[c], idx)
        assert np.array_equal(got[i, :, 0].astype(np.int64), want), (c, k)
        assert np.all(got[i, :, 1] == 0)


@pytest.mark.parametrize("layout", ["shared", "distinct"])
def test_kernel_choice_by_layout_is_integer_exact(capi, oracle, layout):
    """1536 host-submitted items: with overlapping neighbours (a receiver: all channels on one stream) b200_trk_submit takes
    the shared-window kernel, with disjoint sample ranges (every item its own samples) the per-item kernel; forcing either
    kernel (b200_trk_kernel_choice) gives the same integers."""
    n, L, shifts, step = 2000, 1023, [-0.5, 0.0, 0.5], 0.5115
    rng = np.random.default_rng(77)
    n_ch, n_ep = 48, 32
    span = n * n_ep + 64
    total = span * (n_ch if layout == "distinct" else 1)
    x = rng.integers(-9, 10, total)
    codes = [np.where(rng.integers(0, 2, L) > 0, 1, -1) for _ in range(n_ch)]
    e = capi.Engine(0)
    e.iq_create(0, total)
    first = e.iq_push(0, x.astype(np.complex64))
    items = np.zeros(n_ch * n_ep, capi.TRK_ITEM_DTYPE)
    where = []
    for k in range(n_ep):
        for c in range(n_ch):
            if k == 0:
                cid = e.channel_create(0, 3)
                e.channel_set_code(cid, codes[c].astype(np.float32), shifts)
            it = items[len(where)]
            it["channel"] = c
            it["n"] = n
            s0 = k * n + (c % 5) + (c * span if layout == "distinct" else 0)
            it["sample_index"] = first + s0
            it["rem_code_phase_chips"] = 0.25 + c
            it["code_phase_step_chips"] = step
            where.append((c, s0))
    results = {}
    for mode in (2, 0, 1):
        e.trk_kernel_choice(mode)
        results[mode] = e.trk_batch(items, 3)
    e.close()
    assert np.array_equal(results[2], results[0]) and np.array_equal(results[2], results[1])
    got = results[2]
    for i in range(0, len(where), 7):
        c, s0 = where[i]
        _, idx = oracle.port.resampler(1, codes[c].astype(np.float32), 0.25 + c, step, shifts, n, return_idx=True)
        want = int_oracle(x[s0:s0 + n], codes[c], idx)
        assert np.array_equal(got[i].real.astype(np.int64), want), (c, s0)
        assert np.all(got[i].imag == 0)


@pytest.mark.gpu
@pytest.mark.parametrize("item_type", ["gr_complex", "ishort", "ibyte"])
def test_file_source_push_matches_array_push(oracle, tmp_path, item_type):
    """b200_iq_push_file (File_Signal_Source semantics: header, skipped samples, interleaved I/Q item types, blocks
    through pinned double buffers) fills the band with exactly what the array pushes do: taps bit-identical."""
    from gnss_sdr_b200 import capi
    import gnss_synth as gs
    fs, n, prn = 4e6, 4000, 6
    code = gs.gps_ca_code(prn)
    sv = dict(prn=prn, doppler=1250.0, code_phase_chips=77.0, cn0=50.0)
    total = 9 * n + 123
    iq = gs.make_iq({prn: code}, fs, total, [sv], seed=12)
    header, skip = 16, 100
    path = str(tmp_path / "capture.dat")
    if item_type == "gr_complex":
        payload = iq
        arr_push = lambda e, b, a: e.iq_push(b, a)
    else:
        bits = 16 if item_type == "ishort" else 8
        scale = 256.0 if bits == 16 else 16.0
        q = np.clip(np.round(iq.view(np.float32) * scale), -(2 ** (bits - 1) - 1), 2 ** (bits - 1) - 1).astype(np.int16 if bits == 16 else np.int8)
        payload = q
        arr_push = lambda e, b, a: e.iq_push_int(b, a)
    with open(path, "wb") as f:
        f.write(bytes([0x7F]) * header)
        f.write(payload.tobytes())
    per = 1 if item_type == "gr_complex" else 2          # array elements per complex sample
    e = capi.Engine()
    for b in (0, 1):
        e.iq_create(b, 1 << 16)
    first_a = arr_push(e, 0, payload[skip * per:])
    first_b, pushed = e.iq_push_file(1, path, item_type, header_bytes=header, skip_samples=skip, chunk_samples=4096)
    assert pushed == total - skip and first_a == first_b == 0
    first_c, pushed_c = e.iq_push_file(1, path, item_type, header_bytes=header, skip_samples=0, max_samples=5000, chunk_samples=1024)
    assert pushed_c == 5000 and first_c == total - skip
    items = np.zeros(8, capi.TRK_ITEM_DTYPE)
    _, rc, dp, rcode, st = gs.trk_params_for(sv, fs, n, 8)
    out = []
    for b in (0, 1):
        ch = e.channel_create(b, 3)
        e.channel_set_code(ch, code, [-0.5, 0.0, 0.5])
        items["channel"], items["n"] = ch, n
        items["sample_index"] = np.arange(8) * n
        items["rem_carrier_phase_rad"], items["phase_step_rad"] = rc, dp
        items["rem_code_phase_chips"], items["code_phase_step_chips"] = rcode, st
        out.append(e.trk_batch(items, 3))
    assert out[0].tobytes() == out[1].tobytes()
    assert np.abs(out[0][:, 1]).min() > 0
    with pytest.raises(capi.B200Error):
        e.iq_push_file(1, path, "float")
    with pytest.raises(capi.B200Error):
        e.iq_push_file(1, str(tmp_path / "missing.dat"))
    e.close()


def test_push_at_is_idempotent_and_handles_gaps(capi, oracle):
    """b200_iq_push_at: every tracking block of a flowgraph offers the same samples by absolute index - overlapping
    offers copy only what is new, a later start opens a gap, and items outside [valid_from, write_index) are refused."""
    eng = capi.Engine(0)
    rng = np.random.default_rng(5)
    n = 30000
    iq = (rng.integers(-50, 50, n) + 1j * rng.integers(-50, 50, n)).astype(np.complex64)
    eng.iq_create(2, 1 << 16)
    base = 1_000_000  # the first block to track starts long after sample 0
    assert eng.iq_push_at(2, base, iq[:10000]) == 10000
    assert eng.iq_window(2) == (base, base + 10000)
    assert eng.iq_push_at(2, base, iq[:10000]) == 0              # a second block offers the same samples
    assert eng.iq_push_at(2, base + 4000, iq[4000:16000]) == 6000  # overlap: only the tail is copied
    assert eng.iq_push_at(2, base + 2000, iq[2000:9000]) == 0
    assert eng.iq_window(2) == (base, base + 16000)
    code = np.where(rng.integers(0, 2, 1023) > 0, 1.0, -1.0).astype(np.float32)
    shifts = [-0.5, 0.0, 0.5]
    ch = eng.channel_create(2, 3)
    eng.channel_set_code(ch, code, shifts)
    items = np.zeros(1, capi.TRK_ITEM_DTYPE)
    items[0] = (ch, 4000, base + 8000, 0.2, 0.01, 0.0, 0.3, 0.2557, 0.0)
    got = eng.trk_batch(items, 3)[0]
    want = oracle.port.multicorrelator(1, iq[8000:12000], code, shifts, 0.2, 0.01, 0.3, 0.2557)
    assert np.max(np.abs(got - want)) <= 1e-3 * np.abs(want[1])
    items[0]["sample_index"] = base + 14000  # runs past the write index
    with pytest.raises(capi.B200Error):
        eng.trk_batch(items, 3)
    items[0]["sample_index"] = base - 100    # before the gap
    with pytest.raises(capi.B200Error):
        eng.trk_batch(items, 3)
    eng.close()


def test_channel_set_taps_takes_effect_in_stream_order(capi, oracle):
    """b200_trk_channel_set_taps: the batch submitted before the change keeps the old spacing, the next one has the new
    one (the narrow-correlator switch of the tracking block, dll_pll_veml_tracking.cc:2132-2146)."""
    eng = capi.Engine(0)
    rng = np.random.default_rng(6)
    n = 4000
    iq = (rng.standard_normal(8 * n) + 1j * rng.standard_normal(8 * n)).astype(np.complex64)
    code = np.where(rng.integers(0, 2, 1023) > 0, 1.0, -1.0).astype(np.float32)
    eng.iq_create(0, 1 << 16)
    eng.iq_push(0, iq)
    ch = eng.channel_create(0, 3)
    wide, narrow = [-0.5, 0.0, 0.5], [-0.15, 0.0, 0.15]
    eng.channel_set_code(ch, code, wide)
    items = np.zeros(2, capi.TRK_ITEM_DTYPE)
    for k in range(2):
        items[k] = (ch, n, k * n, 0.1, 0.02, 0.0, 0.4, 0.2557, 0.0)
    a = eng.trk_batch(items, 3)
    eng.channel_set_taps(ch, narrow)
    b = eng.trk_batch(items, 3)
    eng.channel_set_taps(ch, wide)
    c = eng.trk_batch(items, 3)
    for k in range(2):
        ww = oracle.port.multicorrelator(1, iq[k * n:(k + 1) * n], code, wide, 0.1, 0.02, 0.4, 0.2557)
        wn = oracle.port.multicorrelator(1, iq[k * n:(k + 1) * n], code, narrow, 0.1, 0.02, 0.4, 0.2557)
        assert np.max(np.abs(a[k] - ww)) <= 1e-3 * np.abs(ww[1])
        assert np.max(np.abs(b[k] - wn)) <= 1e-3 * np.abs(wn[1])
        assert np.array_equal(a[k], c[k])
    eng.close()


def cplx_case():
    """Inputs of the complex-code correlator test: sig, code, shifts, rem_code, step and the (rem_carr, dphi) pairs."""
    rng = np.random.default_rng(41)
    n, L = 8111, 2046
    sig = (rng.integers(-30, 30, n) + 1j * rng.integers(-30, 30, n)).astype(np.complex64)
    code = (rng.integers(-2, 3, L) + 1j * rng.integers(-2, 3, L)).astype(np.complex64)
    return sig, code, [-0.6, -0.1, 0.0, 0.1, 0.6], 0.234, (L + 0.3) / n, [(0.0, 0.0), (0.4, 0.0123)]


def sc16_case():
    """Inputs of the 16-bit correlator test: sig, code (interleaved I,Q), shifts, rem_code, step, (rem_carr, dphi) pairs."""
    rng = np.random.default_rng(43)
    n, L = 8111, 1023
    sig = rng.integers(-4, 5, 2 * n).astype(np.int16)
    code = np.zeros(2 * L, np.int16)
    code[0::2] = rng.choice([-1, 1], L)
    return sig, code, [-0.5, 0.0, 0.5], 0.1, (L + 0.2) / n, [(0.0, 0.0), (0.3, 0.0021)]


@pytest.fixture(scope="module")
def blocks_gold():
    """The reference classes' outputs on cplx_case / sc16_case (tests/golden/make_golden.py, fixture `blocks`)."""
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "blocks_ref_golden.npz"))


def test_complex_code_correlator_matches_reference_class(capi, blocks_gold):
    """Cpu_Multicorrelator (complex local code, cpu_multicorrelator.cc:86-100) against b200_trk_correlate_cplx: integer-valued
    samples and code with a zero carrier are exact; a rotating carrier agrees to the reference's own SIMD tolerance."""
    sig, code, shifts, rem_code, step, carriers = cplx_case()
    want = blocks_gold["trk_cplx/want"]
    eng = capi.Engine(0)
    mc = capi.Multicorrelator(eng, len(sig), len(shifts))
    mc.set_local_code_and_taps_cplx(code, shifts)
    got = mc.correlate_cplx(sig, *carriers[0], rem_code, step)
    assert np.array_equal(got, want[0])
    got = mc.correlate_cplx(sig, *carriers[1], rem_code, step)
    assert np.max(np.abs(got - want[1])) <= 1e-3 * np.max(np.abs(want[1]))
    mc.free()
    eng.close()


def test_16bit_correlator_matches_reference_class(capi, blocks_gold):
    """Cpu_Multicorrelator_16sc (cpu_multicorrelator_16sc.cc:64-91) against b200_trk_correlate_16sc on the shape of the
    reference's kernel QA (vlen 8111, small amplitudes so that the 16-bit accumulator never saturates): zero carrier exact;
    rotating carrier within +-16 LSB, the reference's own tolerance between implementations of this kernel."""
    sig, code, shifts, rem_code, step, carriers = sc16_case()
    want = blocks_gold["trk_16sc/want"]
    eng = capi.Engine(0)
    mc = capi.Multicorrelator(eng, len(sig) // 2, len(shifts))
    mc.set_local_code_and_taps_16sc(code, shifts)
    got = mc.correlate_16sc(sig, *carriers[0], rem_code, step)
    assert np.array_equal(got, want[0])
    got = mc.correlate_16sc(sig, *carriers[1], rem_code, step)
    assert np.max(np.abs(got.astype(int) - want[1].astype(int))) <= 16
    mc.free()
    eng.close()


def test_push_at_restarts_when_the_stream_starts_over(capi, oracle):
    """A stream that begins again at an OLDER absolute index than anything the ring still holds (a new capture, the next
    test in the same process): b200_iq_push_at must not answer "already there" - the band restarts at the offered index."""
    eng = capi.Engine(0)
    rng = np.random.default_rng(8)
    iq = (rng.integers(-50, 50, 40000) + 1j * rng.integers(-50, 50, 40000)).astype(np.complex64)
    eng.iq_create(1, 1 << 14)                       # 16384-sample ring
    assert eng.iq_push_at(1, 5_000_000, iq[:12000]) == 12000
    assert eng.iq_push_at(1, 5_012_000, iq[12000:22000]) == 10000
    assert eng.iq_push_at(1, 5_022_000, iq[22000:30000]) == 8000       # wrapped: the ring now holds [5 013 616, 5 030 000)
    assert eng.iq_window(1) == (5_030_000 - 16384, 5_030_000)
    assert eng.iq_push_at(1, 0, iq[:8000]) == 8000                     # the stream starts over
    assert eng.iq_window(1) == (0, 8000)
    assert eng.iq_push_at(1, 4000, iq[4000:10000]) == 2000
    # a new stream whose indices overlap the old one's cannot be told apart by index: the host says so (b200_iq_forget)
    assert eng.iq_push_at(1, 2000, iq[20000:24000]) == 0               # "already there" - the old samples
    eng.iq_forget(1)
    assert eng.iq_window(1) == (10000, 10000)
    assert eng.iq_push_at(1, 2000, iq[20000:24000]) == 4000
    assert eng.iq_window(1) == (2000, 6000)
    assert eng.iq_push_at(1, 0, iq[:10000]) == 10000                   # and back (older index: restart)
    code = np.where(rng.integers(0, 2, 1023) > 0, 1.0, -1.0).astype(np.float32)
    ch = eng.channel_create(1, 3)
    eng.channel_set_code(ch, code, [-0.5, 0.0, 0.5])
    items = np.zeros(1, capi.TRK_ITEM_DTYPE)
    items[0] = (ch, 4000, 5000, 0.0, 0.0, 0.0, 0.3, 0.2557, 0.0)
    got = eng.trk_batch(items, 3)[0]
    want = oracle.port.multicorrelator(1, iq[5000:9000], code, [-0.5, 0.0, 0.5], 0.0, 0.0, 0.3, 0.2557)
    assert np.array_equal(got, want)
    eng.close()
