"""The DLL/PLL loop oracle (oracle/port_loop.c) pinned against the reference's OWN library code
(oracle/_ref/liboracle_ref_loop.so = tracking_discriminators.cc, tracking_FLL_PLL_filter.cc,
tracking_loop_filter.cc, lock_detectors.cc, exponential_smoother.cc compiled where they lie), and the
closed loop over the reference's CPU correlator.  CPU only.

What the reference returned for these inputs is stored in tests/golden/loop_ref_pins.npz (written by
tests/golden/make_golden.py through the helpers below, on the live reference libraries)."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

from oracle import loop as ol
import gnss_synth as gs
import loop_harness as lh

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "loop_ref_pins.npz")
TRACE_BLOCK = 100   # epochs per stored digest of the cycle trace


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLDEN)


def library_outputs(lib, prefix):
    """Discriminators and lock detectors of `lib` (port_* or ref_* symbols) on seeded inputs -> dict of arrays."""
    fn = lambda name: getattr(lib, prefix + name)
    rng = np.random.default_rng(11)
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
    out = {k: [] for k in ("pll", "fll", "dll", "vemlp", "cn0", "lock")}
    for _ in range(4000):
        v = (rng.standard_normal(8) * 10 ** rng.uniform(-2, 4)).astype(np.float32)
        if rng.random() < 0.05:
            v[rng.integers(0, 8)] = 0.0
        out["pll"].append(fn("disc_pll_cloop")(v[0], v[1]))
        out["fll"].append(fn("disc_fll_diff_atan")(v[0], v[1], v[2], v[3], 0.0, 0.001))
        out["dll"].append(fn("disc_dll_e_minus_l")(v[0], v[1], v[2], v[3], 0.5, 1.0, 1.0))
        out["vemlp"].append(fn("disc_dll_vemlp")(fp(v)))
    for _ in range(300):
        n = int(rng.integers(1, 40))
        buf = (rng.standard_normal(2 * n) * 300 + (2000 if rng.random() < 0.7 else 0)).astype(np.float32)
        out["cn0"].append(fn("cn0_m2m4")(fp(buf), n, 0.001))
        out["lock"].append(fn("carrier_lock_detector")(fp(buf), n))
    return {k: np.array(v, np.float64) for k, v in out.items()}


def test_library_functions_bit_exact(gold):
    got = library_outputs(ol.port_lib(), "port_")
    for k in ("pll", "dll", "vemlp", "lock"):
        assert np.all(got[k] == gold[f"lib/{k}"]), k
    for k in ("fll", "cn0"):
        a, b = got[k], gold[f"lib/{k}"]
        assert np.all((a == b) | (np.isnan(a) & np.isnan(b))), k


CONFS = [
    dict(),
    dict(pll_filter_order=2, dll_filter_order=1),
    dict(pll_filter_order=3, dll_filter_order=3, enable_fll_pull_in=1, pull_in_time_s=1),
    dict(enable_fll_steady_state=1, carrier_aiding=0),
    dict(veml=1, code_samples_per_chip=2, early_late_space_chips=0.15, cn0_samples=10),
    dict(pull_in_time_s=0, max_code_lock_fail=5, cn0_min=40),     # loses lock on the weak stretch
    dict(bit_synchronization_time_limit_s=1, pull_in_time_s=0),     # fail-safe fires after 1 s
]
STATUS_INT = ("state", "loss_of_lock", "sample_counter", "epochs")


def cycle_trace(make_loop, kw, n_epochs=3000):
    """Run one loop over seeded taps: every item scalar and every logged dump-record byte, epoch by epoch, hashed per
    TRACE_BLOCK epochs -> (uint8[blocks, 32] digests, lost, final status as (int64[4], float64[6]))."""
    conf = ol.default_conf(fs_in=4e6, **kw)
    L = make_loop(conf)
    L.start(524.3, 1680.0, 1000, 9000)
    taps_seq = lh.synthetic_taps(n_epochs, 5 if conf.veml else 3, seed=5, weak_from=1500 if conf.cn0_min == 40 else None)
    digests, h, lost = [], hashlib.sha256(), False
    for k in range(n_epochs):
        item = L.prepare()
        if item is None:
            h.update(b"standby")
            lost = True
            break
        h.update(np.uint64(item[0]).tobytes() + np.int32(item[1]).tobytes() + item[2].tobytes())
        logged, rec = L.update(taps_seq[k])
        h.update(b"L" + rec.tobytes() if logged else b"-")
        if (k + 1) % TRACE_BLOCK == 0:
            digests.append(h.digest())
            h = hashlib.sha256()
    digests.append(h.digest())
    s = L.status()
    ints = np.array([getattr(s, f) for f in STATUS_INT], np.int64)
    dbls = np.array([getattr(s, f) for f, _ in ol.LoopStatus._fields_ if f not in STATUS_INT], np.float64)
    return np.frombuffer(b"".join(digests), np.uint8).reshape(-1, 32), lost, (ints, dbls)


@pytest.mark.parametrize("kw", CONFS)
def test_cycle_port_vs_reference_classes_bit_exact(gold, kw):
    """Same taps in, every item scalar and every dump-record byte equal, epoch by epoch."""
    i = CONFS.index(kw)
    got, lost, (ints, dbls) = cycle_trace(ol.PortLoop, kw)
    want = gold[f"cycle{i}/trace"]
    assert got.shape == want.shape, (got.shape, want.shape)
    bad = [b for b in range(len(got)) if not np.array_equal(got[b], want[b])]
    assert not bad, f"first differing epochs: {bad[0] * TRACE_BLOCK} .. {(bad[0] + 1) * TRACE_BLOCK - 1}"
    assert lost == bool(gold[f"cycle{i}/lost"])
    assert np.array_equal(ints, gold[f"cycle{i}/status_int"]) and np.all(dbls == gold[f"cycle{i}/status_dbl"])
    conf = ol.default_conf(fs_in=4e6, **kw)
    if conf.cn0_min == 40 or conf.bit_synchronization_time_limit_s == 1:
        assert lost and ints[0] == 0 and ints[1] == 1
    else:
        assert not lost and ints[0] == 2 and ints[3] == 3000


def closed_loop_records(oracle, correlator):
    """Oracle loop + a CPU correlator (`correlator(code, shifts, max_len)`) over a synthetic 4 Msps signal, 1500 epochs."""
    fs, prn, doppler, cn0 = 4e6, 7, 1234.0, 47.0
    code = oracle.port.gps_ca_code(prn)
    delay = 1337
    n = int(fs * 1.6)
    iq = gs.make_iq({prn: code}, fs, n, [dict(prn=prn, doppler=doppler, code_phase_chips=(-delay * 1.023e6 / fs) % 1023, cn0=cn0)], seed=21)
    conf = ol.default_conf(fs_in=fs, prn=prn, pull_in_time_s=1)
    L = ol.PortLoop(conf)
    L.start(float(delay % 4000) + 0.4, doppler - 60.0, 0, 0)
    recs = lh.run_closed_loop(L, correlator(code, [-0.5, 0.0, 0.5], int(conf.vector_length)), iq, 1500)
    return recs, L.status(), (doppler, cn0)


def test_closed_loop_over_reference_correlator_locks(oracle, gold):
    """Oracle loop + the reference's Cpu_Multicorrelator_Real_Codes on a synthetic 4 Msps signal: pulls in from a
    coarse acquisition and reports the true Doppler, code rate and C/N0 (pins the sign conventions of the cycle).
    Run here over the C port of that correlator; the records must be, byte for byte, the ones the loop produced over
    the reference's own class."""
    recs, s, (doppler, cn0) = closed_loop_records(oracle, lambda code, shifts, _: lh.PortCorrelator(oracle.port, code, shifts))
    assert hashlib.sha256(recs.tobytes()).digest() == gold["closed_loop/records_sha"].tobytes()
    assert len(recs) == 1500
    tail = recs[-300:]
    assert abs(np.mean(tail["carrier_doppler_hz"]) - doppler) < 2.0
    assert abs(np.mean(tail["code_freq_chips"].astype(np.float64)) - 1.023e6 * (1 + doppler / 1575.42e6)) < 0.2  # float32 record: 0.0625 chips/s steps
    assert abs(np.mean(tail["CN0_SNV_dB_Hz"]) - cn0) < 1.5
    # alpha = 0.002 smoother: still climbing from its pull-in average after 1.5 s
    assert np.all(tail["carrier_lock_test"] > 0.5) and tail["carrier_lock_test"][-1] > tail["carrier_lock_test"][0]
    assert np.mean(tail["abs_P"]) > 1.8 * np.mean(tail["abs_E"]) * 0.9
    # PRN start stamps advance by ~4000 samples and follow the true code phase
    d = np.diff(recs["PRN_start_sample_count"].astype(np.int64))
    assert set(np.unique(d)) <= {3999, 4000, 4001}
    assert s.state == 2 and s.epochs == 1500


def dump_records():
    conf = ol.default_conf()
    L = ol.PortLoop(conf)
    L.start(100.0, 500.0, 0, 0)
    taps = lh.synthetic_taps(50, 3, seed=3)
    recs = []
    for k in range(50):
        L.prepare()
        ok, r = L.update(taps[k])
        recs.append(r)
    return np.array(recs, ol.DUMP_RECORD_DTYPE)


def write_dump(path, recs):
    from gnss_sdr_b200 import capi
    assert capi.TRK_DUMP_RECORD_DTYPE == ol.DUMP_RECORD_DTYPE
    capi.trk_dump_write(path, recs[:20])
    capi.trk_dump_write(path, recs[20:], append=True)


def test_dump_file_is_readable_by_the_reference_reader(gold, tmp_path):
    """b200_trk_dump_write (host-only entry point of the product library) -> the reference's own
    Tracking_Dump_Reader (tests/unit-tests/signal-processing-blocks/libs/tracking_dump_reader.cc:22-50).
    The file must be byte for byte the one the reader was given, and what the reader made of it the records."""
    recs = dump_records()
    fn = str(tmp_path / "trk_dump_ch0.dat")
    write_dump(fn, recs)
    with open(fn, "rb") as f:
        assert hashlib.sha256(f.read()).digest() == gold["dump/file_sha"].tobytes()
    got = gold["dump/read"]
    assert got.shape == (50, 24)
    for j, name in enumerate(ol.DUMP_RECORD_DTYPE.names):
        assert np.array_equal(got[:, j], recs[name].astype(np.float64)), name
