"""Pins for the acquisition oracle (oracle/port_acq.c, oracle/acq_np.py).

* sincos / index_max C ports are checked BIT-EXACT against the reference's own kernels (their outputs stored in
  tests/golden/ref_calls.npz, see tests/ref_golden.py).
* The numpy grid search is checked against the reference's own generator-based known answer
  (tests/unit-tests/signal-processing-blocks/acquisition/gps_l1_ca_pcps_acquisition_gsoc2013_test.cc:
  207-263: fs 4 Msps, PRN 10 (we use the same numbers), Doppler 750 Hz, delay 600 chips,
  doppler_max 10000, step 250) and the file-based one (gps_l1_ca_pcps_acquisition_test.cc:302-303,
  357-364: delay 524 samples +-0.5 chip, 1680 Hz +-666 Hz at 4 Msps, doppler_max 5000, step 100) on
  an in-repo synthetic analogue (the sourceforge .dat file is not available offline).
* FFT boundary: float32 pocketfft vs float64 pocketfft -> statistics within 1e-4.
"""
import ctypes as C

import numpy as np
import pytest

from gnss_synth import make_iq
from ref_golden import same_bits


@pytest.mark.parametrize("n", [4000, 25000, 8111, 13])
@pytest.mark.parametrize("freq", [-10125.0, -250.0, 0.0, 1680.0, 9875.0])
def test_sincos_ports_bitexact(oracle, ref, n, freq):
    inc = -np.float32(np.float32(2 * np.pi) * np.float32(freq) / np.float32(25e6))
    for variant, fn in (("generic", oracle.port.lib.port_sincos_generic), ("a_avx2", oracle.port.lib.port_sincos_avx2),
                        ("u_avx2", oracle.port.lib.port_sincos_avx2)):
        want, ph_w = ref.sincos(variant, float(inc), 0.0, n)
        got = np.empty(n, np.complex64)
        ph = C.c_float(0.0)
        fn(C.c_void_p(got.ctypes.data), C.c_float(float(inc)), C.byref(ph), C.c_uint(n))
        assert same_bits(got, want), variant
        assert np.float32(ph.value) == np.float32(ph_w)


def test_index_max_first_maximum(oracle, ref):
    rng = np.random.default_rng(3)
    for n in (1, 7, 8, 9, 4000, 25000):
        x = rng.standard_normal(n).astype(np.float32) ** 2
        t = C.c_uint32(0)
        oracle.port.lib.port_index_max_32u(C.byref(t), C.c_void_p(x.ctypes.data), C.c_uint32(n))
        assert t.value == int(np.argmax(x))
        for v in ("generic", "a_avx", "u_avx", "a_sse4_1"):
            assert ref.index_max(v, x) == t.value
    # ties: generic keeps the first
    x = np.zeros(100, np.float32)
    x[[17, 60]] = 5.0
    assert ref.index_max("generic", x) == 17
    oracle.port.lib.port_index_max_32u(C.byref(t), C.c_void_p(x.ctypes.data), C.c_uint32(100))
    assert t.value == 17


def _make(oracle, prn, fs, doppler, delay_samples, cn0, n_ms=1, seed=1):
    from oracle.acq_np import AcqConf
    code = oracle.port.gps_ca_code(prn)
    spc = fs / 1.023e6
    n = int(fs * 1e-3) * n_ms
    # the replica starts `delay_samples` into the buffer: code phase at sample 0 = -delay (in chips)
    sv = dict(prn=prn, doppler=doppler, code_phase_chips=(-(delay_samples) / spc) % 1023, cn0=cn0, phase0=0.4)
    iq = make_iq({prn: code}, fs, n, [sv], seed=seed)
    return code, iq


def test_known_answer_generator_case(oracle):
    from oracle.acq_np import AcqConf, PcpsAcquisitionOracle
    fs = 4e6
    # 600 chips of delay at 4 Msps -> 600*4000/1023 samples
    delay = round(600 * 4000 / 1023)
    code, iq = _make(oracle, 10, fs, 750.0, delay, 44.0, seed=10)
    conf = AcqConf(fs_in=4000000, samples_per_ms=4000, samples_per_code=4000, samples_per_chip=4, doppler_max=10000,
                   doppler_step=250, pfa=0.001, use_CFAR_algorithm_flag=True)
    acq = PcpsAcquisitionOracle(conf)
    acq.set_local_code(oracle.port.gps_ca_code_complex_sampled(10, 4000000))
    r = acq.acquisition_core(iq)
    assert r["positive"]
    assert abs(r["acq_delay_samples"] - delay) <= 2          # +-0.5 chip = +-2 samples
    assert abs(r["acq_doppler_hz"] - 750.0) <= 250.0          # within one Doppler step
    assert conf.num_doppler_bins == 80


def test_known_answer_file_analogue(oracle):
    """PRN 1, delay 524 samples, 1680 Hz at 4 Msps, doppler_max=5000 step=100, threshold path."""
    from oracle.acq_np import AcqConf, PcpsAcquisitionOracle
    code, iq = _make(oracle, 1, 4e6, 1680.0, 524, 47.0, seed=1)
    conf = AcqConf(fs_in=4000000, samples_per_ms=4000, samples_per_code=4000, samples_per_chip=4, doppler_max=5000,
                   doppler_step=100, pfa=0.0, threshold=0.001, use_CFAR_algorithm_flag=False)
    acq = PcpsAcquisitionOracle(conf)
    acq.set_local_code(oracle.port.gps_ca_code_complex_sampled(1, 4000000))
    r = acq.acquisition_core(iq)
    assert r["positive"]
    assert abs(r["acq_delay_samples"] - 524) <= 2
    assert abs(r["acq_doppler_hz"] - 1680.0) <= 666.0
    assert r["test_statistics"] > 2.0     # first/second peak ratio of a real detection


def test_threshold_formula():
    """compute_threshold (pcps_acquisition.cc:52-56): 2*gamma_p_inv(2*dwells, (1-pfa)^(1/nbins))
    cross-checked against the closed form for a=2: P(2,x) = 1-(1+x)e^-x."""
    from oracle.acq_np import compute_threshold
    th = compute_threshold(0.001, 4000, 80, 1)
    x = th / 2.0
    p = 1.0 - (1.0 + x) * np.exp(-x)
    assert abs(p - (1 - 0.001) ** (1.0 / 320000.0)) < 1e-12
    assert 30 < th < 50


def test_fft_boundary_float32_vs_float64(oracle):
    """statistics from float32 FFTs agree with float64 FFTs to 1e-4 and indices exactly."""
    import scipy.fft as sfft
    from oracle.acq_np import AcqConf, PcpsAcquisitionOracle
    code, iq = _make(oracle, 5, 4e6, -3250.0, 1717, 45.0, seed=5)
    conf = AcqConf(doppler_max=5000, doppler_step=250, pfa=0.001)
    acq = PcpsAcquisitionOracle(conf)
    acq.set_local_code(oracle.port.gps_ca_code_complex_sampled(5, 4000000))
    r = acq.acquisition_core(iq)
    # float64 recomputation of the same grid
    wipe = acq.grid_doppler_wipeoffs.astype(np.complex128)
    codes = np.conj(sfft.fft(oracle.port.gps_ca_code_complex_sampled(5, 4000000).astype(np.complex128)))
    y = sfft.ifft(sfft.fft(iq.astype(np.complex128)[None, :] * wipe, axis=1) * codes[None, :], axis=1, norm="forward")
    mag = np.abs(y) ** 2
    d, t = np.unravel_index(np.argmax(mag), mag.shape)
    assert (d, t) == (r["index_doppler"], r["index_time"])
    opp = (d + conf.num_doppler_bins // 2) % conf.num_doppler_bins
    stat = mag[d, t] / (mag[opp].sum() / 4000 / 2.0)
    assert abs(stat - r["test_statistics"]) / stat < 1e-4
