"""Pin the C restatement (oracle/port_trk.c) BIT-EXACT against the reference's own kernels.

Shapes follow the reference QA: vlen 8111, puppet parameters
(VG kernels/volk_gnsssdr/volk_gnsssdr_32f_resamplerxnpuppet_32f.h:32-56:
 L=2046, step=(L+0.1)/N, rem=-0.234, shifts {-0.1,0,0.1};
 ..._32fc_32f_rotator_dotprodxnpuppet_32fc.h:31-55: rem 0.25 rad, step 0.1 rad, 3 taps)
plus the BASELINE shapes (N=25000 L=1023 3 taps; N=200000 L=8184 5 taps) and ragged sizes.
The reference's outputs for these calls are stored in tests/golden/ref_calls.npz (tests/ref_golden.py).
"""
import numpy as np
import pytest

from ref_golden import same_bits


CASES = [
    # (n, L, shifts, rem, step)
    (8111, 2046, [-0.1, 0.0, 0.1], -0.234, (2046 + 0.1) / 8111),
    (25000, 1023, [-0.5, 0.0, 0.5], 0.37, 1.023e6 * (1 + 3000 / 1575.42e6) / 25e6),
    (25001, 1023, [-0.5, 0.0, 0.5], 0.93, 1.023e6 * (1 - 4500 / 1575.42e6) / 25e6),
    (200000, 8184, [-1.2, -0.3, 0.0, 0.3, 1.2], 1.71, 2 * 1.023e6 / 50e6),
    (4000, 1023, [-0.5, 0.0, 0.5], 0.0, 1.023e6 / 4e6),
    (2048, 1023, [-0.5, 0.0, 0.5], 0.4, 0.3),      # reference timing-test parameters
    (37, 1023, [-700.25, 0.0, 1500.5], 3.3, 0.7),   # multi-period negative / positive wraps
    (7, 11, [-0.5, 0.0], 0.2, 1.9),                 # shorter than one AVX iteration
]


@pytest.mark.parametrize("n,L,shifts,rem,step", CASES)
def test_resampler_generic_bitexact(oracle, ref, n, L, shifts, rem, step):
    rng = np.random.default_rng(n)
    code = rng.choice([-1.0, 1.0], L).astype(np.float32)
    a = oracle.port.resampler(0, code, rem, step, shifts, n)
    b = ref.resampler("generic", code, rem, step, shifts, n)
    assert same_bits(a, b)


@pytest.mark.parametrize("n,L,shifts,rem,step", CASES)
@pytest.mark.parametrize("variant", ["a_avx", "u_avx"])
def test_resampler_avx_bitexact(oracle, ref, variant, n, L, shifts, rem, step):
    rng = np.random.default_rng(n + 1)
    # non-binary code values so that equal outputs imply equal chip indices
    code = rng.standard_normal(L).astype(np.float32)
    a = oracle.port.resampler(1, code, rem, step, shifts, n)
    b = ref.resampler(variant, code, rem, step, shifts, n)
    assert same_bits(a, b)


@pytest.mark.parametrize("n,taps", [(8111, 3), (25000, 3), (200000, 5), (4096, 1), (100, 3), (15, 2), (16, 2), (1041, 4)])
def test_rotator_generic_bitexact(oracle, ref, n, taps):
    rng = np.random.default_rng(n)
    iq = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    codes = rng.choice([-1.0, 1.0], (taps, n)).astype(np.float32)
    inc = np.complex64(np.exp(-1j * 0.1))
    ph0 = np.complex64(np.cos(0.25) - 1j * np.sin(0.25))
    a, pa = oracle.port.rotator_generic(iq, inc, ph0, codes)
    b, pb = ref.rotator("generic", iq, inc, ph0, codes)
    assert same_bits(a, b)
    assert same_bits(np.array([pa]), np.array([pb]))


@pytest.mark.parametrize("n,taps", [(8111, 3), (25000, 3), (200000, 5), (4096, 1), (100, 3), (15, 2), (16, 2), (1041, 4)])
@pytest.mark.parametrize("variant", ["u_avx", "a_avx"])
def test_rotator_avx_bitexact(oracle, ref, variant, n, taps):
    rng = np.random.default_rng(n + 7)
    iq = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    codes = rng.choice([-1.0, 1.0], (taps, n)).astype(np.float32)
    inc = np.complex64(np.exp(-1j * 0.00126))
    ph0 = np.complex64(np.cos(0.4) - 1j * np.sin(0.4))
    a, pa = oracle.port.rotator_avx(iq, inc, ph0, codes)
    b, pb = ref.rotator(variant, iq, inc, ph0, codes)
    assert same_bits(a, b)
    assert same_bits(np.array([pa]), np.array([pb]))


def test_rotator_avx_vs_generic_within_reference_tolerance(ref):
    """The reference's own pin: arch vs generic within 1e-3 (lib/kernel_tests.h:41,87-89)."""
    n, taps = 8111, 3
    rng = np.random.default_rng(0)
    iq = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    codes = np.tile(rng.standard_normal(n).astype(np.float32), (taps, 1))
    inc = np.complex64(np.exp(-1j * 0.1))
    ph0 = np.complex64(np.cos(0.25) - 1j * np.sin(0.25))
    g, _ = ref.rotator("generic", iq, inc, ph0, codes)
    a, _ = ref.rotator("u_avx", iq, inc, ph0, codes)
    assert np.all(np.abs(a - g) / np.abs(g) < 1e-3)


@pytest.mark.parametrize("arch,refarch", [(0, "generic"), (1, "a_avx"), (1, "u_avx")])
@pytest.mark.parametrize("n,L,shifts", [(25000, 1023, [-0.5, 0, 0.5]), (8000, 1023, [-0.5, 0, 0.5]),
                                        (200000, 8184, [-1.2, -0.3, 0, 0.3, 1.2]), (4001, 1023, [-0.25, 0.0, 0.25])])
def test_multicorrelator_class_bitexact(oracle, ref, arch, refarch, n, L, shifts):
    """Whole a3 path against the reference's Cpu_Multicorrelator_Real_Codes (high_dyn=false)."""
    rng = np.random.default_rng(n + arch)
    code = rng.choice([-1.0, 1.0], L).astype(np.float32)
    iq = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    rem_carr, dphi = 1.234, 2 * np.pi * 2500.0 / 25e6
    rem_code, step = 0.61 * (L / 1023), L / n * 1.000002
    ref.select_arch(refarch)
    h = ref.mc_create(n, len(shifts), high_dyn=False)
    ref.mc_set_code(h, code, shifts)
    b = ref.mc_correlate(h, iq, len(shifts), rem_carr, dphi, 0.0, rem_code, step, 0.0)
    ref.mc_destroy(h)
    ref.select_arch("a_avx")
    a = oracle.port.multicorrelator(arch, iq, code, shifts, rem_carr, dphi, rem_code, step)
    assert same_bits(a, b)


def test_hd_resampler_bitexact(oracle, ref):
    rng = np.random.default_rng(5)
    for n, L, shifts, step in [(8111, 2046, [-0.1, 0.0, 0.1], (2046 + 0.1) / 8111), (25000, 1023, [-0.5, 0, 0.5], 0.04092),
                               (70000, 8184, [-0.6, -0.15, 0, 0.15, 0.6], 0.04092)]:
        code = rng.standard_normal(L).astype(np.float32)
        a = oracle.port.hd_resampler(code, -0.234, step, 1e-9, shifts, n)
        b = ref.hd_resampler("generic", code, -0.234, step, 1e-9, shifts, n)
        assert same_bits(a, b)


@pytest.mark.parametrize("variant", ["a_avx", "u_avx"])
def test_hd_resampler_avx_bitexact(oracle, ref, variant):
    rng = np.random.default_rng(15)
    for n, L, shifts, step, rate in [(8111, 2046, [-0.1, 0.0, 0.1], (2046 + 0.1) / 8111, 1e-9),
                                     (25000, 1023, [-0.5, 0, 0.5], 0.04092, 3e-12),
                                     (25003, 1023, [-0.5, 0, 0.5], 0.04092, -3e-12),
                                     (200000, 8184, [-1.2, -0.3, 0, 0.3, 1.2], 0.04092, 1e-13),
                                     (4000, 1023, [-0.5, 0, 0.5], 0.25575, 2e-10)]:
        code = rng.standard_normal(L).astype(np.float32)
        a = oracle.port.hd_resampler_avx(code, 0.37, step, rate, shifts, n)
        b = ref.hd_resampler(variant, code, 0.37, step, rate, shifts, n)
        assert same_bits(a, b), (variant, n)


def test_hd_rotator_bitexact(oracle, ref):
    rng = np.random.default_rng(6)
    n, taps = 3000, 3
    iq = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    codes = rng.choice([-1.0, 1.0], (taps, n)).astype(np.float32)
    inc = np.complex64(np.exp(-1j * 0.0126))
    rate = np.complex64(np.exp(-1j * 1e-8))
    ph0 = np.complex64(np.cos(0.4) - 1j * np.sin(0.4))
    a, pa = oracle.port.hd_rotator_generic(iq, inc, rate, ph0, codes)
    b, pb = ref.hd_rotator("generic", iq, inc, rate, ph0, codes)
    assert same_bits(a, b)
    assert same_bits(np.array([pa]), np.array([pb]))


def test_f64_truth_bounds_float_paths(oracle):
    """float32 CPU paths sit within 1e-5 (relative to |P|) of the float64 truth at C2 shape."""
    n, L = 25000, 1023
    rng = np.random.default_rng(11)
    code = oracle.port.gps_ca_code(7)
    shifts = [-0.5, 0.0, 0.5]
    step = 1.023e6 / 25e6
    # signal + noise at ~45 dB-Hz so the prompt is a real peak
    k = np.arange(n)
    chips = code[np.floor(k * step + 0.3).astype(int) % L]
    iq = (0.05 * chips * np.exp(1j * (0.7 + k * 1e-3)) + (rng.standard_normal(n) + 1j * rng.standard_normal(n))
          ).astype(np.complex64)
    t = oracle.port.multicorrelator_f64(1, iq, code, shifts, 0.7, 1e-3, -0.3, step)
    for arch in (0, 1):
        a = oracle.port.multicorrelator(arch, iq, code, shifts, 0.7, 1e-3, -0.3, step)
        assert np.max(np.abs(a - t)) / np.abs(t[1]) < (2e-4 if arch == 0 else 1e-5)
