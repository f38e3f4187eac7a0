#!/usr/bin/env python
"""Generate tests/golden/*.npz from the REFERENCE's own code (oracle/_ref/*.so, built in place by oracle/Makefile when
the reference tree is present):

    python tests/golden/make_golden.py [fixture ...]      (default: all of them)

Inputs are regenerated from seeds by the tests (tests/gnss_synth.py, numpy default_rng), so the
fixtures hold only parameters and the reference's outputs:
  trk_ref_golden.npz    Cpu_Multicorrelator_Real_Codes (a_avx kernels, high_dyn false/true) taps,
                        and generic-kernel taps, for the shapes in CASES
  loop_ref_golden.npz   per-epoch item scalars and 108-byte dump records of the DLL/PLL cycle evaluated with the
                        reference's own Tracking_loop_filter / Tracking_FLL_PLL_filter / Exponential_Smoother /
                        discriminator / lock-detector code (oracle/ref_loop.cc) for seeded correlator outputs
  acq_ref_golden.npz    volk_gnsssdr_s32f_sincos_32fc a_avx2 wipe-off rows (bit patterns) for a few
                        Doppler bins, and volk_gnsssdr_32f_index_max_32u results
  ref_calls.npz         every oracle.ref call of tests/test_oracle_port_vs_ref.py and tests/test_oracle_acq.py and
                        what it returned (tests/ref_golden.py; recorded by running those tests on the live library)
  loop_ref_pins.npz     the reference's discriminators / lock detectors, per-block digests of its loop cycle, the closed
                        loop over its correlator and its dump-file reader, on the inputs of tests/test_oracle_loop.py
  blocks_ref_golden.npz the reference's acquisition + ChannelFsm + tracking blocks on the signal of the CPU tests of
                        tests/test_integration_blocks.py and the replica they track; its Cpu_Multicorrelator and
                        Cpu_Multicorrelator_16sc on the inputs of two tests of tests/test_trk_gpu.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
HERE = os.path.dirname(os.path.abspath(__file__))

# (name, seed, fs, n, L, prn or None (random +-1 table), shifts, doppler, code_phase, table_chips_per_chip, high_dyn)
CASES = [
    ("gps_4msps", 101, 4e6, 4000, 1023, 1, [-0.5, 0.0, 0.5], 1680.0, 131.25, 1.0, False),
    ("gps_25msps", 102, 25e6, 25000, 1023, 7, [-0.5, 0.0, 0.5], -3217.0, 417.3, 1.0, False),
    ("gps_25msps_ragged", 103, 25e6, 25003, 1023, 19, [-0.5, 0.0, 0.5], 4711.0, 12.9, 1.0, False),
    ("e1_50msps", 104, 50e6, 200000, 8184, None, [-1.2, -0.3, 0.0, 0.3, 1.2], -1234.5, 1000.25, 2.0, False),
    ("gps_25msps_hd", 105, 25e6, 25000, 1023, 9, [-0.5, 0.0, 0.5], 2500.0, 600.1, 1.0, True),
]


# DLL/PLL loop fixture: (name, conf overrides, epochs); taps = loop_harness.synthetic_taps(epochs, taps, LOOP_SEED)
LOOP_SEED = 77
LOOP_CASES = [
    ("gps_default", dict(), 600),
    ("pll2_dll1_fll", dict(pll_filter_order=2, dll_filter_order=1, enable_fll_pull_in=1, pull_in_time_s=1), 600),
    ("veml_e1", dict(veml=1, code_samples_per_chip=2, early_late_space_chips=0.15, dll_filter_order=3), 600),
]


def case_inputs(oracle, case):
    from gnss_synth import make_iq, trk_params_for
    name, seed, fs, n, L, prn, shifts, doppler, cph, tcpc, hd = case
    rng = np.random.default_rng(seed)
    if prn is not None:
        code = oracle.port.gps_ca_code(prn)
    else:
        code = oracle.port.sinboc11(rng.choice([-1, 1], L // 2))
    sv = dict(prn=1, doppler=doppler, code_phase_chips=cph, cn0=45.0, phase0=0.9)
    iq = make_iq({1: code}, fs, n, [sv], seed=seed, chips_per_table_chip=tcpc)
    _, rc, dp, rcode, st = trk_params_for(sv, fs, n, 1, table_chips_per_chip=tcpc, L=L)
    return code, iq, (float(rc[0]), float(dp[0]), float(rcode[0]), float(st[0]))


def trk():
    import oracle
    out = {}
    for case in CASES:
        name, *_rest = case
        hd = case[-1]
        shifts = case[6]
        code, iq, (rc, dp, rcode, st) = case_inputs(oracle, case)
        for arch in ("a_avx", "generic"):
            oracle.ref.select_arch(arch)
            h = oracle.ref.mc_create(len(iq), len(shifts), high_dyn=hd)
            oracle.ref.mc_set_code(h, code, shifts)
            rate = (2e-9, 2e-12) if hd else (0.0, 0.0)
            taps = oracle.ref.mc_correlate(h, iq, len(shifts), rc, dp, rate[0], rcode, st, rate[1])
            oracle.ref.mc_destroy(h)
            out[f"{name}/{arch}"] = taps
        out[f"{name}/params"] = np.array([rc, dp, rcode, st], np.float32)
    oracle.ref.select_arch("a_avx")
    np.savez(os.path.join(HERE, "trk_ref_golden.npz"), **out)


def acq():
    import oracle
    acq = {}
    for fs, n in ((4e6, 4000), (25e6, 25000)):
        for f in (-5000.0, -250.0, 1680.0, 9875.0):
            inc = -np.float32(np.float32(2 * np.pi) * np.float32(f) / np.float32(fs))
            row, ph = oracle.ref.sincos("a_avx2", float(inc), 0.0, n)
            # keep the fixture small: first 64, last 64 samples and a CRC-like checksum of all bit patterns
            bits = row.view(np.uint32)
            acq[f"sincos/{int(fs)}/{int(f)}/head"] = bits[:128].copy()
            acq[f"sincos/{int(fs)}/{int(f)}/tail"] = bits[-128:].copy()
            acq[f"sincos/{int(fs)}/{int(f)}/xor_sum"] = np.array([np.bitwise_xor.reduce(bits), np.sum(bits.astype(np.uint64)) & 0xFFFFFFFFFFFF], np.uint64)
    np.savez(os.path.join(HERE, "acq_ref_golden.npz"), **acq)


def loop():
    # DLL/PLL loop: records and item scalars produced by the reference's own loop-filter / discriminator /
    # lock-detector / smoother objects (oracle/_ref/liboracle_ref_loop.so) for seeded correlator outputs
    from oracle import loop as ol
    import loop_harness as lh
    lp = {}
    for name, kw, n_ep in LOOP_CASES:
        conf = ol.default_conf(fs_in=4e6, **kw)
        R = ol.RefLoop(conf)
        R.start(524.3, 1680.0, 1000, 9000)
        taps = lh.synthetic_taps(n_ep, 5 if conf.veml else 3, seed=LOOP_SEED)
        recs, items = [], []
        for k in range(n_ep):
            s, n, p6 = R.prepare()
            items.append(np.concatenate([[s, n], p6.view(np.uint32)]).astype(np.uint64))
            ok, r = R.update(taps[k])
            assert ok
            recs.append(r)
        lp[f"{name}/records"] = np.frombuffer(np.array(recs, ol.DUMP_RECORD_DTYPE).tobytes(), np.uint8)
        lp[f"{name}/items"] = np.array(items, np.uint64)
    np.savez_compressed(os.path.join(HERE, "loop_ref_golden.npz"), **lp)


def ref_calls():
    """Run the pin tests with the `ref` fixture recording the live library's answers (the tests' own comparisons of the
    port with the live reference run at the same time and must pass)."""
    import subprocess
    env = dict(os.environ, B200_RECORD_REF_CALLS="1")
    subprocess.check_call([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "tests/test_oracle_port_vs_ref.py",
                           "tests/test_oracle_acq.py"], cwd=ROOT, env=env)


def loop_pins():
    import hashlib
    import oracle
    from oracle import loop as ol
    import loop_harness as lh
    import test_oracle_loop as t
    g = {f"lib/{k}": v for k, v in t.library_outputs(ol.ref_lib(), "ref_").items()}
    for i, kw in enumerate(t.CONFS):
        trace, lost, (ints, dbls) = t.cycle_trace(ol.RefLoop, kw)
        g[f"cycle{i}/trace"], g[f"cycle{i}/lost"] = trace, np.array(int(lost))
        g[f"cycle{i}/status_int"], g[f"cycle{i}/status_dbl"] = ints, dbls
    oracle.ref.select_arch("a_avx")
    recs, _, _ = t.closed_loop_records(oracle, lambda code, shifts, max_len: lh.RefCorrelator(oracle.ref, code, shifts, max_len))
    g["closed_loop/records_sha"] = np.frombuffer(hashlib.sha256(recs.tobytes()).digest(), np.uint8)
    recs = t.dump_records()
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        fn = os.path.join(d, "trk_dump_ch0.dat")
        t.write_dump(fn, recs)
        with open(fn, "rb") as f:
            g["dump/file_sha"] = np.frombuffer(hashlib.sha256(f.read()).digest(), np.uint8)
        g["dump/read"] = ol.ref_dump_read(fn)
    np.savez_compressed(os.path.join(HERE, "loop_ref_pins.npz"), **g)


def blocks():
    import hashlib
    import blocks_itf as bi
    import test_integration_blocks as t
    lib = bi.ref_lib()
    assert lib is not None, "build oracle/_ref/liboracle_ref_blocks.so first (make -C oracle blocks)"
    code = bi.code_table(lib, "G", "1C", 1)
    g = {"code/G/1C/1": code}
    iq, _ = t.make_gps_signal(code)
    for name, (over, arch, seconds) in t.REF_RUNS.items():
        x = iq[:int(t.FS * seconds)]
        lib.itf_select_arch(arch.encode())
        r = t.run_chain(lib, t.base_conf(**over), "GPS_L1_CA_PCPS_Acquisition", "GPS_L1_CA_DLL_PLL_Tracking", x)
        g[f"{name}/iq_sha"] = np.frombuffer(hashlib.sha256(np.ascontiguousarray(x).tobytes()).digest(), np.uint8)
        g[f"{name}/acq"] = np.array(r["acq"], np.float64)
        g[f"{name}/acq_events"] = np.array(r["acq_events"], np.int64)
        g[f"{name}/started"] = np.array(r["started"])
        g[f"{name}/out"] = np.frombuffer(r["out"].tobytes(), np.uint8)
        g[f"{name}/trk_events"] = np.array(r["trk_events"], np.int64)
    lib.itf_select_arch(b"simd")
    # Cpu_Multicorrelator (complex code) and Cpu_Multicorrelator_16sc on the inputs of tests/test_trk_gpu.py
    import test_trk_gpu as tt
    sig, code, shifts, rem_code, step, carriers = tt.cplx_case()
    g["trk_cplx/want"] = np.array([bi.ref_mc_cplx_code(lib, sig, code, shifts, rc, dp, rem_code, step) for rc, dp in carriers])
    sig, code, shifts, rem_code, step, carriers = tt.sc16_case()
    g["trk_16sc/want"] = np.array([bi.ref_mc_16sc(lib, sig, code, shifts, rc, dp, rem_code, step) for rc, dp in carriers])
    np.savez_compressed(os.path.join(HERE, "blocks_ref_golden.npz"), **g)


FIXTURES = {"trk": trk, "acq": acq, "loop": loop, "ref_calls": ref_calls, "loop_pins": loop_pins, "blocks": blocks}


def main(names):
    import oracle
    assert oracle.ref is not None, "build oracle/_ref first (needs the reference tree; see oracle/Makefile)"
    for name in names or FIXTURES:
        FIXTURES[name]()
    print("wrote", sorted(os.listdir(HERE)))


if __name__ == "__main__":
    main(sys.argv[1:])
