#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 tracking-correlator hot path (BASELINE.json metric
"Msamples/s through N-channel E/P/L correlator"), workload = BASELINE configs[1] (SURVEY 8d "C2"):
GPS L1 C/A, 32 channels, 25 Msps synthetic IQ, 3 taps (E/P/L), 1 s of signal per step
(1000 epochs of 25000 samples per channel => 8e8 channel-samples per step).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for every field.  --dump-outputs DIR writes the taps
the last timed step returned to DIR/trk_taps.npy, so that two builds can be compared output for output (the inputs
are generated from fixed seeds).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the benchmark may run from a read-only tree: no __pycache__ beside the sources
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "Msamples/s through N-channel E/P/L correlator"
UNIT = "Msamples/s"

# ---- workload C2 -------------------------------------------------------------------------------
FS = 25e6
N_CH = 32
EPOCH = 25000           # vector_length at 25 Msps (gps_l1_ca_dll_pll_tracking.cc:59)
N_EPOCHS = 1000         # 1 s of signal per step
TAPS = 3
SHIFTS = [-0.5, 0.0, 0.5]
SEED = 2
ALGO_BYTES_PER_CHANNEL_SAMPLE = 8   # one cf32 read per channel-sample (SURVEY 8d)


def config_dict(n_gpus):
    return {"workload": "C2: GPS L1 C/A, 32 channels x 25 Msps x 1 s (1000 epochs of 25000 samples), 3 taps E/P/L, "
                        "open-loop per-epoch NCO parameters",
            "channels_per_gpu": N_CH, "fs_sps": FS, "epoch_samples": EPOCH, "epochs_per_step": N_EPOCHS, "taps": TAPS,
            "channel_samples_per_step_per_gpu": N_CH * EPOCH * N_EPOCHS,
            "l2_policy": "IQ band (200 MB) exceeds L2 (126 MB); streamed once per step, shared by the 32 channels",
            "sharding": (f"ONE receiver, ONE band, {N_CH} x {n_gpus} channels: every rank correlates its own {N_CH} channels on the same IQ "
                         "stream; end to end the band crosses PCIe once (rank 0) and fans out to the peers by one NCCL broadcast over "
                         "NVLink per step (SURVEY 8e); no other data-path collective") if n_gpus > 1 else "single GPU"}


def svs_for_rank(rank):
    rng = np.random.default_rng(SEED + 1000 * rank)
    return [dict(prn=p, doppler=float(rng.uniform(-5000, 5000)), code_phase_chips=float(rng.uniform(0, 1023)),
                 cn0=45.0, phase0=float(rng.uniform(0, 2 * np.pi))) for p in range(1, N_CH + 1)]


def build_items(capi, svs, cids, first_index):
    from gnss_synth import trk_params_for
    items = np.zeros(N_CH * N_EPOCHS, capi.TRK_ITEM_DTYPE)
    v = items.reshape(N_EPOCHS, N_CH)      # epoch-major: the 32 channels of one epoch are neighbours (L2 sharing)
    for c, sv in enumerate(svs):
        s, rc, dp, rcode, st = trk_params_for(sv, FS, EPOCH, N_EPOCHS)
        v["channel"][:, c] = cids[c]
        v["n"][:, c] = EPOCH
        v["sample_index"][:, c] = first_index + s
        v["rem_carrier_phase_rad"][:, c] = rc
        v["phase_step_rad"][:, c] = dp
        v["rem_code_phase_chips"][:, c] = rcode
        v["code_phase_step_chips"][:, c] = st
    return items


def synth_iq_device(torch, codes, svs, n, seed, device):
    """Sum of 32 SV signals + AWGN, generated on the GPU in chunks (same model as tests/gnss_synth.make_iq)."""
    from gnss_synth import ca_amplitude, CA_RATE, GPS_L1_FREQ
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty((n, 2), dtype=torch.float32, device=device)
    chunk = 1 << 22
    tabs = {p: torch.from_numpy(codes[p]).to(device) for p in codes}
    for a in range(0, n, chunk):
        b = min(n, a + chunk)
        t = torch.arange(a, b, dtype=torch.float64, device=device)
        re = torch.randn(b - a, generator=g, device=device, dtype=torch.float32).double()
        im = torch.randn(b - a, generator=g, device=device, dtype=torch.float32).double()
        for sv in svs:
            rate = CA_RATE * (1.0 + sv["doppler"] / GPS_L1_FREQ)
            idx = torch.floor(sv["code_phase_chips"] + t * (rate / FS)).long() % 1023
            c = tabs[sv["prn"]][idx].double() * ca_amplitude(sv["cn0"], FS)
            ph = sv["phase0"] + 2 * np.pi * sv["doppler"] / FS * t
            re += c * torch.cos(ph)
            im += c * torch.sin(ph)
        out[a:b, 0] = re.float()
        out[a:b, 1] = im.float()
    return out


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic_bytes():
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        with open(p) as f:
            return json.load(f).get("trk_correlate_kernel_bytes_per_launch")
    except Exception:
        return None


def ncu_acq_traffic_bytes():
    """DRAM bytes of one acq_corr_kernel launch (C4 sweep) from the committed ncu capture."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        with open(p) as f:
            d = json.load(f).get("acq_corr_kernel<512>", {})
            return int(d.get("dram__bytes_read.sum", 0)) + int(d.get("dram__bytes_write.sum", 0))
    except Exception:
        return None


def ncu_limiter():
    """What ncu says bounds the dominant kernel (committed summary of the --set full capture)."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        with open(p) as f:
            return json.load(f).get("limiter")
    except Exception:
        return None


_AFFINITY_BEFORE_BINDING = None


class whole_host:
    """The CPU arms get every CPU the process was started with, not only the GPU's NUMA node."""
    def __enter__(self):
        self.saved = None
        if _AFFINITY_BEFORE_BINDING is not None:
            self.saved = os.sched_getaffinity(0)
            os.sched_setaffinity(0, _AFFINITY_BEFORE_BINDING)
        return self

    def __exit__(self, *a):
        if self.saved is not None:
            os.sched_setaffinity(0, self.saved)
        return False


def bind_to_gpu_numa(torch, local_rank):
    """Bind this rank (and with it the first-touch placement of its pinned buffers) to the NUMA node its GPU hangs off.
    Round 1: eight unbound ranks pushing 54 GB/s each halved the 8-GPU end-to-end efficiency."""
    bus = None
    try:
        if bus is None:
            out = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                 capture_output=True, text=True, timeout=10).stdout.strip()
            bus = out
        bus = bus.lower()
        if bus.count(":") == 2 and len(bus.split(":")[0]) == 8:
            bus = bus[4:]            # nvidia-smi prints an 8-digit domain, sysfs uses 4
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return {"numa_node": None, "bound": False, "why": "single NUMA node"}
        cpulist = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        cpus = set()
        for part in cpulist.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        global _AFFINITY_BEFORE_BINDING
        if _AFFINITY_BEFORE_BINDING is None:
            _AFFINITY_BEFORE_BINDING = set(allowed)
        use = sorted(cpus & allowed) or sorted(allowed)
        os.sched_setaffinity(0, use)
        return {"numa_node": node, "bound": True, "cpus": len(use)}
    except Exception as ex:
        return {"numa_node": None, "bound": False, "why": repr(ex)}


def run_trk_config(torch, capi, dev, name, fs, groups, seconds, steps=20, warmup=3, layout="shared", stream=None, kernel=None):
    """Device-resident throughput of the tracking correlator on one workload.
    groups: list of dict(n_ch, N, L, shifts, table_rate[, pilot_data]); table_rate = table values per second;
    pilot_data=True adds, per channel, the 1-tap data-prompt correlator of a tracked pilot (dll_pll_veml_tracking.cc:1246-1256).
    layout "shared": all channels read one band (a receiver); "distinct": every (channel, epoch) work item reads its own
    region of a channels-times-larger band, so that 8 B per channel-sample really cross HBM (the roofline run of SURVEY 8d)."""
    st = stream or torch.cuda.current_stream(dev)
    eng = capi.Engine(dev.index, st.cuda_stream)
    if kernel is not None:
        eng.trk_kernel_choice(kernel)
    n_ch_total = sum(g["n_ch"] for g in groups)
    n_iq = int(fs * seconds)
    g = torch.Generator(device=dev)
    g.manual_seed(3)
    band_len = n_iq * (n_ch_total if layout == "distinct" else 1)
    iq = torch.randn((band_len + 16, 2), generator=g, device=dev, dtype=torch.float32)
    eng.iq_attach_dev(0, iq.data_ptr(), band_len + 16, 0)
    rng = np.random.default_rng(3)
    items = []
    max_taps = max(len(gr["shifts"]) for gr in groups)
    ch_samples = 0
    c_global = 0
    for gr in groups:
        for c in range(gr["n_ch"]):
            code = rng.choice([-1.0, 1.0], gr["L"]).astype(np.float32)
            cids = [eng.channel_create(0, len(gr["shifts"]))]
            eng.channel_set_code(cids[0], code, gr["shifts"])
            if gr.get("pilot_data"):
                cids.append(eng.channel_create(0, 1))
                eng.channel_set_code(cids[1], rng.choice([-1.0, 1.0], gr["L"]).astype(np.float32), [0.0])
            n_ep = n_iq // gr["N"]
            doppler = rng.uniform(-5000, 5000)
            step = gr["table_rate"] * (1 + doppler / 1575.42e6) / fs
            k = np.arange(n_ep)
            for cid in cids:
                arr = np.zeros(n_ep, capi.TRK_ITEM_DTYPE)
                arr["channel"] = cid
                arr["n"] = gr["N"]
                arr["sample_index"] = k * gr["N"] + (c_global * n_iq if layout == "distinct" else 0)
                arr["rem_carrier_phase_rad"] = np.mod(2 * np.pi * doppler / fs * k * gr["N"], 2 * np.pi)
                arr["phase_step_rad"] = 2 * np.pi * doppler / fs
                arr["rem_code_phase_chips"] = -np.mod(rng.uniform(0, gr["L"]) + step * k * gr["N"], gr["L"])
                arr["code_phase_step_chips"] = step
                items.append(arr)
                ch_samples += n_ep * gr["N"]
            c_global += 1
    items = np.concatenate(items)
    if layout == "shared":
        items = items[np.argsort(items["sample_index"], kind="stable")]     # epoch-major: neighbours share samples
    it_dev = torch.from_numpy(items.view(np.uint8)).to(dev)
    out = torch.zeros((items.size, max_taps, 2), dtype=torch.float32, device=dev)
    for _ in range(warmup):
        eng.trk_batch_dev(it_dev.data_ptr(), items.size, out.data_ptr(), max_taps, 1)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(steps):
        eng.trk_batch_dev(it_dev.data_ptr(), items.size, out.data_ptr(), max_taps, 1)
    e1.record(st)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    line = {"workload": name, "layout": layout, "items": int(items.size), "channel_samples_per_step": int(ch_samples), "ms_per_step": ms,
            "value": ch_samples / (ms * 1e-3) / 1e6, "unit": UNIT, "algorithmic_GBps": ch_samples * 8 / (ms * 1e-3) / 1e9,
            "band_bytes": int(band_len * 8)}
    eng.close()
    del iq, out, it_dev
    return line


E1_SHIFTS = [-1.2, -0.3, 0.0, 0.3, 1.2]     # VE/E/P/L/VL at -0.6,-0.15,0,0.15,0.6 chips x 2 table values per chip (:632-636)


def other_configs(torch, capi, dev, stream, steps, only=None):
    """BASELINE configs[2] (C3) with and without the pilot's data tap, the per-GPU share of configs[4] (C5), and the C2
    workload laid out so that the algorithmic bytes really come from HBM."""
    out = {}
    def leg(key, *a, **kw):
        if only and key not in only:
            return
        try:
            out[key] = run_trk_config(torch, capi, dev, *a, steps=steps, stream=stream, **kw)
        except Exception as ex:
            out[key] = {"error": repr(ex)}
    leg("C3", "C3: Galileo E1 64 ch x 50 Msps x 1 s, N=200000, sinBOC(1,1) table of 8184, 5 taps VE/E/P/L/VL", 50e6,
        [dict(n_ch=64, N=200000, L=8184, shifts=E1_SHIFTS, table_rate=2 * 1.023e6)], 1.0)
    leg("C3_track_pilot", "C3 with track_pilot (default): + one data-prompt tap per channel on the E1B replica", 50e6,
        [dict(n_ch=64, N=200000, L=8184, shifts=E1_SHIFTS, table_rate=2 * 1.023e6, pilot_data=True)], 1.0)
    leg("C5_per_gpu_share", "C5 / 8 GPUs: 12 GPS L1 (N=50000) + 12 Galileo E1 (N=200000, 5 taps) + 8 GPS L5 (N=50000, L=10230) at 50 Msps x 1 s",
        50e6, [dict(n_ch=12, N=50000, L=1023, shifts=SHIFTS, table_rate=1.023e6),
               dict(n_ch=12, N=200000, L=8184, shifts=E1_SHIFTS, table_rate=2 * 1.023e6),
               dict(n_ch=8, N=50000, L=10230, shifts=SHIFTS, table_rate=10.23e6)], 1.0)
    # nothing is shared in this layout: the per-item kernel (one CTA per item) is the one b200_trk_submit picks for it (it sees
    # the items); b200_trk_batch_dev cannot look at device-resident items, so the choice is made explicitly here
    leg("C2_distinct_iq", "C2 arithmetic, but every (channel, epoch) reads its own samples: 32 ch x 25 Msps x 0.5 s from a 3.2 GB band; per-item kernel",
        FS, [dict(n_ch=N_CH, N=EPOCH, L=1023, shifts=SHIFTS, table_rate=1.023e6)], 0.5, layout="distinct", kernel=0)
    leg("C2_distinct_iq_shared_window_kernel", "the same through the shared-window kernel (no window to share: each warp streams its own item)",
        FS, [dict(n_ch=N_CH, N=EPOCH, L=1023, shifts=SHIFTS, table_rate=1.023e6)], 0.5, layout="distinct", kernel=1)
    return out


def coalesced_class_interface():
    """Throughput and per-call latency of the reference-shaped CLASS interface (B200_Multicorrelator_Real_Codes, one
    std::thread per channel, C2 epoch size) through the per-process coalescer: tests/host/test_host_mirror --coalescer."""
    exe = os.path.join(ROOT, "tests", "host", "test_host_mirror")
    if not os.path.exists(exe):
        return {"error": "tests/host/test_host_mirror not built"}
    res = []
    for threads, epochs in ((32, 400), (256, 150)):
        try:
            r = subprocess.run([exe, "--coalescer", str(threads), str(epochs), "200"], capture_output=True, text=True, timeout=300)
            line = [ln for ln in r.stdout.splitlines() if ln.startswith("COALESCED ")]
            res.append(json.loads(line[0][len("COALESCED "):]) if line else {"threads": threads, "error": (r.stdout + r.stderr)[-300:]})
        except Exception as ex:
            res.append({"threads": threads, "error": repr(ex)})
    return res


# ---- acquisition sub-benchmark (BASELINE configs[3], SURVEY 8d "C4") -----------------------------------
ACQ_FS = 25000000
ACQ_N = 25000
ACQ_PRNS = 32
ACQ_DMAX, ACQ_DSTEP = 10125, 250     # 81 bins: -10125 ... +9875 Hz (SURVEY 8d, C4)


def acq_rows_bytes_flops():
    import math
    bins = int(math.ceil(2 * ACQ_DMAX / ACQ_DSTEP))
    rows = ACQ_PRNS * bins
    # SURVEY 8d: 16N algorithmic bytes and N(16 + 10 log2 N) flops per (PRN, bin) row
    return bins, rows, rows * 16 * ACQ_N, rows * ACQ_N * (16 + 10 * math.log2(ACQ_N))


def bench_acq(torch, capi, eng, dev, steps, warmup, with_cpu, dist=None, rank=0, world=1):
    from gnss_synth import make_iq, gps_ca_code, gps_ca_code_complex_sampled
    bins, rows, abytes, aflops = acq_rows_bytes_flops()
    rng = np.random.default_rng(4)
    present = [2, 5, 9, 13, 17, 21, 26, 30]
    codes = {p: gps_ca_code(p) for p in present}
    svs = [dict(prn=p, doppler=float(rng.uniform(-9000, 9000)), code_phase_chips=float(rng.uniform(0, 1023)), cn0=45.0,
                phase0=float(rng.uniform(0, 6.28))) for p in present]
    iq = make_iq(codes, float(ACQ_FS), ACQ_N, svs, seed=4)
    acq = capi.PcpsAcquisition(eng, fs_in=ACQ_FS, samples_per_ms=float(ACQ_N), samples_per_chip=24, doppler_max=ACQ_DMAX,
                               doppler_step=ACQ_DSTEP, n_code_slots=ACQ_PRNS)
    assert acq.conf.num_doppler_bins == bins
    for p in range(1, ACQ_PRNS + 1):
        acq.set_local_code(p - 1, gps_ca_code_complex_sampled(p, ACQ_FS))
    # multi-GPU: the PRN x Doppler grid is sharded by PRN; the only exchange is the peak all-reduce
    from gnss_sdr_b200 import dist as bd
    my_slots = np.array(bd.shard_round_robin(ACQ_PRNS, world, rank), dtype=np.uint32)
    slots = my_slots
    iq_dev = torch.from_numpy(iq.view(np.float32)).to(dev)
    res_dev = torch.zeros(len(my_slots) * capi.ACQ_RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    prn_dev = torch.from_numpy((my_slots + 1).astype(np.int64)).to(dev)

    peak_dev = torch.zeros(4, dtype=torch.int32, device=dev)
    prn32_dev = torch.from_numpy((my_slots + 1).astype(np.int32)).to(dev)

    def local_sweep():
        acq.search_dev(iq_dev.data_ptr(), slots, res_dev.data_ptr())
        if world > 1:
            acq.sweep_best_dev(res_dev.data_ptr(), prn32_dev.data_ptr(), len(my_slots), peak_dev.data_ptr())

    # the sweep's launches are captured once in a CUDA graph (a repeated sweep over the same slots issues no host
    # synchronisation): one graph launch per sweep instead of five kernel launches through ctypes
    graph = None
    try:
        local_sweep()
        torch.cuda.synchronize()
        cur = torch.cuda.current_stream(dev)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=cur):
            local_sweep()
        torch.cuda.synchronize()
    except Exception:
        graph = None
        torch.cuda.synchronize()

    gathered = [None]

    def sweep():
        if graph is not None:
            graph.replay()
        else:
            local_sweep()
        if world > 1:
            # the only exchange: an all-gather of the ranks' 16-byte (statistic, PRN, bin, code phase) records over NVLink
            gathered[0] = bd.allgather_peaks(peak_dev)
        return gathered[0]

    for _ in range(warmup):
        sweep()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    l0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        best = sweep()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if dist is not None:
        tms = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
    launches = (eng.launch_count() - l0) if graph is None else steps * (5 if world == 1 else 6)
    res_local = np.frombuffer(res_dev.cpu().numpy().tobytes(), capi.ACQ_RESULT_DTYPE)
    if world > 1:
        res = bd.gather_results(res_local, [int(x) for x in my_slots], ACQ_PRNS, device=dev)
        winner = bd.best_peak(best.cpu().numpy().view(bd.PEAK_DTYPE))
        w = int(np.argmax(res["test_statistics"]))
        assert int(winner["prn"]) == w + 1 and int(winner["index_time"]) == int(res["index_time"][w]), "exchanged peak != gathered table"
    else:
        res = res_local
    # compute_threshold (pcps_acquisition.cc:52-56): 2 * gamma_p_inv(2 * dwells, (1 - pfa)^(1 / (N * bins)))
    from scipy.special import gammaincinv
    th = 2.0 * float(gammaincinv(2.0, (1.0 - 0.001) ** (1.0 / (ACQ_N * bins))))
    detected = sorted(int(p) for p in range(1, ACQ_PRNS + 1) if res[p - 1]["test_statistics"] > th)
    # e2e: host samples in, host results out, per sweep.  Two acquisition objects (= two channels' acquisition blocks)
    # alternate through the asynchronous entry points, so the next sweep is queued while the previous one's results
    # travel back; every sweep's H2D and D2H are inside the timed region.  The synchronous one-at-a-time figure is kept.
    t0 = time.perf_counter()
    for _ in range(steps):
        r2 = acq.search(iq, slots)
    dt_sync = (time.perf_counter() - t0) / steps
    acq_b = capi.PcpsAcquisition(eng, fs_in=ACQ_FS, samples_per_ms=float(ACQ_N), samples_per_chip=24, doppler_max=ACQ_DMAX,
                                 doppler_step=ACQ_DSTEP, n_code_slots=ACQ_PRNS)
    for p in range(1, ACQ_PRNS + 1):
        acq_b.set_local_code(p - 1, gps_ca_code_complex_sampled(p, ACQ_FS))
    objs = [acq, acq_b]
    for o in objs:
        o.search(iq, slots)
    t0 = time.perf_counter()
    objs[0].search_submit(iq, slots)
    for k in range(1, steps):
        objs[k % 2].search_submit(iq, slots)
        r2 = objs[(k - 1) % 2].search_wait()
    r2 = objs[(steps - 1) % 2].search_wait()
    dt = (time.perf_counter() - t0) / steps
    acq_b.close()
    if dist is not None:
        tdt = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(tdt, op=dist.ReduceOp.MAX)
        dt = float(tdt.item())
    peak, peak_src = measured_peak_gbs()
    out = {"metric": "acquisitions/s over Doppler grid", "unit": "acquisitions/s",
           "config": {"workload": f"C4: GPS L1 C/A PCPS, {ACQ_PRNS} PRNs x {bins} Doppler bins x N={ACQ_N} (25 Msps, 1 ms), CFAR statistic, "
                                  "forward FFTs shared by all PRNs"},
           "value": ACQ_PRNS / (ms * 1e-3), "ms_per_sweep": ms, "rows_per_s": rows / (ms * 1e-3),
           "e2e": {"value": ACQ_PRNS / dt, "unit": "acquisitions/s", "h2d_bytes_per_step": ACQ_N * 8,
                   "d2h_bytes_per_step": ACQ_PRNS * capi.ACQ_RESULT_DTYPE.itemsize, "ms_per_sweep": dt * 1e3,
                   "synchronous_one_object": {"value": ACQ_PRNS / dt_sync, "ms_per_sweep": dt_sync * 1e3},
                   "path": "b200_acq_search_submit / _wait alternating over two acquisition objects"},
           "gpu_launches_per_sweep": launches / steps, "cuda_graph": graph is not None,
           "roofline": {"bound": "hbm", "kernel": "acq_corr_kernel", "achieved": abytes / (ms * 1e-3) / 1e9, "peak": peak,
                        "unit": "GB/s", "frac": abytes / (ms * 1e-3) / 1e9 / peak, "traffic": ncu_acq_traffic_bytes(),
                        "algorithmic_bytes_per_sweep": abytes, "algorithmic_gflop_per_sweep": aflops / 1e9,
                        "achieved_tflops": aflops / (ms * 1e-3) / 1e12, "peak_source": peak_src,
                        "note": "16N bytes per (PRN,bin) row (SURVEY 8d); operands are L2-resident, the kernel is "
                                "shared-memory/FP32 bound, see DESIGN.md"},
           "detected_prns": detected, "present_prns": present,
           "e2e_matches_dev": bool(np.array_equal(r2["index_time"], res_local["index_time"])),
           "n_gpus": world, "sharding": ("PRNs round-robin over ranks; per sweep one CUDA-graph launch per rank and one all-gather of 16-byte peak records "
                        "(b200_acq_sweep_best_dev)") if world > 1 else "single GPU"}
    if with_cpu:
        with whole_host():
            out["cpu_baseline"] = cpu_baseline_acq(iq)
    acq.close()
    if world == 1:
        # a front end at 16.368 Msps: N = 16 368 = 2^4 * 3 * 11 * 31 goes through chirp-z (M = 32 768) on the same kernels
        try:
            fs2, n2, dmax2 = 16_368_000, 16368, 5000
            bins2 = int(np.ceil(2 * dmax2 / ACQ_DSTEP)) + 1
            cz = capi.PcpsAcquisition(eng, fs_in=fs2, samples_per_ms=float(n2), samples_per_chip=16, doppler_max=dmax2, doppler_step=ACQ_DSTEP,
                                      n_code_slots=ACQ_PRNS)
            for p in range(1, ACQ_PRNS + 1):
                cz.set_local_code(p - 1, gps_ca_code_complex_sampled(p, fs2))
            slots_all = np.arange(ACQ_PRNS, dtype=np.uint32)
            x2 = torch.randn((n2, 2), device=dev, dtype=torch.float32)
            r2d = torch.zeros(ACQ_PRNS * capi.ACQ_RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
            for _ in range(3):
                cz.search_dev(x2.data_ptr(), slots_all, r2d.data_ptr())
            torch.cuda.synchronize()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for _ in range(10):
                cz.search_dev(x2.data_ptr(), slots_all, r2d.data_ptr())
            c1.record()
            torch.cuda.synchronize()
            msz = c0.elapsed_time(c1) / 10
            out["chirp_z_16368"] = {"workload": f"{ACQ_PRNS} PRNs x {cz.conf.num_doppler_bins} Doppler bins x N=16368 (16.368 Msps, 1 ms), chirp-z with M=32768",
                                    "ms_per_sweep": msz, "value": ACQ_PRNS / (msz * 1e-3), "unit": "acquisitions/s"}
            cz.close()
        except Exception as ex:
            out["chirp_z_16368"] = {"error": repr(ex)}
    return out


def bench_closed_loop(capi, eng, svs, cids, n_epochs=990, repeats=3, replicas=1, with_launch_mode=True):
    """Free-running DLL/PLL on the device (SURVEY 8f N1): the 32 channels of the C2 band tracked in closed loop,
    correlator launch and loop-update launch alternating on the engine stream, no host round trip per epoch.
    Timed with the engine's CUDA events around b200_trk_loop_run (includes the D2H of the dump records)."""
    from gnss_synth import CA_RATE, GPS_L1_FREQ
    conf = capi.TrkLoopConf()
    conf.fs_in, conf.code_chip_rate, conf.signal_carrier_freq, conf.code_period, conf.carrier_lock_th = FS, CA_RATE, GPS_L1_FREQ, 1e-3, 0.7
    conf.code_length_chips, conf.vector_length, conf.pull_in_time_s, conf.bit_synchronization_time_limit_s = 1023, EPOCH, 1, 0xFFFFFFFF
    conf.code_samples_per_chip, conf.pll_filter_order, conf.dll_filter_order = 1, 3, 2
    conf.cn0_samples, conf.cn0_min, conf.max_code_lock_fail, conf.max_carrier_lock_fail = 20, 25, 50, 5000
    conf.cn0_smoother_samples, conf.carrier_lock_test_smoother_samples = 200, 25
    conf.veml, conf.cloop, conf.carrier_aiding, conf.enable_fll_pull_in, conf.enable_fll_steady_state = 0, 1, 1, 0, 0
    conf.pll_bw_hz, conf.dll_bw_hz, conf.fll_bw_hz, conf.early_late_space_chips = 35.0, 2.0, 35.0, 0.5
    conf.slope, conf.y_intercept, conf.cn0_smoother_alpha, conf.carrier_lock_test_smoother_alpha = 1.0, 1.0, 0.002, 0.002
    # replicas > 1: several independent loops per satellite (own state, different acquisition Doppler errors) to
    # show how closed-loop throughput scales with the number of channels resident on the GPU
    base = getattr(eng, "_n_loops", 0)
    svs = [dict(sv, acq_err=20.0 - 7.0 * r) for r in range(replicas) for sv in svs]
    cids = list(cids) * replicas
    lids = []
    for sv, cid in zip(svs, cids):
        conf.prn = sv["prn"]
        lids.append(eng.loop_create(cid, conf))
    def run_mode(mode):
        eng.loop_set_mode(mode)
        best = None
        for _ in range(repeats):
            for sv, lid in zip(svs, lids):
                rate = CA_RATE * (1.0 + sv["doppler"] / GPS_L1_FREQ)
                delay = ((1023.0 - sv["code_phase_chips"]) % 1023.0) / (rate / FS)      # sample of the first PRN start
                eng.loop_start(lid, delay, sv["doppler"] + sv["acq_err"], 0, 0)         # acquisition-grade Doppler
            l0 = eng.launch_count()
            eng.timer_start()
            rec, cnt = eng.loop_run(n_epochs)
            ms = eng.timer_stop_ms()
            launches = eng.launch_count() - l0
            if best is None or ms < best[0]:
                best = (ms, rec, cnt, launches)
        return best

    per_launch = run_mode(2) if with_launch_mode else None
    best = run_mode(0)
    ms, rec, cnt, launches = best
    rec, cnt = rec[base:], cnt[base:]          # loops created by earlier calls on this engine are in standby
    tail = rec[:, n_epochs - 200:n_epochs - 5]
    dopp_err = np.array([abs(float(np.mean(tail[i]["carrier_doppler_hz"])) - svs[i]["doppler"]) for i in range(len(svs))])
    locked = int(np.sum((dopp_err < 3.0) & (cnt >= n_epochs - 2)))
    ch_samples = float(np.sum(cnt)) * EPOCH
    return {"workload": f"C2 band, {len(svs)} channels, closed loop on the device for {n_epochs} epochs (1 ms each)",
            "ms": ms, "epochs_logged": int(np.sum(cnt)), "value": ch_samples / (ms * 1e-3) / 1e6, "unit": UNIT,
            "realtime_factor": n_epochs * 1e-3 / (ms * 1e-3), "us_per_epoch": ms * 1e3 / n_epochs,
            "gpu_launches": int(launches), "channels_locked": locked, "max_doppler_error_hz": float(np.max(dopp_err)),
            "mean_cn0_dbhz": float(np.mean(tail["CN0_SNV_dB_Hz"])),
            "per_epoch_launch_mode": ({"ms": per_launch[0], "gpu_launches": int(per_launch[3]), "us_per_epoch": per_launch[0] * 1e3 / n_epochs}
                                      if per_launch else None),
            "note": "persistent kernel: one CTA per channel free-runs prepare -> correlate -> discriminators, loop filters, NCO, "
                    "lock detectors, dump record, epoch after epoch with no launch and no host round trip; epoch k+1 depends on "
                    "epoch k, so each channel is latency-bound and throughput scales with the channel count up to the number of "
                    "resident CTAs; per_epoch_launch_mode = the same arithmetic as 2 launches per epoch"}


# ---- CPU baseline (the reference's own SIMD path, timed like its own harness) --------------------
def usable_cpus():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_baseline(budget_s=12.0, sweep=False, threads=None):
    """The reference's Cpu_Multicorrelator_Real_Codes (u_avx kernels) compiled in place: one correlator per host thread,
    threads PINNED round robin over the process's CPUs and started together (oracle/ref_engine.cc ref_mc_bench_pinned),
    shaped like cpu_multicorrelator_real_codes_test.cc:41-62,135-169.  sweep=True adds the T in {1, nproc/2, nproc} x
    length {2048, 4096, 8192 (the reference's), 25000, 200000 (ours)} table BASELINE.md promises, per-thread figures included."""
    import oracle
    cores = usable_cpus()
    if oracle.ref is not None:
        kind = "reference"
        oracle.ref.select_arch("u_avx")   # GNU Radio buffers are unaligned: VOLK dispatches to u_ variants

        def run(iters, threads=cores, n=EPOCH, taps=TAPS, L=1023):
            return oracle.ref.mc_bench(threads, n, taps, L, iters, 8, False, pin=True)
    else:
        kind = "port"
        rng = np.random.default_rng(0)
        iq = (rng.standard_normal(EPOCH * 8) + 1j * rng.standard_normal(EPOCH * 8)).astype(np.complex64)
        code = oracle.port.gps_ca_code(1)

        def run(iters, threads=cores, n=EPOCH, taps=TAPS, L=1023):
            params = np.tile(np.array([[0.4, 0.001, 0.3, 1023.0 / n]], np.float32), (iters * threads, 1))
            t0 = time.perf_counter()
            oracle.port.multicorrelator_batch(1, threads, np.tile(iq, max(1, n // EPOCH + 1)), 0, code, SHIFTS, params, n)
            return time.perf_counter() - t0
    # Hyper-threaded hosts: on the 2 x 32-core box of this pool 128 pinned threads deliver 3.6 Gsamples/s and 64 deliver 13.7
    # (AVX units and L2 shared by sibling threads; round 1's 2 919 vs 15 675 Msamples/s on two boxes was this).  The arm
    # uses the thread count that is FASTEST among {nproc, nproc/2, nproc/4} and says which.
    best = None
    probe = 2000   # epochs per thread: >= 0.15 s per probe, long enough for sibling-thread contention to show
    for T in (sorted({cores, max(1, cores // 2), max(1, cores // 4)}, reverse=True) if threads is None else [threads]):
        t0 = run(probe, threads=T)
        rate = T * probe * EPOCH / t0
        if best is None or rate > best[0]:
            best = (rate, T, t0)
    threads = best[1]
    t = best[2]
    iters = int(max(20, min(400000, probe * budget_s / max(t, 1e-6))))
    t = run(iters, threads=threads)
    samples = threads * iters * EPOCH
    out = {"value": samples / t / 1e6, "unit": UNIT, "cores": threads, "host_cpus": cores, "kind": kind, "per_thread": samples / t / 1e6 / threads,
           "pinned": True,
           "sample": f"{threads} pinned threads (fastest of nproc={cores}, /2, /4) x {iters} epochs of {EPOCH} samples x {TAPS} taps, L=1023 "
                     f"({samples / 1e6:.0f} M channel-samples, {t:.1f} s); "
                     + ("reference Cpu_Multicorrelator_Real_Codes with volk_gnsssdr u_avx kernels "
                        "(harness shaped like cpu_multicorrelator_real_codes_test.cc:41-62,135-169)"
                        if kind == "reference" else "C port of the a_avx/u_avx arithmetic")}
    if sweep:
        table = []
        for T in sorted({1, max(1, cores // 2), cores}):
            for n, taps, L in ((2048, 3, 1023), (4096, 3, 1023), (8192, 3, 1023), (25000, 3, 1023), (200000, 5, 8184)):
                it = max(4, int(4.0e6 / n))
                dt = run(it, threads=T, n=n, taps=taps, L=L)
                table.append({"threads": T, "length": n, "taps": taps, "msamples_per_s": T * it * n / dt / 1e6,
                              "per_thread": it * n / dt / 1e6})
        out["sweep"] = table
    return out, t


def cpu_baseline_acq(iq=None, budget_s=15.0):
    """Acquisition on the host: the reference's OWN chain compiled in place - GpsL1CaPcpsAcquisition adapter ->
    pcps_acquisition block (general_work buffering, doppler_grid, CFAR statistic) - driven by the single-block scheduler of
    oracle/shim, one channel per pinned host thread, threads over PRNs (oracle/blocks_harness.cc itf_acq_bench).  The
    FFT behind gr::fft is our float32 mixed-radix Stockham transform (oracle/shim/gnuradio/fft/fft.h; FFTW is not
    installable here).  Falls back to the numpy restatement where the block library is absent."""
    from gnss_synth import make_iq, gps_ca_code
    cores = usable_cpus()
    if iq is None:
        iq = make_iq({2: gps_ca_code(2)}, float(ACQ_FS), 2 * ACQ_N + 64, [dict(prn=2, doppler=1234.0, code_phase_chips=100.0, cn0=45.0)], seed=4)
    try:
        import blocks_itf as bi
        lib = bi.ref_lib()
    except Exception:
        lib = None
    if lib is not None:
        conf = {"GNSS-SDR.internal_fs_sps": ACQ_FS, "Acquisition_1C.item_type": "gr_complex", "Acquisition_1C.doppler_max": ACQ_DMAX,
                "Acquisition_1C.doppler_step": ACQ_DSTEP, "Acquisition_1C.pfa": 0.001, "Acquisition_1C.blocking": True}
        feed = np.ascontiguousarray(np.resize(iq, 2 * ACQ_N + 64))
        dt1, _ = bi.acq_bench(lib, conf, "GPS_L1_CA_PCPS_Acquisition", feed, 1, 2)
        per_thread = 2 / dt1
        # each channel streams its own 16 MB wipe-off grid and 8 MB magnitude grid: the search is memory-bound long before all
        # hardware threads are busy - use the fastest thread count of {nproc, /2, /4, /8}
        best = None
        for T in sorted({cores, max(1, cores // 2), max(1, cores // 4), max(1, cores // 8)}, reverse=True):
            dtp, _ = bi.acq_bench(lib, conf, "GPS_L1_CA_PCPS_Acquisition", feed, T, 2)
            if best is None or T * 2 / dtp > best[0]:
                best = (T * 2 / dtp, T)
        threads = best[1]
        k = int(max(2, min(64, budget_s * best[0] / threads)))
        dt, pos = bi.acq_bench(lib, conf, "GPS_L1_CA_PCPS_Acquisition", feed, threads, k)
        bins = int(np.ceil(2 * ACQ_DMAX / ACQ_DSTEP))
        cores_used = threads
        return {"value": threads * k / dt, "unit": "acquisitions/s", "cores": cores_used, "host_cpus": cores, "kind": "reference",
                "per_thread_alone": per_thread, "per_thread_loaded": k / dt, "pinned": True,
                "sample": f"{threads} pinned threads (fastest of nproc={cores}, /2, /4, /8) x {k} searches ({bins} Doppler bins x N={ACQ_N}) through the reference's own "
                          f"GpsL1CaPcpsAcquisition adapter + pcps_acquisition block compiled in place ({dt:.1f} s); FFT = float32 "
                          "mixed-radix Stockham shim behind gr::fft (FFTW / GNU Radio not installable)"}
    import oracle
    from oracle.acq_np import AcqConf, PcpsAcquisitionOracle
    conf = AcqConf(fs_in=ACQ_FS, samples_per_ms=float(ACQ_N), samples_per_code=float(ACQ_N), samples_per_chip=24,
                   doppler_max=ACQ_DMAX, doppler_step=ACQ_DSTEP, pfa=0.001)
    o = PcpsAcquisitionOracle(conf, workers=cores)
    o.set_local_code(oracle.port.gps_ca_code_complex_sampled(2, ACQ_FS))
    o.acquisition_core(iq[:ACQ_N])
    t0 = time.perf_counter()
    for _ in range(2):
        o.num_noncoherent_integrations_counter = 0
        o.acquisition_core(iq[:ACQ_N])
    dt = time.perf_counter() - t0
    return {"value": 2 / dt, "unit": "acquisitions/s", "cores": cores, "kind": "port",
            "sample": f"2 PRN searches x {conf.num_doppler_bins} bins x N={ACQ_N}; numpy restatement of pcps_acquisition.cc with scipy.fft"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    vals, times = [], []
    threads = None
    for k in range(args.warmup + args.steps):
        # the thread count is chosen once (first step); whole arm ~1-2 min for any K
        cb, t = cpu_baseline(budget_s=max(0.15, 60.0 / max(1, args.warmup + args.steps)), threads=threads)
        threads = cb["cores"]
        if k >= args.warmup:
            vals.append(cb["value"])
            times.append(t)
    cb["value"] = float(np.mean(vals))
    cb["per_thread"] = cb["value"] / cb["cores"]
    try:
        sw, _ = cpu_baseline(budget_s=0.5, sweep=True)
        cb["sweep"] = sw.get("sweep")
    except Exception as ex:
        cb["sweep"] = {"error": repr(ex)}
    try:
        acq_ref = cpu_baseline_acq()
    except Exception as ex:
        acq_ref = {"error": repr(ex)}
    line = {"metric": METRIC, "value": cb["value"], "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "acq": acq_ref,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(times) * 1e3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args.gpus), "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-acq", action="store_true")
    ap.add_argument("--no-loop", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the sustained leg, the other BASELINE configs and the coalescer leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the taps of the last timed step (float32 [items, taps, re/im], items epoch-major) to DIR/trk_taps.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import gnss_sdr_b200.capi as capi   # raises if libb200gnss.so is missing: no fallback

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL writes its NCCL_DEBUG lines (e.g. "NCCL version ...") to stdout unless told otherwise; stdout is for the JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa(torch, local_rank)   # before any pinned allocation (first touch)

    from gnss_synth import gps_ca_code   # synthetic-input code tables; oracle/ is only touched by the CPU-baseline legs
    codes = {p: gps_ca_code(p) for p in range(1, N_CH + 1)}
    # one receiver: every rank sees the SAME band (the 32 satellites of C2); rank r owns channels 32 r .. 32 r + 31
    svs = svs_for_rank(0)
    n_iq = EPOCH * N_EPOCHS
    iq_dev = synth_iq_device(torch, codes, svs, n_iq + 16, SEED, dev)

    # a dedicated (non-default) torch stream is made current and handed to the engine, so that the
    # torch.cuda.Event timings below are recorded on the very stream the kernels are launched on
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0
    eng = capi.Engine(local_rank, stream)
    # band 0: attached device-resident IQ (value); band 1: ring fed from pinned host memory (e2e)
    eng.iq_attach_dev(0, iq_dev.data_ptr(), n_iq + 16, 0)
    cids = []
    for sv in svs:
        cid = eng.channel_create(0, TAPS)
        eng.channel_set_code(cid, codes[sv["prn"]], SHIFTS)
        cids.append(cid)
    items = build_items(capi, svs, cids, 0)
    n_items = items.size
    items_dev = torch.from_numpy(items.view(np.uint8)).to(dev)
    out_dev = torch.zeros((n_items, TAPS, 2), dtype=torch.float32, device=dev)
    ch_samples_step = N_CH * EPOCH * N_EPOCHS

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step_dev():
        eng.trk_batch_dev(items_dev.data_ptr(), n_items, out_dev.data_ptr(), TAPS, 1)

    # ---- value: inputs resident in HBM -----------------------------------------------------------
    for _ in range(args.warmup):
        step_dev()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    ev[0].record()
    for k in range(args.steps):
        step_dev()
        ev[k + 1].record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "trk_taps.npy"), out_dev.cpu().numpy())
    total_ms = ev[0].elapsed_time(ev[-1])
    launches = eng.launch_count() - l0
    # cross-check with the library's own CUDA-event timer on the engine stream (one extra step)
    eng.timer_start()
    step_dev()
    check_ms = eng.timer_stop_ms()
    per_launch_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    ms_per_step = total_ms_max / args.steps
    value = world * ch_samples_step / (ms_per_step * 1e-3) / 1e6

    # sanity: the prompt taps must show the signal (guards against timing a broken kernel)
    taps = out_dev[:, :, 0].cpu().numpy() + 1j * out_dev[:, :, 1].cpu().numpy()
    prompt_snr = float(np.mean(np.abs(taps[:, 1])) / np.sqrt(EPOCH * 2.0))

    # ---- e2e: host buffers through the public C ABI, copies inside the timed region --------------
    e2e = None
    if not args.no_e2e and world > 1:
        # ---- one receiver on N GPUs: the band crosses PCIe ONCE (rank 0, b200_iq_refill from pinned memory into a device
        # buffer), fans out to the peers with one NCCL broadcast over NVLink, every rank correlates its own 32 channels and
        # returns its taps to its host.  Two band buffers: step k+1's copy + broadcast overlap step k's correlation.
        host_iq = None
        if rank == 0:
            host_iq = torch.empty((n_iq, 2), dtype=torch.float32, pin_memory=True)
            host_iq.copy_(iq_dev[:n_iq])
        bands = [torch.zeros((n_iq + 16, 2), dtype=torch.float32, device=dev) for _ in range(2)]
        items_b, outs_b, outs_host, done_ev = [], [], [], []
        for b in range(2):
            eng.iq_attach_dev(2 + b, bands[b].data_ptr(), n_iq + 16, 0)
            cb_ids = []
            for sv in svs:
                cid = eng.channel_create(2 + b, TAPS)
                eng.channel_set_code(cid, codes[sv["prn"]], SHIFTS)
                cb_ids.append(cid)
            items_b.append(torch.from_numpy(build_items(capi, svs, cb_ids, 0).view(np.uint8)).to(dev))
            outs_b.append(torch.zeros((n_items, TAPS, 2), dtype=torch.float32, device=dev))
            outs_host.append(torch.empty((n_items, TAPS, 2), dtype=torch.float32, pin_memory=True))
            done_ev.append(torch.cuda.Event())
        torch.cuda.synchronize()

        def run_one_receiver(n_steps):
            for k in range(n_steps):
                b = k % 2
                if k >= 2:
                    done_ev[b].synchronize()          # step k-2's taps are on the host: its band buffer is free again
                if rank == 0:
                    eng.iq_refill_ptr(2 + b, host_iq.data_ptr(), n_iq, 0)   # C ABI: pinned host -> device, copy stream, engine stream waits
                dist.broadcast(bands[b], src=0)        # NVLink fan-out, ordered after the refill on the engine stream
                eng.trk_batch_dev(items_b[b].data_ptr(), n_items, outs_b[b].data_ptr(), TAPS, 1)
                outs_host[b].copy_(outs_b[b], non_blocking=True)
                done_ev[b].record()
            torch.cuda.synchronize()
            return outs_host[(n_steps - 1) % 2]

        run_one_receiver(max(3, args.warmup))
        barrier()
        t0 = time.perf_counter()
        res_t = run_one_receiver(args.steps)
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        res = res_t.numpy()[:, :, 0] + 1j * res_t.numpy()[:, :, 1]
        e2e = {"value": world * ch_samples_step * args.steps / dt / 1e6, "unit": UNIT,
               "h2d_bytes_per_step": int(n_iq * 8), "d2h_bytes_per_step": int(world * n_items * TAPS * 8),
               "nvlink_broadcast_bytes_per_step": int((n_iq + 16) * 8), "ms_per_step": dt / args.steps * 1e3,
               "max_rel_diff_vs_value_run": float(np.max(np.abs(res - taps)) / np.max(np.abs(taps))),
               "numa": numa,
               "path": "rank 0: b200_iq_refill (pinned host -> device, once per step for the whole job); all ranks: NCCL broadcast of the "
                       "band over NVLink, b200_trk_batch_dev on the rank's 32 channels, taps D2H to pinned host memory; two band "
                       "buffers so that step k+1's copy and broadcast overlap step k's correlation"}
    elif not args.no_e2e:
        host_iq = torch.empty((n_iq, 2), dtype=torch.float32, pin_memory=True)
        host_iq.copy_(iq_dev[:n_iq])
        torch.cuda.synchronize()
        eng.iq_create(1, 2 * n_iq)   # two steps of samples in flight (software pipelining below)
        cids1 = []
        for sv in svs:
            cid = eng.channel_create(1, TAPS)
            eng.channel_set_code(cid, codes[sv["prn"]], SHIFTS)
            cids1.append(cid)
        items1 = build_items(capi, svs, cids1, 0)
        base_idx = items1["sample_index"].copy()

        E2E_CHUNKS = 8    # pushes and correlation batches overlap (copy engine vs SMs)
        ep_per_chunk = N_EPOCHS // E2E_CHUNKS
        items1_v = items1.reshape(N_EPOCHS, N_CH)

        def enqueue_e2e():
            """All of one step's host -> device copies and launches, asynchronously; returns the tickets."""
            tickets = []
            first0 = None
            for c in range(E2E_CHUNKS):
                a, b = c * ep_per_chunk, (c + 1) * ep_per_chunk if c < E2E_CHUNKS - 1 else N_EPOCHS
                # H2D of this chunk's samples from pinned host memory (async on the copy stream)
                first = eng.iq_push_ptr(1, host_iq.data_ptr() + a * EPOCH * 8, (b - a) * EPOCH)
                if first0 is None:
                    first0 = first
                    items1["sample_index"] = base_idx + np.uint64(first0)
                # items H2D, one launch (ordered after the push), taps D2H -- all asynchronous
                tickets.append(eng.trk_submit(items1_v[a:b].reshape(-1), TAPS))
            return tickets

        def collect_e2e(tickets):
            return np.concatenate([eng.trk_wait(t) for t in tickets], axis=0)

        def run_e2e(n_steps):
            """Steps are software-pipelined as in a running receiver: step k+1's copies are queued behind step k's
            while step k's taps are read back, so the copy engine never waits for the host.  Every step's H2D and
            D2H still happen inside the timed region."""
            prev, out = None, None
            for _ in range(n_steps):
                cur = enqueue_e2e()
                if prev is not None:
                    out = collect_e2e(prev)
                prev = cur
            return collect_e2e(prev)

        res = run_e2e(args.warmup)
        barrier()
        t0 = time.perf_counter()
        res = run_e2e(args.steps)
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        e2e = {"value": world * ch_samples_step * args.steps / dt / 1e6, "unit": UNIT,
               "h2d_bytes_per_step": int(n_iq * 8 + items1.nbytes), "d2h_bytes_per_step": int(n_items * TAPS * 8),
               "ms_per_step": dt / args.steps * 1e3,
               "path": f"{E2E_CHUNKS} x [b200_iq_push (pinned host -> device ring) + b200_trk_submit (items H2D, 1 launch, taps D2H)] "
                       "then b200_trk_wait: copies overlap correlation, and step k+1 is queued before step k's taps are read"}
        # e2e result must agree with the device-resident run
        e2e["max_rel_diff_vs_value_run"] = float(np.max(np.abs(res - taps)) / np.max(np.abs(taps)))
        # what the link alone does: the same pinned 200 MB buffer copied host -> device with nothing else going on
        # (the e2e step cannot be faster than this; it is the PCIe roofline of the cf32 path on this box)
        scratch = torch.empty((n_iq, 2), dtype=torch.float32, device=dev)
        for _ in range(2):
            scratch.copy_(host_iq, non_blocking=True)
        torch.cuda.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(5):
            scratch.copy_(host_iq, non_blocking=True)
        c1.record()
        torch.cuda.synchronize()
        copy_ms = c0.elapsed_time(c1) / 5
        e2e["h2d_copy_only"] = {"ms_per_step": copy_ms, "gb_per_s": n_iq * 8 / copy_ms / 1e6,
                                "value_if_copy_bound": world * ch_samples_step / (copy_ms * 1e-3) / 1e6}
        del scratch

        # ---- same e2e step with 16-bit / 8-bit front-end samples (SURVEY "next" row N3): the raw integers
        # cross PCIe and are converted on the device (b200_iq_push_i16/_i8) instead of on the host.
        for bits, scale in ((16, 256.0), (8, 16.0)):
            q = torch.clamp(torch.round(iq_dev[:n_iq] * scale), -(2 ** (bits - 1) - 1), 2 ** (bits - 1) - 1)
            host_q = torch.empty((n_iq, 2), dtype=torch.int16 if bits == 16 else torch.int8, pin_memory=True)
            host_q.copy_(q.to(host_q.dtype))
            torch.cuda.synchronize()
            del q
            bpc = bits // 8

            def enqueue_int():
                tickets = []
                first0 = None
                for c in range(E2E_CHUNKS):
                    a, b = c * ep_per_chunk, (c + 1) * ep_per_chunk if c < E2E_CHUNKS - 1 else N_EPOCHS
                    first = eng.iq_push_int(1, (host_q.data_ptr() + a * EPOCH * 2 * bpc, bits), (b - a) * EPOCH)
                    if first0 is None:
                        first0 = first
                        items1["sample_index"] = base_idx + np.uint64(first0)
                    tickets.append(eng.trk_submit(items1_v[a:b].reshape(-1), TAPS))
                return tickets

            def run_int(n_steps):
                prev = None
                for _ in range(n_steps):
                    cur = enqueue_int()
                    if prev is not None:
                        collect_e2e(prev)
                    prev = cur
                return collect_e2e(prev)

            ri = run_int(3)
            barrier()
            t0 = time.perf_counter()
            ri = run_int(args.steps)
            barrier()
            dti = time.perf_counter() - t0
            tti = torch.tensor([dti], dtype=torch.float64, device=dev)
            if dist is not None:
                dist.all_reduce(tti, op=dist.ReduceOp.MAX)
            dti = float(tti.item())
            e2e[f"int{bits}_front_end"] = {"value": world * ch_samples_step * args.steps / dti / 1e6, "unit": UNIT,
                                           "h2d_bytes_per_step": int(n_iq * 2 * bpc + items1.nbytes),
                                           "d2h_bytes_per_step": int(n_items * TAPS * 8), "ms_per_step": dti / args.steps * 1e3,
                                           "prompt_over_noise": float(np.mean(np.abs(ri[:, 1])) / scale / np.sqrt(EPOCH * 2.0)),
                                           "path": f"b200_iq_push_i{bits} (raw {bits}-bit I/Q over PCIe, converted on the device)"}
            del host_q

    acq = None
    if not args.no_acq:
        try:
            acq = bench_acq(torch, capi, eng, dev, max(5, min(args.steps, 50)), 3, with_cpu=(world == 1 and not args.no_cpu_baseline),
                            dist=dist, rank=rank, world=world)
        except Exception as ex:  # the headline metric must still be reported
            if world > 1:
                raise
            acq = {"error": repr(ex)}

    closed = None
    if not args.no_loop and rank == 0:
        try:
            closed = bench_closed_loop(capi, eng, svs, cids)
            closed["x8_channels"] = bench_closed_loop(capi, eng, svs, cids, replicas=8, with_launch_mode=False)
        except Exception as ex:
            closed = {"error": repr(ex)}

    # ---- sustained leg: the same step back to back for >= 2 s (the 20-step timed region above is 17 ms) -------------
    sustained = None
    if not args.no_extra:
        n_sus = int(max(args.steps, 2.2 / max(ms_per_step * 1e-3, 1e-6)))
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        sampler2 = ClockSampler(local_rank)
        if rank == 0:
            sampler2.start()
        s0.record()
        for _ in range(n_sus):
            step_dev()
        s1.record()
        barrier()
        sus_ms = s0.elapsed_time(s1)
        tsus = torch.tensor([sus_ms], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(tsus, op=dist.ReduceOp.MAX)
        sus_ms = float(tsus.item())
        sustained = {"steps": n_sus, "seconds": sus_ms * 1e-3, "ms_per_step": sus_ms / n_sus,
                     "value": world * ch_samples_step * n_sus / (sus_ms * 1e-3) / 1e6, "unit": UNIT,
                     "clocks": sampler2.stop() if rank == 0 else None}

    # ---- C5 on N GPUs: every rank runs its 32-channel share (12 GPS L1 + 12 Galileo E1 + 8 GPS L5 at 50 Msps) at the same time;
    # with N = 8 that is BASELINE configs[4] (256 channels, three signals) ------------------------------------------------------
    c5_multi = None
    if not args.no_extra and world > 1:
        try:
            barrier()
            share = other_configs(torch, capi, dev, tstream, steps=10, only=["C5_per_gpu_share"])["C5_per_gpu_share"]
            tms = torch.tensor([share.get("ms_per_step", float("nan"))], dtype=torch.float64, device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms_max = float(tms.item())
            c5_multi = {"workload": f"C5 share x {world} GPUs = {32 * world} channels at 50 Msps x 1 s, three signals, ranks concurrent, no collective",
                        "ms_per_step_max_over_ranks": ms_max,
                        "value": world * share["channel_samples_per_step"] / (ms_max * 1e-3) / 1e6, "unit": UNIT}
        except Exception as ex:
            c5_multi = {"error": repr(ex)}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    extra = None
    coalesced = None
    if not args.no_extra and world == 1:
        extra = other_configs(torch, capi, dev, tstream, steps=max(5, min(args.steps, 20)))
        coalesced = coalesced_class_interface()

    # ---- roofline of the dominant kernel -------------------------------------------------------------------------
    # `achieved` follows the contract: ALGORITHMIC bytes (8 B per channel-sample, SURVEY 8d) per launch / mean launch time of the
    # timed region.  On C2 the 32 channels share one IQ stream, so those bytes do not cross HBM 32 times (`traffic` = what
    # ncu saw) and frac can exceed 1: it is NOT the kernel's distance from a limit.  Two companions say what is:
    #   hbm_true   the same arithmetic with every (channel, epoch) reading its own samples: 8 B per channel-sample really from HBM;
    #   fp32_issue what ncu names as the limiter of the C2 launch (instruction issue / FMA pipe), from profiles/.
    peak, peak_src = measured_peak_gbs()
    launch_ms = float(np.mean(per_launch_ms))
    achieved = ch_samples_step * ALGO_BYTES_PER_CHANNEL_SAMPLE / (launch_ms * 1e-3) / 1e9
    hbm_true = None
    if extra and isinstance(extra.get("C2_distinct_iq"), dict) and "ms_per_step" in extra["C2_distinct_iq"]:
        d = extra["C2_distinct_iq"]
        hbm_true = {"workload": d["workload"], "achieved": d["algorithmic_GBps"], "peak": peak, "unit": "GB/s", "frac": d["algorithmic_GBps"] / peak,
                    "ms_per_launch": d["ms_per_step"], "value": d["value"],
                    "kernel": "trk_correlate_kernel<3> (per-item)",
                    "note": "band = channels x samples: no sharing between channels, DRAM traffic == algorithmic bytes (+ items/taps)"}
    roofline = {"bound": "hbm", "kernel": "trk_shared_kernel<3>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": ncu_traffic_bytes(),
                "algorithmic_bytes_per_launch": ch_samples_step * ALGO_BYTES_PER_CHANNEL_SAMPLE,
                "launch_ms": launch_ms, "peak_source": peak_src, "limiter": ncu_limiter(), "hbm_true": hbm_true,
                "note": "achieved/frac = algorithmic bytes (8 B per channel-sample, SURVEY 8d) over the launch time, as the contract defines "
                        "them; the 32 channels of C2 share one IQ stream, so real DRAM traffic is `traffic` (the 200 MB stream once) and "
                        "frac > 1 is possible - see `hbm_true` for the fraction with distinct samples per channel-epoch and `limiter` for "
                        "what ncu names as the bound of the C2 launch (FP32 instruction issue / FMA pipe)"}
    cb = None
    if not args.no_cpu_baseline and world == 1:
        with whole_host():
            cb, _ = cpu_baseline(sweep=True)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config_dict(world), "clocks": clocks,
            "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cb,
            "stream_msps": value / N_CH, "prompt_over_noise": prompt_snr, "engine_timer_check_ms": check_ms,
            "acq": acq, "closed_loop": closed, "sustained": sustained, "other_configs": extra, "c5_multi_gpu": c5_multi,
            "coalesced_class_interface": coalesced, "numa": numa}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
