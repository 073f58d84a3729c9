#!/usr/bin/env python3
"""bench.py -- headline benchmark of the P25 baseband hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload (BASELINE.json configs[1], unchanged since round 1 so that rounds stay comparable): 1,024 independent
synthetic P25 control-channel IQ streams per GPU, 2.4 MS/s cf32, 150 ms = 360,000 samples per stream per step, /50 to
48 kHz, C4FM-demodulated, frame-synchronised and TSBK-decoded.  One step is one pass of the hot path (p25cu_process:
ddc_fm kernel + decode walker) over that batch, 2.95 GB of input, far larger than the 126 MB L2.  The signal is periodic
and phase-continuous, so consecutive steps are a continuous transmission and every step decodes real TSDUs.

  value      whole-job IQ Msamples/s with the input already resident in HBM: device time (CUDA events on the library's
             stream) of K x p25cu_process plus one final packed event drain.
  sustained  the same metric over a >= 2 s loop in the production call pattern: every step p25cu_process +
             p25cu_poll_start, events of step k-1 collected (p25cu_poll_packed) while step k runs.
  e2e        the same metric through the public call sequence with HOST (pinned) input, in the streaming pattern: each
             step = p25cu_process(host pointer) [H2D copy inside] + p25cu_poll_start, the events of step k-1 collected
             with p25cu_poll_packed [written to pinned host memory] while step k's copy and kernels run;
             frac_of_h2d_ceiling relates its input bytes/s to a plain pinned cudaMemcpyAsync measured in the same run
             on all ranks at once.
  roofline   dominant kernel of the workload: algorithmic bytes per launch / its own CUDA-event time inside the timed
             region, against MEASURED_PEAKS.json hbm_gbs; for the FP32-bound kernels also the measured FFMA2 peak.
  workloads  the other BASELINE configs through the same legs: cfg1 (one 2.4 MS/s stream), cfg2u8 (configs[1] in the
             reference's own 2 B/sample format), cfg3 (8 wideband captures through the channelizer), cfg4 (16,384 voice
             channels), cfg5 (65,536 u8 240 kS/s streams sharded over the N ranks: strong scaling).
  cpu_baseline  the oracle (C++ restatement of the reference chain, -march=native) on the same batch with every host core,
             with and without the per-sample correlator the reference is believed to run while locked.

The timed steps are checked: events of a deterministic sample of streams (first, last, CTA-boundary straddlers) over
the warm-up and every timed step must equal the oracle's, not just carry valid CRCs.

--dump-outputs DIR writes what the last timed step of the headline workload handed back (rank 0), so that two builds can
be compared output for output on the same seeded input:
  events_fields.npy   float64 [N][4]   stream, kind, sample, len of every event of that step, ordered by (stream, sample)
  events_payload.npy  float32 [N][60]  their payload bytes
  baseband.npy        float32 [k][n]   the step's 48 kHz baseband of the dumped streams (read back from the device)
  streams.npy         float64 [k]      the dumped streams: all of them, or a fixed seeded sample that keeps DIR under 64 MB

Multi-GPU: streams shard by rank with no collective on the data path (SURVEY.md section 8e).  torch.distributed (NCCL)
is used only for the barrier and the MAX of the per-rank device times.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True      # the tree may be read-only: nothing is cached beside the sources
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "spec")):
    if p not in sys.path:
        sys.path.insert(0, p)

STREAMS_PER_GPU = 1024
FS = 2_400_000
DECIM = 50
N_PER_STEP = 360_000          # 150 ms = two 360-dibit TSDUs per stream per step
N_BASE = 16                   # distinct seeded transmissions; streams are circular shifts of them
METRIC = "Msamples/s IQ demod+decode (real-time P25 channels = baseband samples/s / 48000)"
ALG_BYTES_PER_SAMPLE = 8.0 + 4.0 / DECIM     # SURVEY.md section 8(d), DESIGN.md section 4
EXTRA_DEFAULT = "cfg1,cfg2u8,cfg3,cfg4,cfg5"


class Workload:
    """One BASELINE.json configuration as a batch of device-resident input rows.

    cfg2   configs[1], the headline: 1,024 cf32 2.4 MS/s control channels per GPU (weak scaling)
    cfg2u8 the same batch as u8 IQ (the reference's sample format, 2 B/sample)
    cfg1   configs[0]: ONE 2.4 MS/s cf32 control channel, 6 s per call
    cfg3   configs[2]: 8 wideband 19.2 MS/s captures per GPU, 64 of 1,536 slots occupied, 150 ms per step
    cfg4   configs[3]: 16,384 voice traffic channels per GPU, u8 240 kS/s, 12 dB
    cfg5   configs[4]: 65,536 control channels, u8 240 kS/s, sharded over the ranks (strong scaling)"""

    def __init__(self, name: str, world: int):
        self.name, self.world = name, world
        self.rows_per_stream = 1
        self.kind, self.snr, self.periods = "control", 20.0, 1
        if name == "cfg5":
            assert 65536 % world == 0
            self.streams, self.fs, self.decim, self.fmt, self.scaling = 65536 // world, 240_000, 5, "u8", "strong"
            self.kernel = "w5i::p25_ddc5_imma_kernel (u8 /5: decimator on the integer tensor pipe, channel filter on FFMA2)"
            self.desc = ("configs[4]: 65,536 synthetic P25 control-channel streams in the reference's own format (u8 IQ, 240 kS/s, "
                         f"/5 -> 48 kHz), {self.streams} per GPU, 36000 samples (150 ms) per stream per step")
        elif name == "cfg4":
            self.streams, self.fs, self.decim, self.fmt, self.scaling = 16384, 240_000, 5, "u8", "weak"
            self.kind, self.snr = "traffic", 12.0
            self.kernel = "w5i::p25_ddc5_imma_kernel (u8 /5: decimator on the integer tensor pipe, channel filter on FFMA2)"
            self.desc = ("configs[3]: 16,384 voice traffic channels per GPU (HDU, LDU1/LDU2 with IMBE frames, TDULC) at 12 dB with "
                         "carrier offset, u8 IQ 240 kS/s, one superframe per stream per step")
        elif name == "cfg1":
            self.streams, self.fs, self.decim, self.fmt, self.scaling = 1, FS, DECIM, "cf32", "weak"
            self.periods = 40
            self.kernel = "fast::p25_ddc_fm_stream_kernel<cf32> (/50)"
            self.desc = "configs[0]: ONE synthetic 2.4 MS/s cf32 control channel (the reference's replay shape), 6 s per call, /50"
        elif name == "cfg3":
            self.streams, self.fs, self.decim, self.fmt, self.scaling = 8 * 1536, 19_200_000, 400, "cf32", "weak"
            self.kind, self.rows_per_stream = "wide", 1536
            self.kernel = "pfb::p25_pfbc_kernel (19.2 MS/s -> 1,536 x 48 kS/s baseband rows, one cluster kernel)"
            self.desc = ("configs[2]: 8 wideband 19.2 MS/s cf32 captures per GPU, 64 of the 1,536 12.5 kHz slots of each carrying a "
                         "control channel, 150 ms per step: polyphase channelizer, every channel demodulated and decoded")
        else:
            u8 = name == "cfg2u8"
            self.streams, self.fs, self.decim, self.fmt, self.scaling = STREAMS_PER_GPU, FS, DECIM, "u8" if u8 else "cf32", "weak"
            self.kernel = ("w50i::p25_ddc50_imma_kernel (u8 /50: both decimating stages as one 290-tap FIR on the integer tensor pipe)"
                           if u8 else "fast::p25_ddc_fm_stream_kernel<cf32> (/50)")
            self.desc = ("configs[1]: 1024 synthetic P25 control-channel IQ streams per GPU, " + ("u8" if u8 else "cf32") +
                         " 2.4 MS/s, 360000 samples (150 ms) per stream per step, /50 -> 48 kHz, C4FM demod + frame sync + NID/TSBK decode")
        self.bps = 2 if self.fmt == "u8" else 8
        self.rows = self.streams // self.rows_per_stream          # input rows per GPU (captures for cfg3)
        # event slots a stream needs per step, and the fewest events a healthy step of the whole rank yields
        self.slot_events = {"control": 8, "traffic": 40, "wide": 8}[self.kind] * self.periods
        self.min_events = {"control": 8 * self.streams * self.periods, "traffic": 20 * self.streams,
                           "wide": int(0.9 * 64 * 8 * self.rows)}[self.kind]
        self._base = None
        self.n = self.base().shape[1]

    # -- input
    def base(self) -> np.ndarray:
        """[N_BASE][n][2] (u8 or f32): one period of N_BASE phase-continuous transmissions (cfg3: one capture)."""
        if self._base is not None:
            return self._base
        from tools import p25tx as tx
        rows = []
        if self.kind == "wide":
            n = self.fs * 150 // 1000
            cap = np.zeros(n, dtype=np.complex128)
            for i in range(64):
                k = (37 * i + 5) % 1536
                f = (k if k < 768 else k - 1536) * 12500.0
                st = tx.control_channel(3000 + i, 2, lead_idle=0)
                iq = tx.modulate_iq_periodic(st.dibits, self.fs, snr_db=None, cfo_cycles=int(round(f * 0.150)), seed=i, amplitude=0.01)
                cap += np.roll(iq, 9973 * i)
            rng = np.random.default_rng(1)
            cap += 10 ** (-60 / 20) / np.sqrt(2) * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
            rows.append(cap.astype(np.complex64).view(np.float32).reshape(n, 2))
        else:
            for b in range(1 if self.streams == 1 else N_BASE):
                st = tx.control_channel(1000 + b, 2, lead_idle=0) if self.kind == "control" else tx.traffic_channel(2000 + b, 1, lead_idle=0)
                iq = tx.modulate_iq_periodic(st.dibits, self.fs, snr_db=self.snr, cfo_cycles=3 * (b - N_BASE // 2), seed=b)
                n = len(iq)
                r = tx.iq_to_u8(iq).reshape(n, 2) if self.fmt == "u8" else iq.view(np.float32).reshape(n, 2)
                rows.append(np.tile(r, (self.periods, 1)) if self.periods > 1 else r)
        self._base = np.stack(rows)
        return self._base

    def shift(self, g: int) -> int:
        """Circular shift of global input row g."""
        b = self.base()
        n = b.shape[1]
        return (400 * 77 * g) % n if self.kind == "wide" else (g // len(b)) * 5003 % n      # tile_on_device's rule

    def device_input(self, rank: int):
        import torch
        from tools.shape_bench import tile_on_device
        base = torch.from_numpy(self.base()).cuda()
        if self.kind == "wide":
            return torch.stack([torch.roll(base[0], -self.shift(rank * self.rows + c), dims=0) for c in range(self.rows)]).contiguous()
        return tile_on_device(base, self.rows, first=rank * self.rows)

    def oracle_row(self, g: int) -> np.ndarray:
        """Host copy of global input row g in the oracle's layout (u8 pairs flattened, or complex64)."""
        b = self.base()
        row = np.roll(b[g % len(b)], -self.shift(g), axis=0)
        return row.reshape(-1) if self.fmt == "u8" else np.ascontiguousarray(row).view(np.complex64).reshape(-1)

    # -- accounting (SURVEY.md 8d)
    def alg_bytes_per_step(self) -> float:
        return self.rows * self.n * float(self.bps) + self.streams * (self.n // self.decim) * 4.0

    def config(self):
        gb = self.rows * self.n * self.bps / 1e9
        return {"workload": self.desc, "streams_per_gpu": self.streams, "samples_per_row_per_step": self.n, "input_rows_per_gpu": self.rows,
                "sample_rate": self.fs, "decimation": self.decim, "input_format": self.fmt, "snr_db": self.snr,
                "l2_policy": f"inputs ({gb:.2f} GB/step) larger than L2" if gb > 0.3 else f"inputs {gb * 1e3:.0f} MB/step; L2 flushed by the 2.95 GB headline batch between legs",
                "parallelism": f"streams sharded over {self.world} GPU(s), no collective"}


class ClockSampler(threading.Thread):
    """NVML poll of SM clock / throttle reasons during the timed region."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.power = index, [], set(), False, []
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1e3)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def result(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples),
                "power_w_max": float(max(self.power)) if self.power else None}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            hbm, src = float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        hbm, src = 6650.0, "fallback (B200_PROFILING.md)"
    fp32 = None
    try:
        with open(os.path.join(ROOT, "profiles", "pipe_peaks_r02.json")) as f:
            fp32 = float(json.load(f)["fp32_ffma2_tflops"])
    except Exception:
        pass
    return hbm, src, fp32


def pipe_peak(key: str):
    try:
        with open(os.path.join(ROOT, "profiles", "pipe_peaks_r02.json")) as f:
            return float(json.load(f)[key])
    except Exception:
        return None


class StreamGate:
    """Holds a CUDA stream back until the host opens it (cuStreamWaitValue32 on a pinned flag).  The timed loop is
    enqueued behind the gate, so the device runs its K steps back to back from a full launch queue -- what a
    steady-state producer sees -- instead of inheriting the scheduling jitter of eight Python ranks sharing one host.
    Falls back to no gate if the driver API is unavailable."""

    def __init__(self, stream_handle: int, enabled: bool = True):
        self.ok = False
        # A closed gate deadlocks anything that makes launches synchronous (a profiler replaying kernels one by one,
        # CUDA_LAUNCH_BLOCKING): never gate then, and a watchdog opens the gate after 250 ms whatever happens.
        blocking = os.environ.get("CUDA_LAUNCH_BLOCKING", "0") not in ("", "0")
        injected = any(k.startswith(("CUDA_INJECTION", "NV_COMPUTE_PROFILER", "NSIGHT", "NV_NSIGHT", "NVTX_INJECTION")) for k in os.environ)
        if not enabled or blocking or injected:
            return
        try:
            import torch
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                from cuda.bindings import driver as drv
            self.flag = torch.zeros(1, dtype=torch.int32).pin_memory()
            err, = drv.cuStreamWaitValue32(drv.CUstream(stream_handle), drv.CUdeviceptr(self.flag.data_ptr()), 1,
                                           drv.CUstreamWaitValue_flags.CU_STREAM_WAIT_VALUE_GEQ)
            self.ok = int(err) == 0
            if self.ok:
                self.watchdog = threading.Timer(0.25, self.open)
                self.watchdog.daemon = True
                self.watchdog.start()
        except Exception:
            self.ok = False

    def open(self):
        if self.ok:
            self.flag[0] = 1


def pin_to_gpu_numa_node(index: int) -> None:
    """Multi-GPU host leg: run this rank on the CPUs next to its GPU so that the pinned staging buffer is allocated
    (first touch) on that NUMA node and eight ranks do not all stream from one socket's memory.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass


# ------------------------------------------------------------------------------------------------ CPU arm (the oracle)
def single_stream_split(po, native: bool, fmt: int, front: bool, row: np.ndarray, decim: int) -> dict:
    """The reference's actual shape (SURVEY.md 8d): one stream on one thread, timed separately for the `demod` thread's
    work (src/demod.rs:62-119) and the `receiver` thread's (src/recv.rs:140-167), a few repetitions of one step's row."""
    reps = 4
    chain, rx = po.DemodChain(fmt, front, native=native), po.MessageReceiver(native=native)
    t0 = time.perf_counter()
    bbs = [chain.feed(row) for _ in range(reps)]
    t1 = time.perf_counter()
    for bb in bbs:
        rx.feed(bb)
    t2 = time.perf_counter()
    n_in = reps * (row.size // (2 if fmt == po.FMT_U8 else 1))
    return {"threads": 1, "demod_iq_msamples_per_s": n_in / (t1 - t0) / 1e6,
            "decode_baseband_msamples_per_s": n_in / decim / (t2 - t1) / 1e6,
            "realtime_channels_one_core": 1.0 / ((t2 - t0) / (n_in / decim / 48000.0))}


def cpu_arm(steps: int, warmup: int, wl: Workload):
    """Oracle CPU implementation on the host cores (rank 0 only).  Returns (Msamples/s, ms/step, info).
    Each step is the whole 1,024-stream batch of the GPU arm (about 8 core-seconds of work); for cfg5 a bounded sample
    of 4,096 of the 65,536 streams.  The headline number runs the receiver WITHOUT the per-sample sync correlation while
    locked -- the same work the GPU walker does; `always_correlate` repeats one step with it (the reference is believed
    to correlate on every sample [RECALL], work whose result is discarded)."""
    from oracle import pyoracle as po
    try:
        po.build(native=True)
        native = True
    except Exception:
        native = False
    cores = len(os.sched_getaffinity(0)) or 1
    L = po.lib(native)
    n_streams = 4096 if wl.name == "cfg5" else wl.streams
    ofmt, front = (po.FMT_U8 if wl.fmt == "u8" else po.FMT_CF32), wl.decim == 50
    iq = np.stack([wl.oracle_row(s) for s in range(n_streams)])

    def run(k: int, w: int, always: int):
        L.p25o_set_always_correlate(always)
        times = []
        for it in range(w + k):
            t0 = time.perf_counter()
            total, _, _ = po.batch_run(ofmt, front, iq, n_streams, wl.n, cores, native=native)
            dt = time.perf_counter() - t0
            if it >= w:
                times.append(dt)
            assert total >= 3 * n_streams, "oracle decoded too few events"   # fresh receivers: >= 1 whole TSDU each
        return 1e3 * float(np.mean(times))

    ms = run(steps, warmup, 0)
    ms_always = run(1, 0, 1)
    L.p25o_set_always_correlate(0)
    val = n_streams * wl.n / (ms * 1e-3) / 1e6
    info = {"value": val, "unit": "Msamples/s", "cores": cores, "kind": "port",
            "sample": f"{n_streams} of {wl.streams * wl.world} streams x {wl.n} samples per step ({steps} timed step(s)), {cores} threads, "
                      f"oracle built {'-march=native' if native else '-march=x86-64-v3'}; receiver without the discarded per-sample "
                      "correlation while locked (same work as the GPU walker); the Rust reference cannot be built here",
            "always_correlate": {"value": n_streams * wl.n / (ms_always * 1e-3) / 1e6, "unit": "Msamples/s", "cores": cores,
                                 "note": "receiver correlates the sync template on every sample even while locked [RECALL of p25.rs]"},
            "single_stream": single_stream_split(po, native, ofmt, front, iq[0], wl.decim)}
    return val, ms, info


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = Workload(args.workload, max(1, args.gpus))
    val, ms, info = cpu_arm(args.steps, args.warmup, wl)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Msamples/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": wl.config(), "cpu_baseline": info,
            "e2e": {"value": val, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "realtime_channels": val * 1e6 / wl.decim / 48000.0, "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm
def sampled_streams(wl: Workload, n_sm: int = 148):
    """Deterministic sample of the rank's streams: first, last and streams in which a CTA's / warp's share of the
    flattened work begins or ends mid-stream (the launch geometry of ddc_fm.cu), plus a stride over the rest."""
    S = wl.streams
    if S <= 24:
        return list(range(S))
    pick = {0, 1, S - 2, S - 1}
    if wl.decim == 50:
        bps, grid = (wl.n // 50 + 63) // 64, n_sm * 3
        n_static = (S * bps // grid) * 7 // 8
        pick |= {(n_static * b) // bps for b in range(1, grid, grid // 6)}
        pick |= {min(S - 1, (n_static * grid) // bps + 3)}
    elif wl.decim == 5:
        ips, gw = (wl.n // 5 + 123) // 124, n_sm * 5 * 4
        pick |= {(S * ips * g // gw) // ips for g in range(1, gw, gw // 6)}
    pick |= set(range(5, S, max(1, S // 5)))
    return sorted(pick)[:16]


class OracleSample:
    """One oracle DemodChain + MessageReceiver per sampled stream, stepped alongside the GPU."""

    def __init__(self, wl: Workload, rank: int, streams):
        from oracle import pyoracle as po
        po.lib().p25o_set_always_correlate(0)
        self.po, self.wl, self.streams = po, wl, list(streams)
        ofmt, mode = (po.FMT_U8 if wl.fmt == "u8" else po.FMT_CF32), (1 if wl.decim == 50 else 0)
        self.chains = [po.DemodChain(ofmt, mode) for _ in self.streams]
        self.rx = [po.MessageReceiver(stream=s) for s in self.streams]
        self.rows = [wl.oracle_row(rank * wl.rows + s) for s in self.streams]
        self.events = []

    def step(self, n_steps: int):
        from concurrent.futures import ThreadPoolExecutor

        def one(i):
            out = []
            for _ in range(n_steps):
                out.append(self.rx[i].feed(self.chains[i].feed(self.rows[i])))
            return out
        with ThreadPoolExecutor(max_workers=min(16, len(self.streams))) as ex:
            for out in ex.map(one, range(len(self.streams))):
                self.events.extend(out)

    def compare(self, gpu_events: np.ndarray):
        key = lambda a: {(int(e["stream"]), int(e["sample"]), int(e["kind"]), bytes(e["payload"][: int(e["len"])])) for e in a}
        ref = np.concatenate(self.events) if self.events else np.zeros(0, dtype=self.po.EVENT_DTYPE)
        got = gpu_events[np.isin(gpu_events["stream"], self.streams)]
        a, b = key(got), key(ref)
        return {"streams": len(self.streams), "oracle_events": len(ref), "gpu_events": len(got), "differing": len(a ^ b)}


DUMP_LIMIT = 64_000_000               # bytes --dump-outputs may write
DUMP_EVENT_BYTES = 4 * 8 + 60 * 4     # one event row of events_fields + events_payload


def last_step_outputs(ctx, wl: Workload, drained, steps_done: int) -> dict:
    """Events and baseband of the last step (see --dump-outputs).  `drained` holds the packed polls that collected it."""
    import p25rx_b200 as p25
    n_out, S = wl.n // wl.decim, wl.streams
    k = min(S, (DUMP_LIMIT - 4096) // (4 * n_out + 2 * wl.slot_events * DUMP_EVENT_BYTES))   # room for twice the usual events
    streams = np.arange(S) if k == S else np.sort(np.random.default_rng(0).choice(S, k, replace=False))
    ev = np.concatenate([ctx.unpack(w, ne) for w, ne in drained] + [np.zeros(0, dtype=p25.EVENT_DTYPE)])
    ev = ev[(ev["sample"] >= (steps_done - 1) * n_out) & np.isin(ev["stream"], streams)]
    ev = ev[np.lexsort((ev["sample"], ev["stream"]))]
    out = {"events_fields": np.stack([ev["stream"], ev["kind"], ev["sample"], ev["len"]], axis=1).astype(np.float64),
           "events_payload": ev["payload"].astype(np.float32),
           "baseband": np.stack([ctx.read_baseband(int(s), n_out) for s in streams]),
           "streams": streams.astype(np.float64)}
    assert sum(a.nbytes + 128 for a in out.values()) <= DUMP_LIMIT, {n: a.shape for n, a in out.items()}
    return out


def measure(wl: Workload, rank: int, local: int, K: int, W: int, barrier, gate_on: bool, verify: bool, sustained_s: float, Ke: int,
            dump: bool = False):
    """All device legs of one workload on this rank.  Returns a dict of per-rank times / counts (caller reduces)."""
    import torch
    import p25rx_b200 as p25
    S, n = wl.streams, wl.n
    dev = wl.device_input(rank)
    torch.cuda.synchronize()          # the library runs on its own stream: inputs complete before they are handed over
    slots = wl.slot_events * (W + K) + 32
    ctx = p25.Context(S, fmt=p25.FMT_U8_IQ if wl.fmt == "u8" else p25.FMT_CF32_IQ, decimation=wl.decim, max_chunk_samples=n,
                      device=local, event_slots=slots)
    stream = torch.cuda.ExternalStream(ctx.cuda_stream, device=local)
    out = {}
    orc = OracleSample(wl, rank, sampled_streams(wl)) if verify else None
    gpu_ev = []

    def take(words, ne):
        if orc is not None and ne:
            e = ctx.unpack(words, ne)
            gpu_ev.append(e[np.isin(e["stream"], orc.streams)].copy())
        return ne

    def drain_raw():
        """Collect every queued event (several polls if the pinned buffer cannot hold them at once).  No host-side
        processing here: the views stay valid until two further polls are started, so only a multi-poll drain copies."""
        got = []
        while True:
            w, ne, more = ctx.poll_packed(copy=False)
            got.append((w.copy() if more or got else w, ne))
            if not more:
                return got

    def account(got):
        return sum(take(w, ne) for w, ne in got), sum(4 * len(w) + 16 for w, _ in got)

    def drain():
        return account(drain_raw())

    # ---------------- leg 1: device-resident input ("value") + the demod kernel's own event-timed duration
    n_events = 0
    for _ in range(W):
        ctx.process(dev, n)
        n_events += drain()[0]
    ctx.sync()
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ctx.launch_count
    ctx.demod_timing(True)
    barrier()
    t_host0 = time.perf_counter()
    with torch.cuda.stream(stream):
        gate = StreamGate(ctx.cuda_stream, enabled=gate_on)   # the device starts when the launch queue holds the first steps
        t_begin.record(stream)
        for k in range(K):
            if k == 48:
                gate.open()                              # bounded: never let a gated queue fill up
            ctx.process(dev, n)                          # demod kernel, then the decode walker (beside the next demod kernel)
        gate.open()
        out["enqueue_ms"] = 1e3 * (time.perf_counter() - t_host0)
        raw = drain_raw()                                # packed compaction straight into pinned host memory (synchronises)
        t_end.record(stream)
    burst_events, out["d2h_burst_bytes"] = account(raw)
    with torch.cuda.stream(stream):
        pass
    barrier()
    out["launches"] = ctx.launch_count - l0
    out["dev_ms"] = t_begin.elapsed_time(t_end)
    out["ddc_ms"], n_timed = ctx.demod_timing(False)     # the library's own event pair right around each kernel launch
    assert n_timed == min(K, 128)
    if dump:
        out["dump"] = last_step_outputs(ctx, wl, raw, W + K)
    n_events += burst_events
    # ---------------- sampled-oracle check of the warm-up and every timed step
    if orc is not None:
        orc.step(W + K)
        out["oracle_check"] = orc.compare(np.concatenate(gpu_ev) if gpu_ev else np.zeros(0, dtype=p25.EVENT_DTYPE))
        d = out["oracle_check"]
        assert d["oracle_events"] >= 6 * d["streams"] * K and d["differing"] <= max(1, d["oracle_events"] // 500), d
    assert burst_events >= wl.min_events * (K - 1), (burst_events, wl.min_events, K)
    out["events_per_step"] = burst_events / K

    # ---------------- per-kernel breakdown with the two kernels serialised on one stream (not part of `value`)
    ctx.set_overlap(False)
    bk = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(5)]
    with torch.cuda.stream(stream):
        for e3 in bk:
            e3[0].record(stream)
            ctx.demod(dev, n, want_baseband=False)
            e3[1].record(stream)
            ctx.decode()
            e3[2].record(stream)
    ctx.sync()
    out["ddc_serial_ms"] = sum(e[0].elapsed_time(e[1]) for e in bk) / len(bk)
    out["walk_ms"] = sum(e[1].elapsed_time(e[2]) for e in bk) / len(bk)
    drain()
    ctx.set_overlap(wl.decim == 50 and wl.fmt == "cf32")     # back to the library's default for this shape

    # ---------------- sustained: the production call pattern for >= sustained_s seconds
    if sustained_s > 0:
        est = max(out["dev_ms"] / K, 1e-3)
        Ks = max(K, int(sustained_s * 1e3 / est))
        sampler = ClockSampler(local)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        sampler.start()
        got = 0
        with torch.cuda.stream(stream):
            s0.record(stream)
            for k in range(Ks):
                ctx.process(dev, n)
                ctx.poll_start()                         # drain of step k queued behind its walker
                if k:
                    got += ctx.poll_packed(copy=False)[1]    # collects step k - 1 while step k runs
            got += ctx.poll_packed(copy=False)[1]
            s1.record(stream)
        barrier()
        sampler.stop_flag = True
        sampler.join()
        out["sustained_ms"] = s0.elapsed_time(s1)
        out["sustained_steps"] = Ks
        out["clocks"] = sampler.result()
        assert got >= wl.min_events * (Ks - 2), (got, wl.min_events, Ks)

    # ---------------- e2e: the public call sequence with pinned host input
    host = ctx.host_alloc(tuple(dev.shape), np.uint8 if wl.fmt == "u8" else np.float32)
    torch.from_numpy(host).copy_(dev)
    torch.cuda.synchronize()
    for _ in range(2):
        ctx.process(host, n)
        ctx.poll_packed(copy=False)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d2h = 0
    barrier()
    with torch.cuda.stream(stream):
        e0.record(stream)
        # the streaming pattern of the sustained leg: step k's H2D copy and kernels are queued before the events of step
        # k - 1 are collected, so the copy of one step overlaps the kernels of the previous one (two staging buffers on
        # the library's copy stream); every step's input copy and event drain still lie inside the timed region
        for k in range(Ke):
            ctx.process(host, n)                         # H2D copy of the step's input happens inside
            ctx.poll_start()                             # pack kernel -> pinned host memory, asynchronous
            if k:
                w, ne, _ = ctx.poll_packed(copy=False)   # events of step k - 1
                d2h += 4 * len(w) + 16
        w, ne, _ = ctx.poll_packed(copy=False)           # ... and of the last step (synchronises)
        d2h += 4 * len(w) + 16
        e1.record(stream)
    barrier()
    out["e2e_ms"] = e0.elapsed_time(e1)
    out["e2e_steps"] = Ke
    out["d2h_per_step"] = d2h // Ke
    ctx.host_free(host)
    ctx.close()
    del dev
    torch.cuda.empty_cache()
    return out


def h2d_ceiling(local: int, barrier):
    """Plain cudaMemcpyAsync from pinned host memory, all ranks at once: the ceiling of any end-to-end number."""
    import torch
    nbytes = 1 << 30
    h = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{local}")
    d.copy_(h, non_blocking=True)
    torch.cuda.synchronize()
    ms = None
    for _ in range(3):                                   # best of three: the ceiling is what the box can deliver
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(4):
            d.copy_(h, non_blocking=True)
        e1.record()
        barrier()
        t = e0.elapsed_time(e1)
        ms = t if ms is None else min(ms, t)
    del h, d
    torch.cuda.empty_cache()
    return 4 * nbytes, ms


def summarise(wl: Workload, m: dict, world: int, K: int, hbm: float, hbm_src: str, fp32: float | None, h2d_gbs: float | None):
    S, n = wl.streams, wl.n
    total = world * wl.rows * n * K
    value = total / (m["dev_ms"] * 1e-3) / 1e6
    e2e_value = world * wl.rows * n * m["e2e_steps"] / (m["e2e_ms"] * 1e-3) / 1e6
    alg = wl.alg_bytes_per_step()
    achieved = alg / (m["ddc_ms"] * 1e-3) / 1e9
    roof = {"kernel": wl.kernel, "bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm,
            "traffic": None, "peak_source": hbm_src, "algorithmic_bytes_per_launch": alg, "kernel_ms": m["ddc_ms"]}
    tf = {"cfg2": "ddc_fm_traffic.json", "cfg2u8": "ddc50_u8_imma_traffic.json", "cfg5": "ddc5_u8_imma_traffic.json",
          "cfg3": "pfb_traffic.json"}.get(wl.name)
    if tf:
        try:
            with open(os.path.join(ROOT, "profiles", tf)) as f:
                tr = json.load(f)
            roof["traffic"] = tr.get("dram_bytes_per_launch")
            roof["traffic_source"] = f"profiles/{tf} (ncu --set full, {tr.get('captured', 'round 1')})"
        except Exception:
            pass
    if wl.decim == 5 or wl.fmt == "u8" or wl.kind == "wide":
        # FP32-bound shapes (SURVEY 8d): FIR FMAs per 48 kHz output against the measured FFMA2 peak
        fma = {5: 2 * (25 + 41), 50: 2 * (250 + 25 + 41), 400: 2 * 15 + 26}[wl.decim]   # FMAs per 48 kHz output (DESIGN.md section 4)
        if wl.decim == 5 and wl.fmt == "u8":
            # the /5 decimator of the u8 kernel runs as u8 x s8 mma.sync (36 x m16n8k32 per 256 outputs, issued ops incl. the
            # zeros of the band); only the 41-tap channel filter is left on the FP32 pipe
            fma = 2 * 41
            roof["tensor_int8_tops"] = 2.0 * 36 * 16 * 8 * 32 / 256 * wl.streams * (n // wl.decim) / (m["ddc_ms"] * 1e-3) / 1e12
            roof["tensor_int8_peak_tops"] = pipe_peak("mma_sync_u8s8_k32_tops")   # legacy mma.sync rate, tools/pipe_peaks.cu
        if wl.decim == 50 and wl.fmt == "u8":
            # 168 x m16n8k32 per 128 outputs (the 290-tap /50 FIR on the raw bytes, three limbs); channel filter on FFMA2
            fma = 2 * 41
            roof["tensor_int8_tops"] = 2.0 * 168 * 16 * 8 * 32 / 128 * wl.streams * (n // wl.decim) / (m["ddc_ms"] * 1e-3) / 1e12
            roof["tensor_int8_peak_tops"] = pipe_peak("mma_sync_u8s8_k32_tops")
        flops = 2.0 * fma * wl.streams * (n // wl.decim)
        roof["fp32_tflops"] = flops / (m["ddc_ms"] * 1e-3) / 1e12
        if fp32:
            roof["fp32_peak_tflops"] = fp32
            roof["fp32_frac"] = roof["fp32_tflops"] / fp32
    e2e = {"value": e2e_value, "unit": "Msamples/s", "h2d_bytes_per_step": wl.rows * n * wl.bps, "d2h_bytes_per_step": m["d2h_per_step"],
           "ms_per_step": m["e2e_ms"] / m["e2e_steps"], "steps": m["e2e_steps"]}
    if h2d_gbs:
        e2e["h2d_ceiling_gbs"] = h2d_gbs
        e2e["frac_of_h2d_ceiling"] = (e2e_value * 1e6 * wl.bps / 1e9) / h2d_gbs
    r = {"value": value, "unit": "Msamples/s", "ms_per_step": m["dev_ms"] / K, "steps": K, "scaling": wl.scaling,
         "realtime_channels": value * 1e6 / wl.decim / 48000.0 if wl.kind != "wide" else None,
         "roofline": roof, "e2e": e2e, "config": wl.config(),
         "kernels": {"demod_kernel_ms": m["ddc_ms"], "step_ms": m["dev_ms"] / K, "host_enqueue_ms_per_step": m["enqueue_ms"] / K,
                     "serialised": {"demod_kernel_ms": m["ddc_serial_ms"], "p25_walk_kernel_ms": m["walk_ms"]}},
         "events_per_step": m["events_per_step"], "d2h_bytes_burst_drain": m["d2h_burst_bytes"]}
    if wl.kind == "wide":
        r["realtime_factor"] = (wl.rows * n / wl.fs) / (m["dev_ms"] * 1e-3 / K)
    if "sustained_ms" in m:
        r["sustained"] = {"value": world * wl.rows * n * m["sustained_steps"] / (m["sustained_ms"] * 1e-3) / 1e6, "unit": "Msamples/s",
                          "seconds": m["sustained_ms"] * 1e-3, "steps": m["sustained_steps"],
                          "pattern": "process + poll_start per step, events of step k-1 collected while step k runs"}
    if "oracle_check" in m:
        r["oracle_check"] = m["oracle_check"]
    return r


def run_b200(args):
    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    full_affinity = os.sched_getaffinity(0)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        pin_to_gpu_numa_node(local)          # pinned staging memory on the GPU's own NUMA node (first touch)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(m: dict):
        keys = [k for k in ("dev_ms", "e2e_ms", "ddc_ms", "walk_ms", "ddc_serial_ms", "sustained_ms") if k in m]
        t = torch.tensor([m[k] for k in keys], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        for k, v in zip(keys, t.tolist()):
            m[k] = float(v)
        return m

    hbm, hbm_src, fp32 = measured_peaks()
    K, W = args.steps, max(args.warmup, 3)
    nbytes, ms = h2d_ceiling(local, barrier)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    h2d_gbs = world * nbytes / (float(t.item()) * 1e-3) / 1e9

    wl = Workload(args.workload, world)
    sampler = ClockSampler(local)
    sampler.start()
    m = reduce_max(measure(wl, rank, local, K, W, barrier, not args.no_gate, not args.no_verify, args.sustained, args.e2e_steps,
                           dump=args.dump_outputs is not None and rank == 0))
    sampler.stop_flag = True
    sampler.join()
    if "dump" in m:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in m.pop("dump").items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    head = summarise(wl, m, world, K, hbm, hbm_src, fp32, h2d_gbs)
    line = {"metric": METRIC, "value": head["value"], "unit": "Msamples/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": head["config"], "realtime_channels": head["realtime_channels"], "e2e": head["e2e"],
            "gpu_launches": int(m["launches"]), "kernels": head["kernels"], "roofline": head["roofline"],
            "clocks": m.get("clocks") or sampler.result(), "h2d_ceiling": {"gbs_all_ranks": h2d_gbs, "how": "4 x 1 GiB pinned cudaMemcpyAsync per rank, all ranks at once, max over ranks, best of 3"}}
    for k in ("sustained", "oracle_check"):
        if k in head:
            line[k] = head[k]
    line["events_checked"] = {"events_per_step": head["events_per_step"], "oracle": head.get("oracle_check")}

    extras = [x for x in (args.extra.split(",") if args.extra else []) if x and x != wl.name]
    if extras:
        line["workloads"] = {}
    for name in extras:
        w2 = Workload(name, world)
        k2 = {"cfg1": 10, "cfg2u8": 20, "cfg3": 10, "cfg4": 10, "cfg5": 10, "cfg2": 20}[name]
        m2 = reduce_max(measure(w2, rank, local, k2, 3, barrier, not args.no_gate, not args.no_verify and name != "cfg3", 0.0,
                                {"cfg5": 2, "cfg4": 3}.get(name, 4)))
        line["workloads"][name] = summarise(w2, m2, world, k2, hbm, hbm_src, fp32, h2d_gbs)

    if rank == 0:
        os.sched_setaffinity(0, full_affinity)
        if world == 1 and not args.no_cpu:
            _, _, info = cpu_arm(1, 0, wl)
            line["cpu_baseline"] = info
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40, help="timed steps of the headline workload (`value`)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-gate", action="store_true", help="do not hold the stream back while the timed steps are enqueued")
    ap.add_argument("--no-verify", action="store_true", help="skip the sampled-oracle check of the timed steps")
    ap.add_argument("--sustained", type=float, default=2.0, help="seconds of the sustained leg of the headline workload (0 = skip)")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--workload", default="cfg2", choices=["cfg1", "cfg2", "cfg2u8", "cfg3", "cfg4", "cfg5"],
                    help="headline workload (default cfg2 = BASELINE configs[1], the configuration the metric is quoted on)")
    ap.add_argument("--extra", default=None, help=f"comma list of further workloads reported under `workloads` (default: {EXTRA_DEFAULT} "
                                                  "when the headline is cfg2; '' for none)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the events and baseband of the last timed step of the headline workload to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs dumps the GPU path (--impl b200)")
    if args.extra is None:
        args.extra = EXTRA_DEFAULT if args.workload == "cfg2" and args.impl == "b200" else ""
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
