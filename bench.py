#!/usr/bin/env python
"""bench.py — Gsamples/s of 8-bit baseband through the full coherent-dedispersion chain
(unpack -> fft_r2c -> rfi_s1 -> dedisperse -> watfft -> rfi_s2 -> signal_detect) on B200,
with per-stage achieved HBM GB/s against the measured copy peak, next to the restated
reference CPU path timed on the same box.

Usage: python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]
  * a "step" = one block of synthetic baseband through the whole chain on each rank; every timed window is K steps;
  * --dump-outputs DIR writes what the last timed step computed (dump_block_outputs) for output-by-output comparison
    of two builds; apart from that bench.py writes no files (the source tree may be read-only);
  * workload = BASELINE.json configs[2], the J1644-4559 shape the north star names: dual-polarisation
    8-bit, 2^26 samples per stream per block, 400 MHz, DM 562.05, C = 2^11 channels (rows of 2^14 time
    samples), manual zap list, SK and the boxcar detector; one block in two of the ring carries an injected
    dispersed pulse, so the candidate path (host series from the detector kernel) is inside the timed region.
    N > 1 shards independent blocks across ranks (weak scaling, no collective on the data path);
    `secondary` repeats value / e2e on BASELINE configs[1] (2^24 samples, one stream);
  * `value`  = samples / time with the blocks already resident in HBM (ring of distinct blocks larger than L2);
    through ONE context per GPU for multi-stream blocks (a context spreads the streams of a block over two lanes
    itself), over several contexts for single-stream ones (`contexts_per_gpu`), two blocks in flight per context;
    `single_context` is the same through ONE context (the reference drives one queue per device);
  * `e2e`    = the same from pinned HOST buffers through srtb_b200_submit_block()/collect_block() (the
    pinned-host ring: H2D of block i overlaps the compute of block i-1); every block's H2D and the D2H
    of its detector result (and of positive series) are inside the timed region;
  * `roofline` = the dominant kernel of the block path (the one-kernel waterfall group: s1 + chirp + waterfall FFT + SK +
    column sums): its compulsory bytes per launch / its launch time, CUDA events inside the library on the launching
    stream, vs the measured copy peak (MEASURED_PEAKS.json hbm_gbs, else 6650 fallback); `traffic` = its DRAM bytes per
    launch from the committed ncu capture; `roofline.fused` has every kernel group of the block path against the bytes
    THEY must move; `stages` every per-pipe C-ABI stage alone (SURVEY.md §8d bytes); `roofline.chain` the whole block on
    three byte counts (unfused algorithmic, the launched kernels' sweep bytes, measured DRAM bytes);
  * `cpu_baseline` = the CPU oracle (port of the reference operators, OpenMP, all host cores) on a bounded
    sample of the same workload (rank 0, N = 1 only).
--impl reference times that CPU path alone (rank 0) with the same JSON shape.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

# The two lanes of a context rely on the driver giving their CUDA streams separate hardware work queues. With NCCL in
# the process (torchrun, N > 1) and this variable unset the lanes were seen to alias (config 3: 120 instead of 131
# Gsamples/s per GPU); 8 — the documented default — set explicitly restores it, 1 serialises them, 32 co-schedules the
# big sweeps and is slower (profiles/r02s_connections.md). Must be in the environment before CUDA initialises.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "8")

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT / "simple-radio-telescope-backend_b200"))
sys.path.insert(0, str(ROOT / "tests"))
sys.dont_write_bytecode = True   # no __pycache__ beside the modules imported from the (possibly read-only) tree

import numpy as np  # noqa: E402

SRTB_RING_SLOTS = 3   # SRTB_B200_RING_SLOTS in include/srtb_b200.h
METRIC = "Gsamples/s 8-bit baseband through full dedisperse chain"
UNIT = "Gsamples/s"

WORKLOADS = {
    # BASELINE.json configs[0] shape (srtb_config_1644-4559.cfg): 2^30 two-bit samples, inverted 64 MHz band
    "config1": dict(log2n=30, bits=2, fmt="simple", channels=1 << 11, dm=-478.80, f_low=1437.0, bw=-64.0,
                    fs=128e6, avg_thr=1.5, sk_thr=1.05, snr=8.0, chan_thr=0.9, maxbox=256, freq_list="1418-1422"),
    # BASELINE.json configs[1]
    "config2": dict(log2n=24, bits=-8, fmt="simple", channels=1 << 11, dm=56.778, f_low=1000.0, bw=500.0,
                    fs=1e9, avg_thr=5.0, sk_thr=1.05, snr=8.0, chan_thr=0.9, maxbox=256, freq_list=""),
    # BASELINE.json configs[2]: dual-pol 400 MHz, 2^26 per stream, DM 562.05, full RFI + detect
    "config3": dict(log2n=26, bits=-8, fmt="naocpsr_snap1", channels=1 << 11, dm=562.05, f_low=1000.0,
                    bw=400.0, fs=8e8, avg_thr=1.5, sk_thr=1.05, snr=8.0, chan_thr=0.9, maxbox=256,
                    freq_list="1018-1022"),
    # BASELINE.json configs[3]: Crab giant-pulse injection, 2^27-sample blocks, DM sweep 0..1000 (21 trials), block-sharded
    "config4": dict(log2n=27, bits=-8, fmt="simple", channels=1 << 11, dm=56.78, f_low=1000.0, bw=500.0,
                    fs=1e9, avg_thr=5.0, sk_thr=1.05, snr=8.0, chan_thr=0.9, maxbox=256, freq_list="",
                    dms=[0.0, 56.78] + [50.0 * i for i in range(2, 21)]),      # trial 1 is the Crab's DM itself
    # BASELINE.json configs[4]: continuous UDP-shaped stream (fastmb_roach2 framing), 1 Gsample/s per GPU, pinned ring
    "config5": dict(log2n=26, bits=-8, fmt="simple", channels=1 << 11, dm=56.778, f_low=1000.0, bw=500.0,
                    fs=1e9, avg_thr=5.0, sk_thr=1.05, snr=8.0, chan_thr=0.9, maxbox=256, freq_list="",
                    rate_per_gpu=1e9, seconds=10.0),
}

STAGES = ["unpack", "fft_r2c", "rfi_s1", "dedisperse", "watfft", "rfi_s2", "signal_detect"]
FORMAT_STREAM_COUNT = {"simple": 1, "naocpsr_snap1": 2, "interleaved_samples_2": 2, "gznupsr_a1": 2, "gznupsr_a1_4": 4}


def workload_string(wname: str, w: dict) -> str:
    """identical in both arms (the driver compares them)"""
    streams = FORMAT_STREAM_COUNT[w["fmt"]]
    return (f"{wname}: 2^{w['log2n']}-sample blocks x{streams} stream(s), {abs(w['bits'])}-bit {w['fmt']}, "
            f"C=2^11, DM={w['dm']}, full RFI + detect")


def sweep_bytes_per_sample(w: dict) -> float:
    """bytes the kernels process_block launches for this workload MUST move per input sample (every sweep reads and
    writes its tile once): fused first sweep b/8 + 4, every further R2C sweep 8, then either the one-kernel
    waterfall (8; + 2 for the tabulated chirp phases, 4 bytes per bin) or, for rows of 2^15..2^18, chirp-on-load
    column sweep 8 + last sweep 8 + zap-aware column sums 4"""
    q = w["log2n"] - 1                      # complex points of the packed transform
    r2c_sweeps = 1 if q <= 12 else (2 if q <= 20 else (3 if q <= 26 else 4))
    rows = (1 << q) // w["channels"]
    fused_first = (abs(w["bits"]) == 8 and w["fmt"] in ("simple", "naocpsr_snap1", "interleaved_samples_2", "gznupsr_a1")) or \
                  (abs(w["bits"]) in (2, 4) and w["fmt"] == "simple")
    # a stream's first sweep reads the bytes of EVERY stream of an interleaved block (each stream picks its own samples)
    raw = abs(w["bits"]) / 8 * (FORMAT_STREAM_COUNT[w["fmt"]] if fused_first else 1)
    first = (raw + 4) if fused_first else (raw + 4 + 8)  # else: unpack kernel, then the sweep
    if "dms" in w:                           # DM sweep: R2C once, then per trial the waterfall group (on-the-fly chirp)
        per_trial = 8 if 1024 <= rows <= 16384 else 8 + 8 + 4
        return first + 8 * (r2c_sweeps - 1) + per_trial * len(w["dms"])
    waterfall = (8 + 2) if 1024 <= rows <= 16384 else 8 + 8 + 4
    return first + 8 * (r2c_sweeps - 1) + waterfall



def stage_bytes(n: int, bits: int) -> dict:
    """algorithmic bytes per stream per block, SURVEY.md §8(d)"""
    b = abs(bits)
    return {"unpack": n * b / 8 + 4 * n, "fft_r2c": 8 * n, "rfi_s1": 12 * n, "dedisperse": 8 * n,
            "watfft": 8 * n, "rfi_s2": 4 * n, "signal_detect": 4 * n}


def hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# kernels of each per-pipe stage, for summing the ncu DRAM traffic of profiles/traffic.json
STAGE_KERNELS = {
    "unpack": r"^unpack_",
    "fft_r2c": r"^(fft_col(16)?_tma_kernel<.*, 0>|fft_trans(16)?_tma_kernel|fft_trans_r2c(16)?_tma_kernel|fft_pass_kernel|"
               r"r2c_post_kernel|r2c_col0_fixup_kernel)",
    "rfi_s1": r"^(power_sum_kernel|rfi_s1_apply_kernel|rfi_zero_ranges_kernel)",
    "dedisperse": r"^dedisperse_kernel<0>",
    "watfft": r"^fft_row(16)?_tma_kernel<.*, 0>$",
    "rfi_s2": r"^sk_kernel",
    "signal_detect": r"^(colsum_|detect_)",
}


def measured_dram_bytes_per_sample(wname: str):
    """DRAM bytes (read + write) of one fused block per input sample from the committed ncu capture of this workload
    (profiles/traffic_<workload>.json, written by tools/summarize_profiles.py), or None"""
    p = ROOT / "profiles" / f"traffic_{wname}.json"
    if not p.exists():
        return None
    try:
        d = json.loads(p.read_text())
        return float(d["block_dram_bytes"]) / float(d["block_samples"])
    except Exception:
        return None


def measured_kernel_traffic(wname: str, needle: tuple):
    """(mean DRAM read + write bytes per launch, mean ncu duration in us, kernel name) of the kernels of the committed
    capture whose name contains one of `needle`, or (None, None, None)"""
    p = ROOT / "profiles" / f"traffic_{wname}.json"
    try:
        ks = [k for k in json.loads(p.read_text())["kernels"] if any(nd in k["kernel"] for nd in needle)]
        if not ks:
            return None, None, None
        return (float(np.mean([k["dram_read"] + k["dram_write"] for k in ks])), float(np.mean([k["time_us"] for k in ks])),
                ks[0]["kernel"].split("(")[0])
    except Exception:
        return None, None, None


_NCU_US = {}   # per-stage sum of kernel durations in the same committed capture (no launch / event overhead)


def stage_traffic():
    """per-stage DRAM bytes (read + write) per launch from the committed ncu capture, or {}"""
    import re
    p = ROOT / "profiles" / "traffic.json"
    if not p.exists():
        return {}, None
    try:
        d = json.loads(p.read_text())
        out = {}
        seen_fused = False
        for k in d["kernels"]:
            # the capture ends with one fused process_block: stop at its first kernel (RAW first sweep)
            if re.search(r"fft_col(16)?_tma_kernel<.*, [12]>$", k["kernel"]):
                seen_fused = True
            if seen_fused:
                continue
            for stage, pat in STAGE_KERNELS.items():
                if re.search(pat, k["kernel"]):
                    out[stage] = out.get(stage, 0.0) + k["dram_read"] + k["dram_write"]
                    _NCU_US[stage] = _NCU_US.get(stage, 0.0) + k.get("time_us", 0.0)
        return out, d.get("tag")
    except Exception:
        return {}, None


def synth_block(n_samples: int, streams: int, seed: int, bits: int = -8) -> np.ndarray:
    """V1/V2-style synthetic voltage (SURVEY §8d): Gaussian sigma 20 + CW tone + a short burst,
    int8, clipped; multi-stream blocks are laid out by the caller. Sub-byte widths: uniform random
    packed samples (white noise)."""
    rng = np.random.default_rng(0x53525442 + seed)
    if abs(bits) < 8:
        return rng.integers(0, 256, n_samples * streams * abs(bits) // 8, dtype=np.uint8).view(np.int8)
    v = rng.standard_normal(n_samples * streams, dtype=np.float32) * 20.0
    t = np.arange(n_samples * streams, dtype=np.float32)
    v += 30.0 * np.cos(np.float32(2 * np.pi * 0.1185) * (t % 4096))
    mid = (n_samples * streams) // 2
    v[mid:mid + 2048] *= 4.0
    return np.clip(np.rint(v), -127, 127).astype(np.int8)


def dispersed_pulse(n: int, w: dict, amp: float = 1000.0, t0_frac: float = 0.37) -> np.ndarray:
    """float32 time series whose R2C spectrum is amp * conj(chirp) * delay(t0): dedispersion with the workload's DM
    folds it back into one impulse at sample t0 (the V3 "pulse" of SURVEY §8d). Per-sample amplitude is
    amp / sqrt(n) << 1 count: it rides on the noise as dither and survives the 8-bit quantisation statistically."""
    import scipy.fft as sfft
    nc = n // 2
    f_min, bw = np.float32(w["f_low"]), np.float32(w["bw"])
    f_c = float(np.float32(f_min + bw))
    df = float(np.float32(bw / np.float32(nc)))
    spec = np.zeros(nc + 1, np.complex64)
    step = min(nc, 1 << 18)                        # cache-sized chunks, buffers reused (fresh pages are slow here)
    t0 = int(n * t0_frac)
    k = np.empty(step, np.float64)
    f = np.empty(step, np.float64)
    g = np.empty(step, np.float64)
    base = np.arange(step, dtype=np.float64)
    cs = np.empty(step, np.complex128)
    c_dm = (4.148808e3 * 1e6) * float(np.float32(w["dm"]))
    for a in range(0, nc, step):
        np.add(base, float(a), out=k)
        np.multiply(k, df, out=f)
        f += float(f_min)                          # f = f_min + df * k
        np.subtract(f, f_c, out=g)
        g /= f_c
        g *= g
        g /= f
        g *= c_dm                                  # kk = D * dm / f * ((f - f_c) / f_c)^2
        g -= np.floor(g)
        k *= float(t0)
        np.fmod(k, float(n), out=k)
        k /= float(n)
        g -= k                                     # phase in cycles: +chirp (inverse of dedispersion), delay t0
        g *= 2 * np.pi
        cs.real = np.cos(g)
        cs.imag = np.sin(g)
        spec[a:a + step] = amp * cs
    return sfft.irfft(spec, n=n, workers=min(16, os.cpu_count() or 1)).astype(np.float32)


def synth_block_with_pulse(n: int, streams: int, seed: int, w: dict) -> np.ndarray:
    """synth_block plus the same dispersed pulse in every stream (8-bit formats only), re-quantised"""
    rng = np.random.default_rng(0x53525442 + seed)
    pulse = dispersed_pulse(n, w)
    out = np.empty(n * streams, np.int8)
    for s_ in range(streams):
        v = rng.standard_normal(n, dtype=np.float32) * 20.0 + pulse
        q = np.clip(np.rint(v), -127, 127).astype(np.int8)
        if streams == 1:
            out[:] = q
        elif w["fmt"] == "naocpsr_snap1":           # "1 1 2 2"
            out.reshape(-1, 4)[:, 2 * s_:2 * s_ + 2] = q.reshape(-1, 2)
        else:                                        # "1 2 1 2"
            out.reshape(-1, streams)[:, s_] = q
    return out


def bind_to_gpu_numa_node(torch, device_index: int):
    """Multi-rank runs: keep this rank's thread (and with it the pinned host blocks it allocates from now on) on the
    NUMA node its GPU hangs off — eight ranks pulling 55 GB/s each out of host memory otherwise depend on where the
    scheduler happened to start them (8 GPUs: 430 against 270 Gsamples/s end to end, profiles/r02t_scaling.md).
    Returns the node, or None when the topology cannot be read (nothing is changed then)."""
    try:
        pr = torch.cuda.get_device_properties(device_index)
        bus = "%04x:%02x:%02x.0" % (int(pr.pci_domain_id), int(pr.pci_bus_id), int(pr.pci_device_id))
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text().strip())
        if node < 0:
            return None
        cpus = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        target = cpus & set(os.sched_getaffinity(0))
        if len(target) < 2:
            return None
        os.sched_setaffinity(0, target)
        return node
    except Exception as e:  # unknown attribute names, no sysfs, restricted cpuset: run unbound
        print(f"[bench] NUMA binding skipped: {e}", file=sys.stderr)
        return None


class RankSync:
    """Plumbing between the ranks of one node. The default process group is NCCL, as the launch contract says, but it
    is created lazily and this path has no data-path collective, so NO NCCL communicator exists while blocks are timed:
    barriers and the max-over-ranks go through a gloo group on host scalars. (A communicator in the process costs the
    two-lane path up to 8 %: its streams take hardware work queues, profiles/r02s_connections.md.) NCCL is exercised
    once, after everything is measured, by close(). SRTB_BENCH_EAGER_NCCL=1 restores an eager communicator and NCCL
    barriers for comparison."""

    def __init__(self, dist_mod, torch, local_rank):
        self.d, self.torch = dist_mod, torch
        self.eager = os.environ.get("SRTB_BENCH_EAGER_NCCL") == "1"
        self.host_only = os.environ.get("SRTB_BENCH_SYNC_BACKEND") == "gloo"   # CPU tests of this class: no NCCL at all
        if self.eager:
            dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            self.group = None
        elif self.host_only:
            dist_mod.init_process_group("gloo")
            self.group = None
        else:
            dist_mod.init_process_group("nccl")
            self.group = dist_mod.new_group(backend="gloo")
        self.ReduceOp = dist_mod.ReduceOp

    def get_world_size(self):
        return self.d.get_world_size()

    def barrier(self):
        self.d.barrier(group=self.group) if self.group is not None else self.d.barrier()

    def all_gather_scalar(self, value: float):
        t = self.torch.tensor([value], dtype=self.torch.float64, device="cuda" if self.eager else "cpu")
        every = [self.torch.zeros_like(t) for _ in range(self.get_world_size())]
        self.d.all_gather(every, t, group=self.group)
        return [float(x.item()) for x in every]

    def all_reduce(self, t, op):
        if self.eager:
            self.d.all_reduce(t, op=op)
            return
        c = t.cpu()
        self.d.all_reduce(c, op=op, group=self.group)
        t.copy_(c)

    def destroy_process_group(self):
        if self.host_only:
            self.d.destroy_process_group()
            return
        # one NCCL collective over NVLink after the measurements: the ranks agree on the world size
        try:
            t = self.torch.ones(1, device="cuda")
            self.d.all_reduce(t)
            if int(t.item()) != self.get_world_size():
                print(f"[bench] NCCL all-reduce returned {t.item()} for world size {self.get_world_size()}", file=sys.stderr)
        except Exception as e:  # the measurements are already printed: report, do not fail the run
            print(f"[bench] closing NCCL collective failed: {e}", file=sys.stderr)
        self.d.destroy_process_group()


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def snapshot(self):
        """one immediate query (used when the timed region was shorter than the sampling period)"""
        try:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                  "-i", str(self.gpu_index)], capture_output=True, text=True, timeout=10).stdout
            for line in out.strip().splitlines():
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if not self.rows:
            self.snapshot()
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                                  ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def oracle_chain_config(w: dict, n: int, pairs):
    import oracle_lib
    oc = oracle_lib.ChainConfig()
    oc.baseband_input_count = n
    oc.baseband_input_bits = w["bits"]
    oc.window = 0
    oc.baseband_freq_low, oc.baseband_bandwidth = w["f_low"], w["bw"]
    oc.baseband_sample_rate, oc.dm = w["fs"], w["dm"]
    oc.baseband_reserve_sample = 0
    oc.rfi_average_threshold, oc.rfi_sk_threshold = w["avg_thr"], w["sk_thr"]
    oc.spectrum_channel_count = w["channels"]
    oc.snr_threshold, oc.channel_threshold = w["snr"], w["chan_thr"]
    oc.max_boxcar_length = w["maxbox"]
    flat = [v for p in pairs for v in p]
    arr = (C.c_float * max(1, len(flat)))(*flat)
    oc._keep = arr
    oc.rfi_pairs = C.cast(arr, C.POINTER(C.c_float))
    oc.n_rfi_pairs = len(pairs)
    return oc


_CPU_THREADS = None


def pick_cpu_threads(w: dict) -> int:
    """the box may expose more logical CPUs than the container may use: time a small block at a few
    thread counts once and keep the fastest ("all the host threads it can use")"""
    global _CPU_THREADS
    if _CPU_THREADS is not None:
        return _CPU_THREADS
    import oracle_lib
    o = oracle_lib.load()
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    cands = sorted({t for t in (avail, avail // 2, avail // 4, 32, 16, 8) if 1 <= t <= avail})
    cfg = oracle_chain_config(w, 1 << 20, [])
    blk = synth_block(1 << 20, 1, 7, w["bits"]).view(np.uint8)
    best, best_t = None, None
    for t in cands:
        o.set_threads(t)
        o.chain(blk, cfg)
        t0 = time.perf_counter()
        o.chain(blk, cfg)
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, best_t = dt, t
    o.set_threads(best_t)
    _CPU_THREADS = best_t
    return best_t


def cpu_chain_seconds(w: dict, n: int, reps: int, streams: int):
    """time the CPU oracle chain (restated reference operators, OpenMP) on `reps` blocks of n samples
    per stream. Multi-stream formats are timed as `streams` independent simple-format streams (the
    de-interleave is a negligible part of the CPU time)."""
    import oracle_lib
    o = oracle_lib.load()
    pick_cpu_threads(w)
    pairs = o.eval_rfi_ranges(w["freq_list"]) if w["freq_list"] else []
    cfg = oracle_chain_config(w, n, pairs)
    blocks = [synth_block(n, 1, 1000 + i, w["bits"]) for i in range(min(reps, 2))]
    t0 = time.perf_counter()
    stage = np.zeros(7)
    for i in range(reps):
        for _ in range(streams):
            _, _, _, st = o.chain(blocks[i % len(blocks)].view(np.uint8), cfg)
            stage += st
    dt = time.perf_counter() - t0
    return dt, o.num_threads(), (stage / reps).tolist()


def run_reference(args, w, wname):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    n = 1 << w["log2n"]
    streams = FORMAT_STREAM_COUNT[w["fmt"]]
    sample_n = min(n, 1 << 24)      # one step = one block of at most 2^24 samples per stream
    for _ in range(args.warmup):
        cpu_chain_seconds(w, min(sample_n, 1 << 20), 1, 1)
    dt, threads, stage = cpu_chain_seconds(w, sample_n, args.steps, streams)
    samples = sample_n * streams * args.steps
    value = samples / dt / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (fp64 chirp phase)",
        "data": "synthetic",
        "config": {"workload": workload_string(wname, w),
                   "sample": f"each step = one block of 2^{int(np.log2(sample_n))} samples/stream"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{args.steps} block(s) of 2^{int(np.log2(sample_n))} samples x{streams} "
                                   "stream(s); restated reference operators + naive radix-2 FFT "
                                   "(what srtb runs without FFTW), OpenMP",
                         "stage_seconds_per_block": dict(zip(STAGES, stage))},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(json.dumps(line))
    return 0


_RESULT_OUT = None


def claim_stdout():
    """Keep the process's stdout for the ONE JSON line: everything else that writes to fd 1 during the run (NCCL's
    version banner, library chatter) goes to stderr."""
    global _RESULT_OUT
    if _RESULT_OUT is None:
        sys.stdout.flush()
        _RESULT_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(text: str):
    out = _RESULT_OUT or sys.stdout
    out.write(text + "\n")
    out.flush()


def default_contexts(w: dict) -> int:
    """contexts (CUDA streams) per GPU that blocks alternate over: short blocks leave gaps between their kernels that
    other blocks fill; long sweeps are pure HBM streams with little left to overlap"""
    if FORMAT_STREAM_COUNT[w["fmt"]] >= 2 and w["log2n"] >= 26:
        return 1  # a context spreads the streams of a block over two lanes itself: more contexts add nothing here
    return 6 if w["log2n"] <= 24 else (4 if w["log2n"] < 28 else 2)


class Harness:
    """one workload on this rank's GPU: contexts, ring of distinct synthetic blocks (host pinned + device copies),
    device-resident and end-to-end stepping through the ring API"""

    def __init__(self, torch, srtb_b200, wname, w, n_contexts, rank, local_rank, inject_pulse):
        self.torch, self.srtb = torch, srtb_b200
        self.wname, self.w = wname, w
        self.n = 1 << w["log2n"]
        self.fmt = srtb_b200.FORMAT_BY_NAME[w["fmt"]]
        self.streams = srtb_b200.FORMAT_STREAMS[self.fmt]
        self.block_bytes = self.n * self.streams * abs(w["bits"]) // 8
        self.ring = max(2, min(16, (288 << 20) // self.block_bytes))      # > L2 (126 MB) of distinct input
        self.stream = torch.cuda.current_stream()
        self.extra_streams = [torch.cuda.Stream() for _ in range(max(0, n_contexts - 1))]
        self.ctxs = [srtb_b200.Context(local_rank, self.stream.cuda_stream)] + \
                    [srtb_b200.Context(local_rank, st.cuda_stream) for st in self.extra_streams]
        self.pairs = srtb_b200.eval_rfi_ranges(w["freq_list"]) if w["freq_list"] else []
        cfg = srtb_b200.BlockConfig()
        cfg.baseband_input_count = self.n
        cfg.baseband_input_bits = w["bits"]
        cfg.baseband_format = self.fmt
        cfg.window = 0
        cfg.baseband_reserve_sample = 0
        cfg.baseband_freq_low, cfg.baseband_bandwidth = w["f_low"], w["bw"]
        cfg.baseband_sample_rate, cfg.dm = w["fs"], w["dm"]
        cfg.mitigate_rfi_average_method_threshold = w["avg_thr"]
        cfg.mitigate_rfi_spectral_kurtosis_threshold = w["sk_thr"]
        cfg.spectrum_channel_count = w["channels"]
        cfg.signal_detect_signal_noise_threshold = w["snr"]
        cfg.signal_detect_channel_threshold = w["chan_thr"]
        cfg.signal_detect_max_boxcar_length = w["maxbox"]
        flat = [v for p_ in self.pairs for v in p_]
        self._arr = (C.c_float * max(1, len(flat)))(*flat)
        cfg.rfi_freq_pairs = C.cast(self._arr, C.POINTER(C.c_float))
        cfg.n_rfi_freq_pairs = len(self.pairs)
        self.cfg = cfg
        # synthetic blocks: distinct per rank and per ring slot; every second one carries a dispersed pulse
        self.host_blocks, self.pulse_blocks = [], 0
        for i in range(self.ring):
            if inject_pulse and abs(w["bits"]) == 8 and i % 2 == 0:
                b = synth_block_with_pulse(self.n, self.streams, seed=rank * 1000 + i, w=w)
                self.pulse_blocks += 1
            else:
                b = synth_block(self.n, self.streams, seed=rank * 1000 + i, bits=w["bits"])
            self.host_blocks.append(torch.from_numpy(b.view(np.uint8)).pin_memory())
        self.dev_blocks = [hb.cuda(non_blocking=True) for hb in self.host_blocks]
        torch.cuda.synchronize()
        self.detections = 0
        self.blocks_with_detection = 0
        self._tickets = []
        self.last_block = None

    def close(self):
        for c in self.ctxs:
            c.close()

    @property
    def launch_count(self):
        return sum(c.launch_count for c in self.ctxs)

    def _collect(self):
        c, t = self._tickets.pop(0)
        res, h_series, d_spectra = c.collect_block_ex(t)
        self.last_block = (res, h_series, d_spectra)   # ring-slot buffers: valid until the slot is submitted again
        found = sum(int(r.signal_count[b]) for r in res for b in range(r.n_boxcars))
        self.detections += found
        self.blocks_with_detection += 1 if found else 0

    def step_device(self, i):
        c = self.ctxs[i % len(self.ctxs)]
        self._tickets.append((c, c.submit_block_device(self.cfg, self.dev_blocks[i % self.ring], self.block_bytes)))
        if len(self._tickets) >= 2 * len(self.ctxs):
            self._collect()

    def step_e2e(self, i):
        c = self.ctxs[i % len(self.ctxs)]
        self._tickets.append((c, c.submit_block(self.cfg, self.host_blocks[i % self.ring], self.block_bytes)))
        if len(self._tickets) >= 2 * len(self.ctxs):
            self._collect()

    def drain(self):
        while self._tickets:
            self._collect()

    def timed(self, fn, steps, dist):
        """K steps between two CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks"""
        torch = self.torch

        def barrier():
            torch.cuda.synchronize()
            if dist:
                dist.barrier()
            torch.cuda.synchronize()

        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for st in self.extra_streams:
            st.wait_stream(self.stream)
        for i in range(steps):
            fn(i)
        self.drain()
        for st in self.extra_streams:
            self.stream.wait_stream(st)
        e1.record(self.stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        self.last_ms_by_rank = [ms]
        if dist:
            self.last_ms_by_rank = dist.all_gather_scalar(ms)   # the reported time is the slowest rank's
            ms = max(self.last_ms_by_rank)
        barrier()
        return ms

    def warm(self, fn, warmup):
        # at least W steps, and enough that EVERY context has seen every ring slot once (first use allocates scratch,
        # builds twiddle tables and sets kernel attributes: cudaMalloc would stall the timed region)
        warm = max(warmup, (SRTB_RING_SLOTS + 1) * len(self.ctxs))
        for i in range(warm):
            fn(i)
        self.drain()
        return warm


DUMP_SPECTRUM_SAMPLES = 1 << 20   # per stream: 8 MiB of the 256 MiB dynamic spectrum of a config3 stream
DUMP_SEED = 0x53525442


class _LibraryDeviceFloats:
    """a float32 device buffer owned by libsrtb_b200, seen by torch without a copy"""

    def __init__(self, ptr: int, count: int):
        self.__cuda_array_interface__ = {"shape": (count,), "typestr": "<f4", "data": (ptr, False), "version": 2}


def dump_block_outputs(out_dir: str, torch, srtb_b200, H):
    """Writes what collect_block_ex hands the caller for the last block the timed loop collected, as .npy files:
    per stream the detector result (entries past n_boxcars zeroed), the boxcar series it marked positive
    ([stream][boxcar][L], zero elsewhere) and a fixed seeded sample of the dynamic spectrum [C][L] (complex64 as
    float32 pairs, at the flat indices in spectrum_sample_index). 28 MiB for config3. The blocks are seeded, so the
    same arguments dump the same outputs from any build."""
    res, h_series, d_spectra = H.last_block
    streams, mb = len(res), srtb_b200.MAX_BOXCARS
    nc = H.n // 2
    L = nc // min(H.w["channels"], nc)
    fields = {k: np.zeros((streams, mb), np.float64) for k in ("boxcar_length", "series_length", "signal_count")}
    fields.update({k: np.zeros((streams, mb), np.float32) for k in ("variance", "threshold")})
    summary = np.zeros((streams, 4), np.float64)
    series = np.zeros((streams, mb, L), np.float32)
    host_series = np.ctypeslib.as_array(C.cast(h_series, C.POINTER(C.c_float)), shape=(streams, mb, L))
    for s, r in enumerate(res):
        nb = r.n_boxcars
        summary[s] = (r.zero_count, r.time_series_count, r.detect_enabled, nb)
        for k, a in fields.items():
            a[s, :nb] = getattr(r, k)[:nb]
        for b in range(nb):
            if r.signal_count[b] > 0:
                series[s, b, :r.series_length[b]] = host_series[s, b, :r.series_length[b]]
    count = min(nc, DUMP_SPECTRUM_SAMPLES)
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(nc, count, replace=False))
    d_idx = torch.from_numpy(idx).cuda()
    spectrum = np.stack([torch.as_tensor(_LibraryDeviceFloats(d_spectra[s], 2 * nc), device="cuda").view(nc, 2)[d_idx]
                         .cpu().numpy() for s in range(streams)])
    os.makedirs(out_dir, exist_ok=True)
    arrays = dict(detect_summary=summary, series=series, spectrum_sample=spectrum,
                  spectrum_sample_index=idx.astype(np.float64), **fields)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def run_dm_sweep(args, torch, srtb_b200, w, wname, rank, local_rank, world, dist):
    """BASELINE config #4: one 2^27-sample block per step, 21 trial DMs each (unpack + R2C once, then s1 + chirp ->
    waterfall -> SK -> detector per DM: srtb_b200_process_block_dm_sweep). Blocks are sharded over the ranks; block 0
    of the ring carries a Crab-like pulse dispersed at DM 56.78, so the trial nearest to it must light up."""
    H = Harness(torch, srtb_b200, wname, w, 1, rank, local_rank, inject_pulse=True)
    ctx, dms = H.ctxs[0], w["dms"]
    by_dm = np.zeros(len(dms), np.int64)

    def step(i, host):
        blk = (H.host_blocks if host else H.dev_blocks)[i % H.ring]
        res = ctx.process_block_dm_sweep(H.cfg, blk, H.block_bytes, dms, on_device=not host)
        for j, per_stream in enumerate(res):
            by_dm[j] += sum(int(r.signal_count[b]) for r in per_stream for b in range(r.n_boxcars))

    for i in range(max(args.warmup, 3)):
        step(i, False)
    steps = args.steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    by_dm[:] = 0
    l0 = H.launch_count
    ms = H.timed(lambda i: step(i, False), steps, dist) / steps
    launches = H.launch_count - l0
    found = by_dm.copy()
    for i in range(3):
        step(i, True)
    ms_e2e = float(np.median([H.timed(lambda i: step(i, True), steps, dist) / steps for _ in range(3)]))
    clocks = sampler.stop() if rank == 0 else None
    sps = H.n * H.streams * world
    if rank == 0:
        peak, peak_src = hbm_peak()
        line = {
            "metric": METRIC, "value": sps / (ms * 1e-3) / 1e9, "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (fp64 chirp phase)", "data": "synthetic",
            "config": {"workload": workload_string(wname, w) + f", {len(dms)} trial DMs 0..{dms[-1]:g} per block",
                       "parallelism": f"block-sharded x{world} (no collective)",
                       "l2": f"inputs larger than L2: ring of {H.ring} distinct blocks ({H.ring * H.block_bytes >> 20} MiB)",
                       "contexts_per_gpu": 1, "dm_trials": len(dms),
                       "dm_trial_gsamples_per_s": sps * len(dms) / (ms * 1e-3) / 1e9,
                       "detections_by_dm": {f"{d:g}": int(c) for d, c in zip(dms, found)},
                       "injected_pulse": "DM 56.78 in every second block"},
            "clocks": clocks,
            "e2e": {"value": sps / (ms_e2e * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": H.block_bytes * world,
                    "d2h_bytes_per_step": C.sizeof(srtb_b200.DetectResult) * H.streams * len(dms) * world},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                         "note": "sweep bytes: raw-fused R2C once per block (21 bytes per sample), then per trial the long-row "
                                 "group: chirp-on-load column sweep 8 + last sweep 8 + zap-aware column sums 4",
                         "bytes_per_sample": sweep_bytes_per_sample(w),
                         "achieved": sweep_bytes_per_sample(w) * H.n / (ms * 1e-3) / 1e9,
                         "frac": sweep_bytes_per_sample(w) * H.n / (ms * 1e-3) / 1e9 / peak},
            "cpu_baseline": None,
        }
        emit(json.dumps(line))
    H.close()
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_udp_stream(args, torch, w, wname, rank, local_rank, world, dist):
    """BASELINE config #5: a continuous UDP-shaped stream (fastmb_roach2 packets: 8-byte counter + 4096 samples) at
    1 Gsample/s per GPU for >= 10 s through the product executable (src/srtb_b200: paced packet source -> counter-keyed
    block assembler into pinned host memory -> H2D ring -> fused chain -> detector), one process per GPU. Reported:
    achieved rate, lost packets (a consumer that falls more than 64 MiB behind loses packets like a socket would), and
    the unpaced rate the same path sustains."""
    exe = ROOT / "src" / "srtb_b200"
    if not exe.exists():
        raise SystemExit(f"bench.py: {exe} not built: run __graft_entry__.build() first")

    def run(rate, seconds):
        cmd = [str(exe), "--config_file_name", "/nonexistent.cfg", "--gpu_devices", str(local_rank), "--chains_per_gpu", "2",
               "--ring_depth", "3", "--discard_output", "1", "--synthetic_udp_rate", repr(float(rate)),
               "--synthetic_duration", repr(float(seconds)), "--baseband_input_count", f"2 ** {w['log2n']}",
               "--baseband_input_bits", str(w["bits"]), "--baseband_format_type", "fastmb_roach2",
               "--baseband_freq_low", str(w["f_low"]), "--baseband_bandwidth", str(w["bw"]),
               "--baseband_sample_rate", repr(float(w["fs"])), "--dm", str(w["dm"]), "--baseband_reserve_sample", "0",
               "--spectrum_channel_count", str(w["channels"]), "--mitigate_rfi_average_method_threshold", str(w["avg_thr"]),
               "--mitigate_rfi_spectral_kurtosis_threshold", str(w["sk_thr"]),
               "--signal_detect_signal_noise_threshold", str(w["snr"]), "--signal_detect_max_boxcar_length", str(w["maxbox"]),
               "--log_level", "2"]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        if r.returncode != 0:
            raise SystemExit(f"srtb_b200 failed: {r.stderr[-1500:]}")
        return json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])

    if dist:
        dist.barrier()
    live = run(w["rate_per_gpu"], w["seconds"])
    if dist:
        dist.barrier()
    fast = run(0.0, 4.0)
    vals = torch.tensor([live["gsamples_per_s"], float(live["lost_packets"]), float(live["received_packets"]),
                         float(live["blocks"]), fast["gsamples_per_s"], live["seconds"]], dtype=torch.float64, device="cuda")
    if dist:
        mx = vals.clone()
        dist.all_reduce(vals, op=dist.ReduceOp.SUM)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        seconds = float(mx[5])
    else:
        seconds = float(vals[5])
    if rank == 0:
        v = vals.cpu().numpy()
        n = 1 << w["log2n"]
        line = {
            "metric": METRIC, "value": float(v[0]), "unit": UNIT, "n_gpus": world, "steps": int(v[3]), "warmup": 0,
            "ms_per_step": seconds * 1e3 / max(1.0, v[3] / world), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (fp64 chirp phase)", "data": "synthetic",
            "config": {"workload": workload_string(wname, w) + ", UDP-shaped live stream",
                       "parallelism": f"one receiver + fused chain per GPU x{world} (no collective)",
                       "target_gsamples_per_s": w["rate_per_gpu"] * world / 1e9, "stream_seconds": seconds,
                       "lost_packets": int(v[1]), "received_packets": int(v[2]),
                       "real_time": bool(v[1] == 0 and v[0] > 0.97 * w["rate_per_gpu"] * world / 1e9),
                       "max_sustained_gsamples_per_s": float(v[4]),
                       "note": "timed by the host clock of the paced source (a live stream has no device-resident form)"},
            "clocks": None,
            "e2e": {"value": float(v[0]), "unit": UNIT, "h2d_bytes_per_step": n * world, "d2h_bytes_per_step": 1048 * world},
            "gpu_launches": int(v[3]) * 9,
            "cpu_baseline": None,
        }
        emit(json.dumps(line))
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default=os.environ.get("SRTB_BENCH_WORKLOAD", "config3"))
    ap.add_argument("--secondary", default=os.environ.get("SRTB_BENCH_SECONDARY", "config2"),
                    help="second workload measured briefly (value + e2e) in the same line; 'none' skips it")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pulse", action="store_true", help="noise-only blocks (no injected dispersed pulse)")
    ap.add_argument("--stage-iters", type=int, default=5)
    ap.add_argument("--contexts", type=int, default=int(os.environ.get("SRTB_BENCH_CONTEXTS", "0")),
                    help="contexts per GPU that blocks alternate over (0 = 1 for multi-stream blocks of >= 2^26 samples, whose "
                         "streams the context overlaps itself; else 6 up to 2^24-sample blocks, 4 up to 2^27, 2 above)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0; "
                         "workloads config1..config3)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload in ("config4", "config5")):
        ap.error("--dump-outputs covers the block-ring path of workloads config1..config3")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    wname = args.workload
    w = WORKLOADS[wname]
    if args.impl == "reference":
        return run_reference(args, w, wname)

    import torch
    import srtb_b200

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    numa_node = bind_to_gpu_numa_node(torch, local_rank) if world > 1 and args.impl != "reference" else None
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = RankSync(dist_mod, torch, local_rank)

    if wname == "config4":
        return run_dm_sweep(args, torch, srtb_b200, w, wname, rank, local_rank, world, dist)
    if wname == "config5":
        return run_udp_stream(args, torch, w, wname, rank, local_rank, world, dist)

    n_ctx = args.contexts if args.contexts > 0 else default_contexts(w)
    H = Harness(torch, srtb_b200, wname, w, n_ctx, rank, local_rank, inject_pulse=not args.no_pulse)
    n, streams, block_bytes, ring = H.n, H.streams, H.block_bytes, H.ring
    ctx, stream = H.ctxs[0], H.stream
    samples_per_step = n * streams * world

    # ---- device-resident throughput (`value`)
    warm = H.warm(H.step_device, args.warmup)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = H.launch_count
    H.detections = H.blocks_with_detection = 0
    ms_total = H.timed(H.step_device, args.steps, dist)
    ms_by_rank = [m / args.steps for m in H.last_ms_by_rank]
    launches = H.launch_count - l0
    detections, det_blocks = H.detections, H.blocks_with_detection
    if rank == 0 and not sampler.rows:
        sampler.snapshot()          # short run: take one sample while the GPU is still under load
    ms_per_step = ms_total / args.steps
    value = samples_per_step / (ms_per_step * 1e-3) / 1e9
    if args.dump_outputs and rank == 0:
        dump_block_outputs(args.dump_outputs, torch, srtb_b200, H)

    # ---- end to end from pinned host memory (`e2e`)
    H.warm(H.step_e2e, args.warmup)
    e2e_runs = [H.timed(H.step_e2e, args.steps, dist) / args.steps for _ in range(3)]
    ms_e2e = float(np.median(e2e_runs))           # host-side jitter (PCIe, the feeding thread): median of three
    clocks = sampler.stop() if rank == 0 else None
    e2e_value = samples_per_step / (ms_e2e * 1e-3) / 1e9
    series_bytes = 0                               # positive series written by the detector kernel: rare, small
    d2h = C.sizeof(srtb_b200.DetectResult) * streams + series_bytes

    # ---- the same through ONE context (one CUDA stream per GPU, as the reference drives its device)
    single = None
    if len(H.ctxs) > 1:
        extra, H.ctxs, H.extra_streams = (H.ctxs[1:], H.extra_streams), H.ctxs[:1], []
        H.warm(H.step_device, args.warmup)
        ms1 = H.timed(H.step_device, args.steps, dist) / args.steps
        single = {"value": samples_per_step / (ms1 * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms1, "contexts_per_gpu": 1}
        H.ctxs, H.extra_streams = H.ctxs + extra[0], extra[1]
    else:
        single = {"value": value, "unit": UNIT, "ms_per_step": ms_per_step, "contexts_per_gpu": 1}

    # ---- per-stage CUDA-event timing (rank 0): each stage called through the C ABI on one stream's data
    stages, fused = {}, {}
    roofline = None
    if rank == 0:
        peak, peak_src = hbm_peak()
        bytes_per = stage_bytes(n, w["bits"])
        nc = n // 2
        batch = min(w["channels"], nc)
        L = nc // batch
        pairs = H.pairs
        coef = srtb_b200.norm_coefficient(nc, w["channels"])
        bins = [r for r in (srtb_b200.rfi_range_to_bins(a, b, w["f_low"], w["bw"], nc) for a, b in pairs) if r]
        f_min, bw = np.float32(w["f_low"]), np.float32(w["bw"])
        f_c, df = float(f_min + bw), float(bw / np.float32(nc))
        outs = [torch.empty(n + 2, dtype=torch.float32, device="cuda") for _ in range(streams)]
        buf = outs[0]
        fmt, dev_blocks = H.fmt, H.dev_blocks
        calls = {
            "unpack": lambda i: ctx.unpack(dev_blocks[i % ring], block_bytes, w["bits"], fmt, 0, outs, n),
            "fft_r2c": lambda i: ctx.fft_r2c_inplace(buf, n),
            "rfi_s1": lambda i: ctx.rfi_s1(buf, nc, w["avg_thr"], coef, bins),
            "dedisperse": lambda i: ctx.dedisperse(buf, nc, float(f_min), f_c, df, w["dm"]),
            "watfft": lambda i: ctx.watfft_c2c_backward(buf, L, batch),
            "rfi_s2": lambda i: ctx.rfi_s2_sk(buf, L, batch, w["sk_thr"]),
            "signal_detect": lambda i: ctx.signal_detect(buf, L, batch, 0, w["snr"], w["chan_thr"], w["maxbox"]),
        }
        flush = torch.empty(192 << 20, dtype=torch.uint8, device="cuda")
        for idx, name in enumerate(STAGES):
            times = []
            for it in range(args.stage_iters + 1):
                for prev in STAGES[:idx]:           # realistic input: run the chain up to this stage
                    calls[prev](it)
                flush.fill_(it & 0xFF)              # flush L2 between timed launches
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                calls[name](it)
                e1.record(stream)
                torch.cuda.synchronize()
                if it > 0:
                    times.append(e0.elapsed_time(e1))
            ms = float(np.mean(times))
            per_call_streams = streams if name == "unpack" else 1
            gbs = bytes_per[name] * per_call_streams / (ms * 1e-3) / 1e9
            stages[name] = {"ms": ms, "bytes": bytes_per[name] * per_call_streams, "gbs": gbs, "frac": gbs / peak}
        # ---- the kernel groups the block path really launches (last stream of a block), L2 flushed before each block,
        # timed by CUDA events inside the library on the launching stream, against the bytes each group must move
        ctx.stage_stats_enable(True)
        acc = {k: [] for k in ("r2c", "waterfall", "detect_tail")}
        grp_bytes = {}
        for it in range(args.stage_iters + 1):
            flush.fill_(it & 0xFF)
            t_ = ctx.submit_block_device(H.cfg, dev_blocks[it % ring], block_bytes)
            ctx.collect_block(t_)
            if it == 0:
                continue
            for key, sid in (("r2c", 7), ("waterfall", 8), ("detect_tail", 9)):
                try:
                    ms_, b_ = ctx.stage_stats(sid)
                    acc[key].append(ms_)
                    grp_bytes[key] = b_
                except Exception:
                    pass
        ctx.stage_stats_enable(False)
        for key, v_ in acc.items():
            if v_:
                ms_ = float(np.mean(v_))
                gbs = grp_bytes[key] / (ms_ * 1e-3) / 1e9
                fused[key] = {"ms": ms_, "compulsory_bytes": grp_bytes[key], "gbs": gbs, "frac": gbs / peak}
        dom = max((s_ for s_ in STAGES), key=lambda s_: stages[s_]["ms"])
        traffic, traffic_tag = stage_traffic() if wname == "config2" else ({}, None)
        for k_, v_ in traffic.items():
            if k_ in stages:
                stages[k_]["dram_traffic"] = v_
                if _NCU_US.get(k_):   # offline: kernel time under ncu (cold cache), for comparison with the live `ms`
                    stages[k_]["ncu_kernel_us"] = _NCU_US[k_]
                    stages[k_]["ncu_frac"] = stages[k_]["bytes"] / (_NCU_US[k_] * 1e-6) / 1e9 / peak
        # chain: three byte counts, each with its own fraction of the copy peak at the measured block time
        per_sample_s = ms_per_step * 1e-3 / (n * streams)
        unfused_bps = sum(bytes_per.values()) / n
        sweep_bps = sweep_bytes_per_sample(w)
        dram_bps = measured_dram_bytes_per_sample(wname)
        chain = {
            "algorithmic_unfused": {"bytes_per_sample": unfused_bps, "gbs": unfused_bps / per_sample_s / 1e9,
                                    "frac": unfused_bps / per_sample_s / 1e9 / peak,
                                    "note": "SURVEY 8d per-pipe bytes: what the chain would move pipe by pipe; a fused chain "
                                            "can exceed 1.0 of this, it is not a roofline fraction"},
            "sweep_bytes": {"bytes_per_sample": sweep_bps, "gbs": sweep_bps / per_sample_s / 1e9,
                            "frac": sweep_bps / per_sample_s / 1e9 / peak,
                            "note": "what the launched kernels must read + write (each sweep once)"},
            "dram_measured": None if dram_bps is None else {
                "bytes_per_sample": dram_bps, "gbs": dram_bps / per_sample_s / 1e9,
                "frac": dram_bps / per_sample_s / 1e9 / peak,
                "note": "ncu dram__bytes_read + write of one process_block at this workload (profiles/)"},
        }
        if fused.get("waterfall"):
            # the dominant kernel of the block path: the one-kernel waterfall group (s1 + chirp + waterfall FFT + SK +
            # column sums) — its compulsory bytes per launch over its launch time, measured above with CUDA events
            # inside the library; DRAM traffic per launch from the committed ncu capture of the same workload
            kt, kus, kname = measured_kernel_traffic(wname, ("fft_bigrow_kernel", "fft_row16_tma_kernel"))
            group_ms = sum(v_["ms"] for v_ in fused.values())
            roofline = {"bound": "hbm", "kernel": kname or "waterfall kernel (s1 + chirp + FFT + SK + column sums)",
                        "achieved": fused["waterfall"]["gbs"], "peak": peak, "unit": "GB/s",
                        "frac": fused["waterfall"]["frac"], "bytes_per_launch": fused["waterfall"]["compulsory_bytes"],
                        "ms_per_launch": fused["waterfall"]["ms"], "share_of_stream_time": fused["waterfall"]["ms"] / group_ms,
                        "traffic": kt, "ncu_us_per_launch": kus,
                        "traffic_source": (f"profiles/traffic_{wname}.json (ncu dram__bytes_read.sum + dram__bytes_write.sum, "
                                           "mean per launch)") if kt else None,
                        "peak_source": peak_src, "per_pipe_dominant": {"stage": dom, **stages[dom]}, "fused": fused,
                        "chain": chain}
        else:
            roofline = {"bound": "hbm", "kernel": dom, "achieved": stages[dom]["gbs"], "peak": peak,
                        "unit": "GB/s", "frac": stages[dom]["frac"], "traffic": traffic.get(dom),
                        "traffic_source": (f"ncu --set full capture profiles/{traffic_tag}_summary.md (dram read+write of the "
                                           "stage's kernels, one launch each, L2 flushed)") if traffic_tag else None,
                        "peak_source": peak_src, "fused": fused, "chain": chain}

    # ---- secondary workload (BASELINE configs[1]) in brief: value + e2e
    secondary = None
    if args.secondary not in ("none", "", wname) and args.secondary in WORKLOADS:
        H.close()
        del H
        torch.cuda.empty_cache()
        w2 = WORKLOADS[args.secondary]
        H2 = Harness(torch, srtb_b200, args.secondary, w2, default_contexts(w2), rank, local_rank, inject_pulse=False)
        steps2 = args.steps
        H2.warm(H2.step_device, args.warmup)
        ms2 = H2.timed(H2.step_device, steps2, dist) / steps2
        H2.warm(H2.step_e2e, args.warmup)
        ms2e = float(np.median([H2.timed(H2.step_e2e, steps2, dist) / steps2 for _ in range(3)]))
        sps2 = H2.n * H2.streams * world
        secondary = {"workload": workload_string(args.secondary, w2), "value": sps2 / (ms2 * 1e-3) / 1e9, "unit": UNIT,
                     "ms_per_step": ms2, "steps": steps2, "contexts_per_gpu": len(H2.ctxs),
                     "e2e": {"value": sps2 / (ms2e * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms2e,
                             "h2d_bytes_per_step": H2.block_bytes * world},
                     "sweep_bytes_per_sample": sweep_bytes_per_sample(w2)}
        H2.close()
        n_ctx_used = n_ctx
    else:
        n_ctx_used = n_ctx
        H.close()

    # ---- CPU baseline (oracle port) on a bounded sample of the same workload
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            sample_n = min(n, 1 << 24)
            cpu_chain_seconds(w, 1 << 18, 1, 1)        # warm the OpenMP pool
            dt, threads, stage = cpu_chain_seconds(w, sample_n, 2, streams)
            cpu_baseline = {"value": sample_n * streams * 2 / dt / 1e9, "unit": UNIT, "cores": threads,
                            "kind": "port",
                            "sample": f"2 blocks of 2^{int(np.log2(sample_n))} samples x{streams} stream(s) of "
                                      "this workload; restated reference operators with the in-tree naive "
                                      "radix-2 FFT, OpenMP over all host cores",
                            "stage_seconds_per_block": dict(zip(STAGES, stage))}
        except Exception as e:  # the oracle is test infrastructure: report, never fail the bench
            cpu_baseline = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (fp64 chirp phase)", "data": "synthetic",
            "config": {"workload": workload_string(wname, w),
                       "parallelism": f"block-sharded x{world} (no collective)",
                       "l2": f"inputs larger than L2: ring of {ring} distinct blocks ({ring * block_bytes >> 20} MiB)",
                       "contexts_per_gpu": n_ctx_used, "warmup_steps_run": warm,
                       "ms_per_step_by_rank": [round(m, 4) for m in ms_by_rank],
                       "rank0_numa_node": numa_node,
                       "injected_pulse": "every second block of the ring carries a dispersed pulse (S/N ~ 25)" if not args.no_pulse else "none",
                       "detections": detections, "blocks_with_detection": det_blocks},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e,
                    "runs_ms_per_step": e2e_runs, "note": "median of three runs of K steps each",
                    "h2d_bytes_per_step": block_bytes * world, "d2h_bytes_per_step": d2h * world},
            "gpu_launches": launches,
            "single_context": single,
            "secondary": secondary,
            "roofline": roofline,
            "stages": stages,
            "cpu_baseline": cpu_baseline,
        }
        emit(json.dumps(line))
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
