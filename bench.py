#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 phase-rotation backend.

Metric (BASELINE.json): Gsample-angles/s of the min-peak theta sweep.
Workload at N=1 (north_star target): stereo 48 kHz, 1 hour of synthetic
programme material, 0.1 degree grid (subsample 10 -> 1800 angles on [0, 180)),
digital peak, CLI block size 8192 — one "step" is one whole-file analysis pass
(the reference's analyze_file(), cli/phase-rotate.cc:565-587).
sample-angles per step = frames x channels x angles.

  value : input already resident in HBM (interleaved float32), CUDA events on
          the launching stream, K steps, max over ranks
  e2e   : the same pass through the C ABI with a pinned HOST buffer
          (phaserot_sweep): H2D of the whole file and D2H of the peak table
          inside the timed region
  roofline : the dominant kernel (FFT convolution + filter) timed live with
          CUDA events around every launch; achieved = 4 B/sample algorithmic
          bytes / kernel time, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline : the reference's own analysis code (oracle/_ref, unmodified
          sources + stand-in FFT) on the host cores, bounded sample

N > 1 (torchrun): weak scaling by sample range — every rank sweeps its own
1-hour shard of an N-hour stream (halo = one block of history), then one NCCL
max all-reduce over the [channels x angles] peak table.

`--impl reference` runs only the reference CPU arm with the same JSON shape.

`--dump-outputs DIR` writes what the last timed step returned to its caller -
the combined peak table of phaserot_peaks, [channels x 180 * subsample] float32:
index 0 the raw input peak, index i the peak at i / subsample degrees - as
DIR/peaks.npy.  The inputs are generated from fixed seeds, so two builds run
with the same arguments can be compared table for table.  Only the GPU arm has
this output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR = 48000
CHANNELS = 2
BLKSIZ = 8192
SUBSAMPLE = 10
GEN_CHUNK = 1 << 21  # frames per generator chunk (absolute-index aligned)
N_PARTIALS = 16


# ---------------------------------------------------------------------------
# synthetic programme material: 16 random-phase partials (1/f), slow AM, noise
# ---------------------------------------------------------------------------

def _partials(seed, channels=CHANNELS, n_partials=N_PARTIALS):
    rng = np.random.default_rng(seed)
    f = np.exp(rng.uniform(np.log(50.0), np.log(15000.0), (channels, n_partials)))
    ph = rng.uniform(0, 1.0, (channels, n_partials))
    amp = 50.0 / f
    amp /= amp.sum(axis=1, keepdims=True)
    return f, ph, amp


def gen_chunk_torch(torch, chunk_id, device, seed=43, channels=CHANNELS, sr=SR, n_partials=N_PARTIALS):
    """Frames [chunk_id*GEN_CHUNK, (chunk_id+1)*GEN_CHUNK) -> [GEN_CHUNK, channels] float32 on `device`."""
    f, ph, amp = _partials(seed, channels, n_partials)
    t = torch.arange(chunk_id * GEN_CHUNK, (chunk_id + 1) * GEN_CHUNK, device=device, dtype=torch.float64) / sr
    out = torch.empty((GEN_CHUNK, channels), device=device, dtype=torch.float32)
    g = torch.Generator(device=device)
    g.manual_seed(seed * 1000003 + chunk_id)
    for c in range(channels):
        acc = torch.zeros(GEN_CHUNK, device=device, dtype=torch.float32)
        for k in range(n_partials):
            frac = torch.frac(t * float(f[c, k]) + float(ph[c, k])).to(torch.float32)
            acc += float(amp[c, k]) * torch.sin(frac * (2.0 * np.pi))
        env = 0.6 + 0.4 * torch.sin((torch.frac(t * 0.37) * (2.0 * np.pi)).to(torch.float32) + float(c))
        noise = torch.randn(GEN_CHUNK, device=device, dtype=torch.float32, generator=g)
        out[:, c] = 0.8 * acc * env + 0.02 * noise
    return out


def gen_range_torch(torch, f0, f1, device, **kw):
    """Frames [f0, f1) of the synthetic stream (any alignment), built from whole generator chunks."""
    k0, k1 = f0 // GEN_CHUNK, (f1 + GEN_CHUNK - 1) // GEN_CHUNK
    ch = kw.get("channels", CHANNELS)
    out = torch.empty((f1 - f0, ch), device=device, dtype=torch.float32)
    for k in range(k0, k1):
        c = gen_chunk_torch(torch, k, device, **kw)
        lo, hi = max(f0, k * GEN_CHUNK), min(f1, (k + 1) * GEN_CHUNK)
        out[lo - f0:hi - f0] = c[lo - k * GEN_CHUNK:hi - k * GEN_CHUNK]
        del c
    return out


def gen_numpy(n_frames, seed=43):
    """CPU twin of the generator for the reference arm (same recipe; noise stream differs)."""
    f, ph, amp = _partials(seed)
    t = np.arange(n_frames, dtype=np.float64) / SR
    rng = np.random.default_rng(seed)
    out = np.empty((n_frames, CHANNELS), np.float32)
    for c in range(CHANNELS):
        acc = np.zeros(n_frames)
        for k in range(N_PARTIALS):
            acc += amp[c, k] * np.sin(2 * np.pi * ((t * f[c, k] + ph[c, k]) % 1.0))
        env = 0.6 + 0.4 * np.sin(2 * np.pi * ((t * 0.37) % 1.0) + c)
        out[:, c] = 0.8 * acc * env + 0.02 * rng.standard_normal(n_frames)
    return out


# ---------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------

class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.  NVML in-process (a step is ~1.4 ms, the
    timed region some 15 ms: nvidia-smi's loop mode does not even start that fast), sampled every
    0.5 ms on a thread; nvidia-smi -lms as the fallback when pynvml is not importable."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.nvml = None
        self.samples = []
        self.stop_flag = False
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                import torch
                uuid = "GPU-" + str(torch.cuda.get_device_properties(gpu_index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                try:
                    rs = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append((sm, rs))
            except Exception:
                break
            time.sleep(0.0005)

    def start(self):
        if self.nvml is not None:
            self.stop_flag = False
            self.thr = threading.Thread(target=self._poll, daemon=True)
            self.thr.start()
            return
        self._start_smi()

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thr.join(timeout=2)
            n = self.nvml
            try:
                mx = float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM))
            except Exception:
                mx = None
            sm = [float(a) for a, _ in self.samples]
            reasons = set()
            for _, rs in self.samples:
                for bit, nm in self.BITS.items():
                    if rs & bit:
                        reasons.add(nm)
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons),
                    "source": "nvml, 0.5 ms period, timed region only"}
        return self._stop_smi()

    def _start_smi(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._pump, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def _stop_smi(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [s.strip() for s in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
            except ValueError:
                continue
            for nm, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------
# reference CPU arm
# ---------------------------------------------------------------------------

def run_reference(sample_seconds, steps, warmup, threads_total=None):
    """Times the reference's analyze_file() (unmodified source, oracle/_ref) on the host cores.

    The reference uses one thread per channel (cli/phase-rotate.cc:437-443); to
    occupy the box, nproc // channels independent instances run side by side,
    each over the whole sample.  Grid: the reference's full 0.5 degree grid
    (`-s 1`: 360 indices), the finest it supports.
    """
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    if not O.have_ref():
        raise RuntimeError("oracle/_ref is missing (built from /root/reference in the authoring container)")
    n_frames = int(sample_seconds * SR)
    x = gen_numpy(n_frames)
    nproc = os.cpu_count() or 1
    inst = max(1, (threads_total or nproc) // CHANNELS)
    lib = O.ref_cli(f32=True)
    peaks = [np.zeros((CHANNELS, 360), np.float32) for _ in range(inst)]

    def one(i):
        lib.ref_cli_analyze(x, n_frames, CHANNELS, BLKSIZ, 0, 360, 1, -1, peaks[i])

    def step():
        th = [threading.Thread(target=one, args=(i,)) for i in range(inst)]
        t0 = time.perf_counter()
        for t in th:
            t.start()
        for t in th:
            t.join()
        return time.perf_counter() - t0

    for _ in range(warmup):
        step()
    times = [step() for _ in range(steps)]
    sa_per_step = float(inst) * n_frames * CHANNELS * 360
    total = sum(times)
    value = sa_per_step * steps / total / 1e9
    best = sa_per_step / min(times) / 1e9
    return {
        "value": value, "best": best, "unit": "Gsample-angles/s", "cores": inst * CHANNELS, "kind": "reference",
        "ms_per_step": 1e3 * total / steps,
        "sample": f"{sample_seconds:g} s of the same stereo 48 kHz programme, reference grid 0.5 deg (360 indices, -s 1), "
                  f"{inst} concurrent instances x {CHANNELS} threads; reference sources unmodified, FFTW replaced by the stand-in float FFT",
    }


def reference_main(args):
    r = run_reference(args.ref_seconds, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": "min-peak theta sweep throughput", "value": r["value"], "unit": "Gsample-angles/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, ref=True),
        "cpu_baseline": {"value": r["value"], "unit": r["unit"], "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "Gsample-angles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(args, wl=None, frames_per_gpu=None, world=1, strong=False, ref=False):
    wl = wl or dict(WORKLOADS["headline"], S=args.subsample, seconds=args.seconds or 3600.0)
    frames_per_gpu = frames_per_gpu if frames_per_gpu is not None else int(wl["seconds"] * wl["sr"])
    per = "in total, cut into one sample-range shard per GPU" if strong else "per GPU"
    cfg = {
        "workload": f"{wl['label']}, {wl['seconds']:g} s {per}, {1.0 / wl['S']:g} deg grid ({180 * wl['S']} angles), blksiz {wl['blksiz']}",
        "frames_per_gpu": int(frames_per_gpu), "channels": wl["C"], "angles": 180 * wl["S"], "sample_rate": wl["sr"],
        "l2": f"input ({4e-9 * frames_per_gpu * wl['C']:.2f} GB per GPU) is larger than the 126 MB L2; no explicit flush",
        "sharding": "sample-range, one shard per rank, NCCL max all-reduce of the peak table",
    }
    if ref:
        cfg["reference_arm"] = (f"bounded sample: {args.ref_seconds:g} s of the same material on the reference's own grid "
                                "(0.5 deg, 360 indices: the reference cannot run finer grids); rate in the same unit; "
                                "the GPU arm's `same_grid` object is measured on exactly this configuration")
    return cfg


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------

def secondary_legs(torch, capi, dev, local, x, frames, hbm_peak):
    """BASELINE.json's metric also names 'rotated Msamples/s': the CLI render (cli/phase-rotate.cc:950-1003,
    config 4 style) and the plugin run() (src/phaserotate.c:774-852, config 2) measured on the same box,
    plus the true-peak variant of the sweep (config 3).  Bounded to a few seconds."""
    out = {}
    ev = lambda: torch.cuda.Event(enable_timing=True)
    # -- CLI render, device resident: 10 min stereo per call, fixed per-channel angles
    rf = min(frames, 600 * SR)
    rf -= rf % BLKSIZ
    y = torch.empty(((rf // BLKSIZ + 1) * BLKSIZ, CHANNELS), device=dev, dtype=torch.float32)
    with capi.Phaserot(mode=capi.MODE_CLI, n_channels=CHANNELS, blksiz=BLKSIZ, device=local) as hr:
        hr.set_stream(torch.cuda.current_stream().cuda_stream)
        for _ in range(2):
            hr.render_device(x.data_ptr(), rf, [37, 181], 1, y.data_ptr())
        torch.cuda.synchronize()
        e0, e1 = ev(), ev()
        e0.record()
        n_r = 5
        for _ in range(n_r):
            hr.render_device(x.data_ptr(), rf, [37, 181], 1, y.data_ptr())
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n_r
        hr.set_profiling(True)
        hr.render_device(x.data_ptr(), rf, [37, 181], 1, y.data_ptr())
        hr.sync()
        kt = hr.kernel_times()
        gbs = 8.0 * rf * CHANNELS / (ms * 1e-3) / 1e9
        out["render"] = {"value": rf * CHANNELS / (ms * 1e-3) / 1e6, "unit": "rotated Msamples/s", "ms_per_call": ms,
                         "workload": f"CLI render, stereo 48 kHz, {rf / SR:g} s per call, device resident, angles 18.5/90.5 deg",
                         "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                                      "algorithmic_bytes_per_sample": 8},
                         "kernels_ms": {k: round(v["ms"], 4) for k, v in kt.items() if v["launches"]}}
    del y
    # -- plugin run(): mono 48 kHz, angle port at 90 deg from the first call (ramp included), 1024-frame calls
    rng = np.random.default_rng(42)
    n_calls, blk = 2000, 1024
    xin = (0.25 * rng.standard_normal(n_calls * blk)).astype(np.float32)
    yout = np.zeros_like(xin)
    ang = np.array([90.0], np.float32)
    with capi.Phaserot(mode=capi.MODE_PLUGIN, n_channels=1, sample_rate=48000.0, device=local) as hp:
        ins = (ctypes.c_void_p * 1)()
        outs = (ctypes.c_void_p * 1)()
        def run(lo, hi):
            for k in range(lo, hi):
                ins[0] = xin.ctypes.data + 4 * k * blk
                outs[0] = yout.ctypes.data + 4 * k * blk
                hp.process_raw(ins, outs, blk, ang)
        run(0, 200)
        t0 = time.perf_counter()
        run(200, n_calls)
        dt = time.perf_counter() - t0
        out["plugin"] = {"value": (n_calls - 200) * blk / dt / 1e6, "unit": "rotated Msamples/s", "us_per_call": 1e6 * dt / (n_calls - 200),
                         "workload": "LV2 run(): mono 48 kHz, 1024-frame calls, angle 90 deg, host buffers in and out (synchronous round trip per call)"}
        # bulk: 10 min in one call (host buffers; H2D + D2H inside)
        nb = 600 * SR
        xb = (0.25 * rng.standard_normal(nb)).astype(np.float32)
        yb = np.zeros_like(xb)
        hp.reset()
        ins[0], outs[0] = xb.ctypes.data, yb.ctypes.data
        hp.process_raw(ins, outs, nb, ang)
        hp.reset()
        t0 = time.perf_counter()
        hp.process_raw(ins, outs, nb, ang)
        dt = time.perf_counter() - t0
        out["plugin_bulk"] = {"value": nb / dt / 1e6, "unit": "rotated Msamples/s", "ms_per_call": 1e3 * dt,
                              "workload": "LV2 run(): mono 48 kHz, one 600 s call, pageable host buffers in and out"}
    # -- end to end from a 16-bit PCM file image (SURVEY 8f rank 1): the headline workload quantised to int16 in
    #    pinned host memory, through phaserot_sweep_pcm (H2D of 2 bytes per sample + widening on the device)
    q = torch.empty((frames, CHANNELS), dtype=torch.int16, pin_memory=True)
    q.copy_((x * 32768.0).round().clamp_(-32768, 32767).to(torch.int16))
    torch.cuda.synchronize()
    with capi.Phaserot(mode=capi.MODE_CLI, n_channels=CHANNELS, blksiz=BLKSIZ, subsample=SUBSAMPLE, device=local) as hq:
        for _ in range(2):
            hq.reset()
            hq.sweep_pcm((q.data_ptr(), frames, np.int16))
        n_q = 3
        t0 = time.perf_counter()
        for _ in range(n_q):
            hq.reset()
            hq.sweep_pcm((q.data_ptr(), frames, np.int16))
            hq.peaks()
        dt = (time.perf_counter() - t0) / n_q
        out["e2e_pcm16"] = {"value": float(frames) * CHANNELS * 180 * SUBSAMPLE / dt / 1e9, "unit": "Gsample-angles/s", "ms_per_step": 1e3 * dt,
                            "h2d_bytes_per_step": int(q.numel() * 2),
                            "workload": "the headline sweep from a 16-bit PCM image in pinned host memory (phaserot_sweep_pcm): integers over PCIe, widened on the device"}
    del q
    # -- true-peak sweep (4x), same 1800-angle grid, 10 min stereo device resident
    tf = min(frames, 600 * SR)
    tf -= tf % (32768 - BLKSIZ)
    with capi.Phaserot(mode=capi.MODE_CLI, n_channels=CHANNELS, blksiz=BLKSIZ, subsample=SUBSAMPLE, device=local, oversample=4) as ht:
        ht.set_stream(torch.cuda.current_stream().cuda_stream)
        for _ in range(2):
            ht.reset()
            ht.sweep_device(x.data_ptr(), tf)
            ht.peaks()
        e0, e1 = ev(), ev()
        e0.record()
        n_t = 3
        for _ in range(n_t):
            ht.reset()
            ht.sweep_device(x.data_ptr(), tf)
            ht.peaks()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n_t
        ht.set_profiling(True)
        ht.reset()
        ht.sweep_device(x.data_ptr(), tf)
        ht.peaks()
        kt = ht.kernel_times()
        out["true_peak"] = {"value": float(tf) * CHANNELS * 180 * SUBSAMPLE / (ms * 1e-3) / 1e9, "unit": "Gsample-angles/s", "ms_per_step": ms,
                            "workload": f"4x oversampled true-peak sweep (new capability), stereo 48 kHz, {tf / SR:g} s, 1800 angles, device resident",
                            "hbm_frac_algorithmic": 4.0 * tf * CHANNELS / (ms * 1e-3) / 1e9 / hbm_peak,
                            "kernels_ms": {k: round(v["ms"], 4) for k, v in kt.items() if v["launches"]}}
    return out


def bind_to_gpu_numa_node(torch, local):
    """Run this rank on the CPUs NVML reports as local to its GPU (what `numactl --cpunodebind` does for a
    production launch), BEFORE any page-locked buffer is allocated: with 8 ranks uploading at once, host
    buffers that sit on the other socket share the inter-socket link and the end-to-end rate of those
    ranks drops to a third.  Returns the CPU list, or None when nothing was changed."""
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = "GPU-" + str(torch.cuda.get_device_properties(local).uuid)
        h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
        ncpu = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {i for i in range(ncpu) if (mask[i // 64] >> (i % 64)) & 1} & set(os.sched_getaffinity(0))
        if cpus and cpus != set(os.sched_getaffinity(0)):
            os.sched_setaffinity(0, cpus)
            return sorted(cpus)
    except Exception:
        pass
    return None


WORKLOADS = {
    # name: channels, sample rate, block size (cli:749-755 from the rate), angle grid density, seconds, partials of the generator
    "headline": dict(C=CHANNELS, sr=SR, blksiz=BLKSIZ, S=SUBSAMPLE, seconds=3600.0, partials=N_PARTIALS,
                     label="CLI min-peak sweep: stereo 48 kHz, synthetic programme (16 partials x AM + noise), digital peak"),
    # BASELINE.json config 5: dense sweep 0.01 deg over 8-channel 192 kHz 1 h audio (22 GB of float32)
    "config5": dict(C=8, sr=192000, blksiz=32768, S=100, seconds=3600.0, partials=6,
                    label="BASELINE config 5: dense sweep, 8 ch 192 kHz, synthetic programme (6 partials x AM + noise), digital peak"),
}


class SweepBench:
    """One sharded analysis pass, timed: every rank owns frames [f0, f1) of a synthetic stream (device resident,
    generated by absolute position), the blksiz frames in front of it as history, and one handle; a step is
    reset -> phaserot_sweep_shard_device -> NCCL max all-reduce of the device table -> table read-back."""

    def __init__(self, torch, dist, capi, wl, f0, f1, first, last, rank, world, local, flags=0, seed=43, two_phase=False):
        self.two_phase = two_phase and world > 1  # bootstrap waves of all ranks combined before the contiguous passes (strong scaling)
        self.torch, self.dist, self.capi, self.wl = torch, dist, capi, wl
        self.rank, self.world, self.local, self.first, self.last = rank, world, local, first, last
        self.dev = torch.device("cuda", local)
        self.kw = dict(seed=seed, channels=wl["C"], sr=wl["sr"], n_partials=wl["partials"])
        self.frames = f1 - f0
        L = wl["blksiz"]
        self.x = gen_range_torch(torch, f0, f1, self.dev, **self.kw) if f1 > f0 else torch.zeros((0, wl["C"]), device=self.dev)
        self.hist = gen_range_torch(torch, f0 - L, f0, self.dev, **self.kw) if (f0 >= L and not first) else None
        self.hist_ptr = self.hist.data_ptr() if self.hist is not None else None
        torch.cuda.synchronize()
        self.flags = flags
        self.h = capi.Phaserot(mode=capi.MODE_CLI, n_channels=wl["C"], blksiz=L, subsample=wl["S"], device=local, flags=flags)
        self.stream = torch.cuda.current_stream()
        self.h.set_stream(self.stream.cuda_stream)
        self.tables = {}
        self.A = 180 * wl["S"]

    def combine(self, handle):
        """NCCL max all-reduce, in place, on the handle's device-resident table of the pending sweep
        (per-angle maxima + raw peaks + the library's list-overflow flag; phaserot_pending_table): no host round trip."""
        torch = self.torch
        ptr, nc, na = handle.pending_table()
        n = nc * na + nc + 1
        t = self.tables.get((ptr, n))
        if t is None:
            class _Dev:
                __cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 2}
            t = self.tables[(ptr, n)] = torch.as_tensor(_Dev(), device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)

    def combined_peaks(self, handle):
        """all-reduce + read-back; E_AGAIN (some rank's survivor list overflowed: every rank has re-enqueued its shard in
        dense mode, see phaserot_pending_table) means: reduce the new pending tables once more."""
        while True:
            self.combine(handle)
            try:
                return handle.peaks()  # sync + D2H of the combined table
            except self.capi.PhaserotError as ex:
                if ex.code != self.capi.E_AGAIN:
                    raise

    def step_device(self):
        h = self.h
        h.reset()
        if self.two_phase:
            h.sweep_shard_boot_device(self.x.data_ptr(), self.frames, self.hist_ptr, self.first, self.last)
            self.combine(h)                 # every rank now prunes with the thresholds of the whole stream's sample
            h.sweep_shard_resume()
        else:
            h.sweep_shard_device(self.x.data_ptr(), self.frames, self.hist_ptr, self.first, self.last)
        if self.world > 1:
            return self.combined_peaks(h)
        return h.peaks()  # sync + D2H of the table

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps, wall=False):
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        self.barrier()
        w = time.perf_counter() - w0
        self.last_output = out
        ms = e0.elapsed_time(e1)
        # the table read-back is a host sync inside the step; wall and event time agree, keep the larger
        t = torch.tensor([max(ms / 1e3, w if wall else 0.0)], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def check_ranks_agree(self):
        """Every rank must hold the same combined table (max and min over the ranks coincide): catches a collective
        that was not ordered behind the sweep, or ranks that disagreed about a repeat."""
        if self.world == 1:
            return
        torch = self.torch
        t = torch.from_numpy(self.step_device()).to(self.dev)
        hi, lo = t.clone(), t.clone()
        self.dist.all_reduce(hi, op=self.dist.ReduceOp.MAX)
        self.dist.all_reduce(lo, op=self.dist.ReduceOp.MIN)
        if not torch.equal(hi, lo) or not bool((t[:, 1:] > 0).all()):
            raise RuntimeError("ranks disagree about the combined peak table")

    def run_device(self, steps, warmup, sampler=None, wall=False):
        for _ in range(max(warmup, 3)):
            self.step_device()
        self.check_ranks_agree()
        self.h.reset_stats()
        if sampler is not None:
            sampler.start()
        t = self.timed(self.step_device, steps, wall)
        clocks = sampler.stop() if sampler is not None else None
        st = self.h.stats()
        return t, st, clocks

    def run_e2e(self, steps):
        """The same pass from pinned HOST memory through the library's chunked, overlapped upload
        (phaserot_sweep at N = 1, phaserot_sweep_shard per rank at N > 1): H2D of the rank's whole shard and
        D2H of the table inside the timed region."""
        torch, capi = self.torch, self.capi
        xh = torch.empty((self.frames, self.wl["C"]), dtype=torch.float32, pin_memory=True)
        xh.copy_(self.x)
        torch.cuda.synchronize()
        he = capi.Phaserot(mode=capi.MODE_CLI, n_channels=self.wl["C"], blksiz=self.wl["blksiz"], subsample=self.wl["S"], device=self.local, flags=self.flags)
        if self.world > 1:
            he.set_stream(self.stream.cuda_stream)  # the sweep and the all-reduce are ordered on one stream

        def step():
            he.reset()
            if self.world == 1:
                he.sweep((xh.data_ptr(), self.frames))
            else:
                he.sweep_shard(xh.data_ptr(), self.frames, self.hist_ptr, self.first, self.last)
                self.combined_peaks(he)
                return
            he.peaks()

        for _ in range(2):
            step()
        self.barrier()
        w0 = time.perf_counter()
        for _ in range(steps):
            step()
        self.barrier()
        t = torch.tensor([time.perf_counter() - w0], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        he.close()
        # the ceiling of this leg: the same pinned buffer copied to the device and nothing else, all ranks at once
        # (one PCIe link per GPU, but the ranks share the host's memory system)
        for _ in range(2):
            self.x.copy_(xh, non_blocking=True)
        self.barrier()
        w0 = time.perf_counter()
        for _ in range(steps):
            self.x.copy_(xh, non_blocking=True)
            torch.cuda.synchronize()
        self.barrier()
        tb = torch.tensor([time.perf_counter() - w0], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(tb, op=self.dist.ReduceOp.MAX)
        self.bare_h2d_ms = 1e3 * float(tb.item()) / steps
        del xh
        return float(t.item())

    def kernel_times(self):
        self.h.set_profiling(True)
        self.step_device()
        kt = self.h.kernel_times()
        self.h.set_profiling(False)
        return kt

    def close(self):
        self.h.close()
        del self.x


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, peaks):
    """The table the last timed step returned to its caller (phaserot_peaks), as out_dir/peaks.npy."""
    peaks = np.asarray(peaks, np.float32)
    if peaks.nbytes > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: the table's {peaks.nbytes} bytes exceed {DUMP_LIMIT_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "peaks.npy"), peaks)


def shard_range(capi, wl, total_frames, rank, world, local):
    """Frames [f0, f1) of rank `rank` when one stream of total_frames is cut on the FFT segment grid."""
    with capi.Phaserot(mode=capi.MODE_CLI, n_channels=wl["C"], blksiz=wl["blksiz"], subsample=wl["S"], device=local) as h:
        al = h.shard_align()
    per = -(-total_frames // world)
    per = max(al, -(-per // al) * al)
    f0 = min(total_frames, rank * per)
    f1 = min(total_frames, (rank + 1) * per)
    used = max(1, min(world, -(-total_frames // per)))
    return f0, f1, used


def fp2_per_segment():
    """Packed fp32 warp instructions one segment of the FFT convolution executes (ncu, profiles/ncu_traffic.json)."""
    try:
        return float(json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["fftconv_fp2_warp_inst_per_segment"])
    except Exception:
        return None


def roofline_of(kt, alg_bytes, step_ms, frames, wl, sm_mhz, n_sm=148):
    conv = kt["fftconv_filter"]
    peak, peak_src = measured_hbm_peak()
    achieved = alg_bytes / (conv["ms"] * 1e-3) / 1e9 if conv["ms"] > 0 else 0.0
    r = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None, "traffic": None,
         "kernel": "fftconv_kernel<EPI_POINTS>", "peak_source": peak_src,
         "algorithmic_bytes_per_step_per_gpu": alg_bytes, "kernel_ms_per_step": conv["ms"], "launches_per_step": conv["launches"],
         "kernel_share_of_step": conv["ms"] / step_ms if step_ms else None,
         "whole_step_frac": alg_bytes / (step_ms * 1e-3) / 1e9 / peak if step_ms else None,
         "all_kernels_ms": {k: round(v["ms"], 4) for k, v in kt.items() if v["launches"]}}
    # second roofline (SURVEY 8d "report both"): share of the kernel's cycles in which the FP32 pipe of an SM sub-partition is
    # busy with the FFT's packed instructions (2 issue cycles each: FADD2 / FMUL2 / FFMA2 are 64 lane-operations on 32 lanes)
    fp2 = fp2_per_segment()
    if fp2 and conv["ms"] > 0 and sm_mhz:
        V = 16384 - (wl["blksiz"] // 2 if wl["blksiz"] <= 16384 else 8192)
        segs = -(-(frames // 2 + wl["blksiz"] // 2) // V) * wl["C"]       # segments per pass (bootstrap wave not counted)
        cyc_busy = segs * fp2 * 2.0 / (4.0 * n_sm)                         # per SM sub-partition
        cyc_elapsed = conv["ms"] * 1e-3 * sm_mhz * 1e6
        r["fp32_issue_frac"] = cyc_busy / cyc_elapsed
        r["fp32_issue_note"] = ("packed fp32 warp instructions per segment (ncu) x 2 cycles / (4 sub-partitions x SMs), over the kernel's "
                                "elapsed cycles at the sampled SM clock: the FFT is bound by this pipe, not by HBM (DESIGN.md section 4)")
    return r


def gpu_main(args):
    import torch
    import torch.distributed as dist
    from phaserotate.lv2_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # Everything runs on ONE explicit stream: the handles are told to use it (phaserot_set_stream) and torch orders
    # its NCCL collectives against the current stream.  The legacy default stream has handle 0, which
    # phaserot_set_stream() reads as "back to the handle's private stream" - the all-reduce would then not be
    # ordered behind the sweep at all.
    torch.cuda.set_stream(torch.cuda.Stream(device=dev))
    numa = bind_to_gpu_numa_node(torch, local)  # before any page-locked buffer exists: host memory local to the GPU's socket
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=90))  # a mismatched collective must not hold the box for ten minutes

    wl = dict(WORKLOADS["config5" if args.config == "5" else "headline"])
    wl["S"] = args.subsample if args.config != "5" else wl["S"]
    wl["seconds"] = args.seconds if args.seconds else wl["seconds"]
    strong = args.scaling == "strong" or args.config == "5"
    seg2 = 2 * (16384 - (wl["blksiz"] // 2 if wl["blksiz"] <= 16384 else 8192))       # frames per FFT segment
    total = int(wl["seconds"] * wl["sr"])
    total -= total % seg2                                                              # whole blocks, cut on the FFT segment grid (phaserot_shard_align)

    def make(wl_, total_, strong_, flags=0, two_phase=False):
        if strong_:
            f0, f1, used = shard_range(capi, wl_, total_, rank, world, local)
            return SweepBench(torch, dist, capi, wl_, f0, f1, rank == 0, rank >= used - 1, rank, world, local, flags, two_phase=two_phase), total_
        # weak: rank r owns stretch r of a world x longer stream
        return SweepBench(torch, dist, capi, wl_, rank * total_, (rank + 1) * total_, rank == 0, rank == world - 1, rank, world, local, flags), total_ * world

    flags = capi.FLAG_NO_PRUNE if args.no_prune else 0
    sb, job_frames = make(wl, total, strong, flags, two_phase=args.config == "5")
    A = sb.A
    sampler = ClockSampler(local) if rank == 0 else None
    t_dev, st, clocks = sb.run_device(args.steps, args.warmup, sampler, args.wall)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sb.last_output)
    launches = torch.tensor([st["kernel_launches"]], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(launches)
    sa_step = float(job_frames) * wl["C"] * A
    value = sa_step * args.steps / t_dev / 1e9
    surv = st["points_evaluated"] / max(1, st["points_total"])
    step_ms = 1e3 * t_dev / args.steps

    e2e_steps = max(2, min(args.steps, 5))
    t_e2e = sb.run_e2e(e2e_steps)
    e2e_value = sa_step * e2e_steps / t_e2e / 1e9

    kt = sb.kernel_times()
    alg_bytes = 4.0 * sb.frames * wl["C"]  # per rank, per pass (SURVEY 8d: 4 B per input sample)
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    roof = roofline_of(kt, alg_bytes, step_ms, sb.frames, wl, sm_mhz) if rank == 0 else None

    # ---- the other scaling view and BASELINE config 5, measured in the same run at every N (objects on the line)
    extra = {}
    if not args.no_strong and args.config != "5" and args.scaling != "strong":
        if world == 1:
            extra["strong"] = {"value": value, "ms_per_step": step_ms, "note": "N = 1: identical to the headline run"}
        else:
            ss, jf = make(wl, total, True, flags)
            t, _, _ = ss.run_device(args.steps, args.warmup)
            te = ss.run_e2e(e2e_steps)
            k2 = ss.kernel_times()
            extra["strong"] = {"value": float(jf) * wl["C"] * A * args.steps / t / 1e9, "ms_per_step": 1e3 * t / args.steps,
                               "e2e_value": float(jf) * wl["C"] * A * e2e_steps / te / 1e9, "e2e_ms_per_step": 1e3 * te / e2e_steps,
                               "bare_h2d_ms_per_step": ss.bare_h2d_ms,
                               "kernels_ms_rank0": {k: round(v["ms"], 4) for k, v in k2.items() if v["launches"]}}
            ss.close()
        extra["strong"].update({"unit": "Gsample-angles/s", "scaling": "strong",
                                "workload": f"ONE {wl['seconds']:g} s stereo file cut on the FFT segment grid into {world} sample-range shard(s), "
                                            "one per GPU, NCCL max all-reduce of the table (north_star's >= 7x at 8 GPUs is about this)"})
    if not args.no_config5 and args.config != "5":
        w5 = dict(WORKLOADS["config5"])
        s5 = 2 * (16384 - 8192)
        tot5 = int(w5["seconds"] * w5["sr"])
        tot5 -= tot5 % s5
        # two-phase: the ranks' bootstrap waves are combined before the contiguous passes.  With 18000 angles every
        # survivor is expensive, and a rank that prunes against its own shard's peaks only keeps 30x more of them
        # (N = 8, one-phase: 11.4 ms per step, survivor fraction 7e-4; two-phase: 6.6 ms, 1e-5).  The 1-h stereo file
        # (`strong`) is the opposite case: the second all-reduce (35 us) costs more than it saves (0.34 vs 0.30 ms).
        c5, jf = make(w5, tot5, True, 0, two_phase=True)
        st5 = max(2, min(args.steps, 3))
        t, stt, _ = c5.run_device(st5, 2)
        k5 = c5.kernel_times()
        ms5 = 1e3 * t / st5
        peak, _ = measured_hbm_peak()
        extra["config5"] = {"value": float(jf) * w5["C"] * c5.A * st5 / t / 1e9, "unit": "Gsample-angles/s", "ms_per_step": ms5, "scaling": "strong",
                            "workload": f"{w5['label']}, {w5['seconds']:g} s ({4.0 * jf * w5['C'] / 1e9:.1f} GB), 0.01 deg grid (18000 angles), blksiz 32768, "
                                        f"cut into {world} sample-range shard(s), device resident",
                            "hbm_frac_algorithmic_whole_step": 4.0 * jf * w5["C"] / world / (ms5 * 1e-3) / 1e9 / peak,
                            "kernels_ms_rank0": {k: round(v["ms"], 4) for k, v in k5.items() if v["launches"]},
                            "survivor_fraction": stt["points_evaluated"] / max(1, stt["points_total"]),
                            "protocol": "two-phase (phaserot_sweep_shard_boot_device, all-reduce, phaserot_sweep_shard_resume, all-reduce)" if world > 1 else "single pass"}
        c5.close()

    # ---- secondary legs (rank 0, N=1): the other callers of the path, other inputs, the reference grid.  Not part of `value`.
    if world == 1 and not args.no_extra and args.config != "5":
        peak, _ = measured_hbm_peak()
        extra.update(secondary_legs(torch, capi, dev, local, sb.x, sb.frames, peak))
        extra["inputs"] = input_legs(torch, capi, dev, local, sb.x, sb.frames, step_ms)
        extra["same_grid"] = same_grid_leg(torch, capi, dev, local, sb.x, args.ref_seconds)

    line = None
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            try:
                r = run_reference(args.ref_seconds, 2, 1)
                cpu = {"value": r["value"], "unit": r["unit"], "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
            except Exception as ex:  # the oracle build is test infrastructure; never fatal for the GPU line
                cpu = {"value": None, "unit": "Gsample-angles/s", "cores": 0, "kind": "reference", "sample": f"unavailable: {ex}"}
        if cpu and cpu.get("value") and "same_grid" in extra:
            extra["same_grid"]["vs_cpu_baseline"] = {"device_resident": extra["same_grid"]["value"] / cpu["value"], "e2e": extra["same_grid"]["e2e_value"] / cpu["value"],
                                                      "same_config": True}
        if "plugin" in extra and world == 1 and not args.no_cpu:
            extra["plugin"]["cpu_baseline"] = plugin_cpu_baseline()
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath) and args.config != "5":
            try:
                roof["traffic"] = json.load(open(tpath)).get("fftconv_filter_dram_bytes_per_launch")
            except Exception:
                pass
        cfg = workload_config(args, wl, sb.frames, world, strong)
        line = {
            "metric": "min-peak theta sweep throughput", "value": value, "unit": "Gsample-angles/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "Gsample-angles/s", "h2d_bytes_per_step": int(job_frames * wl["C"] * 4),
                    "host_numa_binding": ("rank bound to %d GPU-local CPUs" % len(numa)) if numa else "none",
                    "d2h_bytes_per_step": int((wl["C"] * A + wl["C"]) * 4 * world), "steps": e2e_steps,
                    "ms_per_step": 1e3 * t_e2e / e2e_steps,
                    "bare_h2d_ms_per_step": sb.bare_h2d_ms, "vs_bare_h2d": 1e3 * t_e2e / e2e_steps / sb.bare_h2d_ms,
                    "path": "phaserot_sweep (N = 1) / phaserot_sweep_shard (N > 1): pinned host buffer, chunked upload overlapped with the sweep"},
            "gpu_launches": int(launches.item()),
            "roofline": roof,
            "pruning": {"enabled": not args.no_prune, "survivor_fraction": surv, "points_per_step_per_gpu": st["points_total"] // max(1, args.steps),
                        "dense_repeats": st["dense_repeats"]},
            "cpu_baseline": cpu,
        }
        line.update(extra)
    sb.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line))


def input_legs(torch, capi, dev, local, prog, frames, programme_ms):
    """The sweep's cost as a function of the INPUT (exact pruning makes the time depend on how many samples lie near
    the hull of the (x_d, H) point set): the same 1 h / 0.1 degree pass on config-1 two-sine material, on a pure sine
    (constant envelope: the worst case, every sample is on the hull) and on the programme with pruning switched off."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import input_legs as IL
    out = {}
    for name, (x, fl) in IL.materials(torch, dev, frames, SR, prog).items():
        if name == "programme":
            continue
        r, _ = IL.run_leg(torch, capi, x.contiguous(), frames, BLKSIZ, SUBSAMPLE, fl, steps=3, device=local)
        r["vs_programme_leg"] = r["ms_per_step"] / programme_ms
        out[name] = r
        del x
    out["note"] = ("stereo 48 kHz, 1 h, 1800 angles, device resident, steady state of a handle (first_call_ms includes the one-off dense-mode repeat); "
                   "every table is bit-identical to brute force (tests/test_gpu_round2.py, tools/input_legs.py --check)")
    return out


def same_grid_leg(torch, capi, dev, local, prog, ref_seconds):
    """The GPU arm on exactly the reference arm's configuration: ref_seconds of the same programme, the reference's own
    0.5 degree grid (360 indices).  Rates on the headline's 0.1 degree grid are ~5x higher for the same time because exact
    pruning makes the GPU time almost independent of the angle count; this object is the like-for-like anchor."""
    frames = int(ref_seconds * SR)
    x = prog[:frames].contiguous()
    ev = lambda: torch.cuda.Event(enable_timing=True)
    with capi.Phaserot(mode=capi.MODE_CLI, n_channels=CHANNELS, blksiz=BLKSIZ, subsample=2, device=local) as h:
        h.set_stream(torch.cuda.current_stream().cuda_stream)
        for _ in range(3):
            h.reset()
            h.sweep_device(x.data_ptr(), frames)
            h.peaks()
        e0, e1 = ev(), ev()
        n = 10
        e0.record()
        for _ in range(n):
            h.reset()
            h.sweep_device(x.data_ptr(), frames)
            h.peaks()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
    xh = torch.empty((frames, CHANNELS), dtype=torch.float32, pin_memory=True)
    xh.copy_(x)
    torch.cuda.synchronize()
    with capi.Phaserot(mode=capi.MODE_CLI, n_channels=CHANNELS, blksiz=BLKSIZ, subsample=2, device=local) as h:
        for _ in range(2):
            h.reset()
            h.sweep((xh.data_ptr(), frames))
        t0 = time.perf_counter()
        for _ in range(5):
            h.reset()
            h.sweep((xh.data_ptr(), frames))
            h.peaks()
        dt = (time.perf_counter() - t0) / 5
    sa = float(frames) * CHANNELS * 360
    return {"value": sa / (ms * 1e-3) / 1e9, "e2e_value": sa / dt / 1e9, "unit": "Gsample-angles/s", "ms_per_step": ms, "e2e_ms_per_step": 1e3 * dt,
            "workload": f"{ref_seconds:g} s of the stereo 48 kHz programme, reference grid 0.5 deg (360 indices), blksiz {BLKSIZ}: the reference arm's configuration"}


def plugin_cpu_baseline():
    """BASELINE.md row 2 on the host cores: the reference plugin built from the unmodified source (oracle/_ref/phaserotate_ref.so,
    stand-in float FFT) and this repository's LV2 BINARY, both driven through the same minimal LV2 host (oracle/lv2_harness.c)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    try:
        import oracle_lib as O
        from phaserotate.lv2_b200 import build as B
        rng = np.random.default_rng(42)
        out = {}
        n_small, n_bulk = 1024 * 2000, 600 * SR
        xs = (0.25 * rng.standard_normal(n_small)).astype(np.float32)[None, :]
        xb = (0.25 * rng.standard_normal(n_bulk)).astype(np.float32)[None, :]
        ref_so = os.path.join(O.REF_DIR, "phaserotate_ref.so")
        our_so = os.path.join(B.BIN_DIR, "phaserotate_cuda.so")
        for tag, so in (("reference_cpu", ref_so), ("cuda_lv2_binary", our_so)):
            if not os.path.exists(so):
                out[tag] = {"unavailable": os.path.relpath(so, ROOT)}
                continue
            O.lv2_render(so, xs[:, :1024 * 200], 48000.0, 1024, 90.0)  # warm
            _, _, dt = O.lv2_render(so, xs, 48000.0, 1024, 90.0)
            _, _, db = O.lv2_render(so, xb, 48000.0, n_bulk, 90.0)
            out[tag] = {"us_per_1024_frame_call": 1e6 * dt / 2000, "msamples_per_s_1024": n_small / dt / 1e6,
                        "bulk_ms_per_600s_call": 1e3 * db, "msamples_per_s_bulk": n_bulk / db / 1e6}
        out["cores"] = 1
        out["kind"] = "reference"
        out["sample"] = "mono 48 kHz white noise, angle 90 deg: 2000 run() calls of 1024 frames, and one 600 s call; seconds spent inside run()"
        return out
    except Exception as ex:
        return {"unavailable": str(ex)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--seconds", type=float, default=0.0, help="audio seconds (per GPU for weak scaling, in total for strong); default: the workload's 1 hour")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: one --seconds stretch per GPU (default); strong: ONE --seconds file cut into one shard per GPU")
    ap.add_argument("--config", default="headline", choices=["headline", "5"], help="5: BASELINE config 5 (8 ch, 192 kHz, 1 h, 0.01 deg, blksiz 32768), strong scaling")
    ap.add_argument("--no-strong", action="store_true", help="skip the `strong` object (the 1 h file cut across the ranks) of a weak-scaling run")
    ap.add_argument("--no-config5", action="store_true", help="skip the `config5` object")
    ap.add_argument("--subsample", type=int, default=SUBSAMPLE)
    ap.add_argument("--ref-seconds", type=float, default=240.0, help="bounded CPU sample for the reference arm")
    ap.add_argument("--no-prune", action="store_true", help="evaluate every sample at every angle")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the render / plugin / true-peak secondary legs")
    ap.add_argument("--wall", action="store_true", help="use max(wall, events) as the step time")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="GPU arm only: write the peak table of the last timed step as DIR/peaks.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm")
    if args.impl == "reference":
        # under torchrun only rank 0 works; the other ranks exit quietly
        if int(os.environ.get("RANK", "0")) != 0:
            return
        reference_main(args)
        return
    gpu_main(args)


if __name__ == "__main__":
    main()
