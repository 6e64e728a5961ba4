"""Cost of the integrated loudness (phaserot_loudness_device) next to the sweep on the same data.

Device-resident stereo 48 kHz programme from bench.py's generator, 1 h, blksiz 8192, bench.py's grid.
Cases: phaserot_loudness_device with 2 angle sets (the CLI's input + output) and with 360 sets (every
half degree), and phaserot_sweep_device + phaserot_peaks.  Every timing is a host clock around a device
synchronise, after two warm-up calls, mean of `--steps` calls; the input (1.4 GB) is far larger than L2.
Then one profiled call per case (phaserot_set_profiling: CUDA events around every launch; the loudness
kernels are charged to "other", its FFT launches to "truepeak_filter") and the card's name and power limit.

"model_bytes" is the HBM traffic the loudness pass needs at least: x read twice (the two K-weighting
passes), K(x) written once and read twice (FFT pass, sums), the Hilbert branch written and read once.

    python tools/loudness_probe.py [--seconds 3600] [--steps 3] [--out profiles/loudness_probe.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(torch, fn, steps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / steps * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=3600.0)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import bench
    from phaserotate.lv2_b200 import capi

    dev = torch.device("cuda", 0)
    frames = int(a.seconds * bench.SR)
    x = bench.gen_range_torch(torch, 0, frames, dev).contiguous()
    h = capi.Phaserot(n_channels=2, blksiz=bench.BLKSIZ, subsample=bench.SUBSAMPLE, device=0)
    MS = h.maxsample
    sets2 = [[0, 0], [MS // 4, MS // 3]]
    sets360 = [[k * MS // 360] * 2 for k in range(360)]
    res = {}

    def loud(sets):
        res[len(sets)] = h.loudness_device(x.data_ptr(), frames, sets, bench.SR)

    def sweep():
        h.reset()
        h.sweep_device(x.data_ptr(), frames)
        h.peaks()

    T = frames + bench.BLKSIZ // 2
    model_bytes = 4 * 2 * (2 * frames + 3 * T + 2 * T)
    lines = []
    for case, fn in [("loudness_2_sets", lambda: loud(sets2)), ("loudness_360_sets", lambda: loud(sets360)), ("sweep", sweep)]:
        ms = timed(torch, fn, a.steps)
        h.reset_stats()
        h.set_profiling(True)
        fn()
        kt = h.kernel_times()
        h.set_profiling(False)
        st = h.stats()
        r = {"case": case, "ms": round(ms, 3), "kernel_launches": st["kernel_launches"],
             "kernel_ms": {k: round(v["ms"], 3) for k, v in kt.items() if v["launches"]},
             "kernel_launch_counts": {k: v["launches"] for k, v in kt.items() if v["launches"]}}
        if case.startswith("loudness"):
            r["model_bytes"] = model_bytes
            r["model_GB_per_s"] = round(model_bytes / (ms * 1e-3) / 1e9, 1)
        print(json.dumps(r), flush=True)
        lines.append(r)
    lines.append({"lufs_input": res[2][0], "lufs_2nd_set": res[2][1], "lufs_360_range": [float(res[360].min()), float(res[360].max())],
                  "angle0_equal_in_both_calls": bool(res[2][0] == res[360][0])})
    print(json.dumps(lines[-1]), flush=True)
    h.close()
    info = {"card": card(), "seconds": a.seconds, "channels": 2, "sample_rate": bench.SR, "blksiz": bench.BLKSIZ, "subsample": bench.SUBSAMPLE,
            "timing": f"host clock around a device synchronise, mean of {a.steps} calls after 2 warm-up calls, device-resident input"}
    print(json.dumps(info), flush=True)
    lines.append(info)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
