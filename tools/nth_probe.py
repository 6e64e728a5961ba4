"""Cost of the rank table (phaserot_nth_peaks_device) next to the sweep on the same data.

Device-resident stereo 48 kHz, 1 h, blksiz 8192, bench.py's 0.1 degree grid.  Legs:
  programme (bench.py's generator), digital and true-peak 4x, ranks 1, 11 and 256;
  two_sine (997 Hz + 3 kHz, 0.45 each) and a pure 997 Hz sine (0.8), digital, rank 11.
Per row: ms of phaserot_nth_peaks_device (CUDA events on the handle's stream, mean of `--steps` calls after one
warm-up call), FFT + kernel launches, survivor fraction (points evaluated / points examined), dense_repeats
(launches whose candidates or lists overflowed and were re-run in pieces), phaserot_sweep_device +
phaserot_peaks on the same data in the same run, and whether rank 1 of the table is the sweep's peak table bit for
bit.  Programme legs also time the two parts of the call alone: grid index 0 (the raw input, ang 0 .. 1) and the
other angles (ang 1 .. MS).  Then the card's name and power limit.  The input (1.4 GB) is far larger than L2.

    python tools/nth_probe.py [--seconds 3600] [--steps 3] [--out profiles/nth_probe.jsonl]
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(torch, fn, steps):
    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


def tones(torch, frames, dev, freqs, amp):
    t = torch.arange(frames, device=dev, dtype=torch.float64) / 48000.0
    x = sum(amp * torch.sin(2 * math.pi * ((t * f) % 1.0) + 0.3 * k) for k, f in enumerate(freqs))
    return torch.stack([x, torch.roll(x, 17)], 1).to(torch.float32).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=3600.0)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    import bench
    from phaserotate.lv2_b200 import capi

    dev = torch.device("cuda", 0)
    frames = int(a.seconds * bench.SR)
    lines = []

    def emit(r):
        print(json.dumps(r), flush=True)
        lines.append(r)

    def legs(name, x, oversample, ranks, split=False):
        h = capi.Phaserot(n_channels=2, blksiz=bench.BLKSIZ, subsample=bench.SUBSAMPLE, device=0, oversample=oversample)
        h.set_stream(torch.cuda.current_stream().cuda_stream)

        def sweep():
            h.reset()
            h.sweep_device(x.data_ptr(), frames)
            h.peaks()

        sweep_ms = timed(torch, sweep, a.steps)
        pk = h.peaks()
        for N in ranks:
            ms = timed(torch, lambda: h.nth_peaks_device(x.data_ptr(), frames, N), a.steps)
            h.reset_stats()
            t = h.nth_peaks_device(x.data_ptr(), frames, N)
            st = h.stats()
            r = {"leg": name, "detector": "true-peak 4x" if oversample else "digital", "rank": N,
                 "ms": round(ms, 3), "sweep_ms": round(sweep_ms, 3), "kernel_launches": st["kernel_launches"],
                 "survivor_fraction": st["points_evaluated"] / max(1, st["points_total"]), "dense_repeats": st["dense_repeats"],
                 "rank1_equals_sweep": bool(np.array_equal(t[:, :, 0], pk)),
                 "lowest_rank_level_dbfs": [round(20 * math.log10(max(float(t[c, :, N - 1].min()), 1e-30)), 3) for c in range(2)]}
            if split:
                r["index0_only_ms"] = round(timed(torch, lambda: h.nth_peaks_device(x.data_ptr(), frames, N, 0, 1), a.steps), 3)
                r["other_angles_only_ms"] = round(timed(torch, lambda: h.nth_peaks_device(x.data_ptr(), frames, N, 1, h.maxsample), a.steps), 3)
            emit(r)
        h.close()

    x = bench.gen_range_torch(torch, 0, frames, dev).contiguous()
    for os_ in (0, 4):
        legs("programme", x, os_, (1, 11, 256), split=True)
    del x
    for name, freqs, amp in (("two_sine", (997.0, 3000.0), 0.45), ("sine", (997.0,), 0.8)):
        x = tones(torch, frames, dev, freqs, amp)
        legs(name, x, 0, (11,))
        del x
    emit({"card": card(), "seconds": a.seconds, "channels": 2, "sample_rate": bench.SR, "blksiz": bench.BLKSIZ, "subsample": bench.SUBSAMPLE,
          "timing": f"CUDA events on the handle's stream, mean of {a.steps} calls after 1 warm-up call, device-resident input"})
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
