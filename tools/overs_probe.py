"""Cost of the overs table (phaserot_overs_device) as the ceiling drops, next to the sweep on the same data.

Device-resident stereo 48 kHz, 1 h, blksiz 8192, bench.py's 0.1 degree grid.  Legs:
  programme (bench.py's generator), digital and true-peak 4x, ceilings at the table's min peak and 1, 3, 6 and
  12 dB below the whole-stream max peak;
  two_sine (997 Hz + 3 kHz, 0.45 each) and a pure 997 Hz sine (0.8), digital, 3 dB below the max peak.
Per row: ms of phaserot_overs_device (CUDA events on the handle's stream, mean of `--steps` calls after one
warm-up call), FFT + kernel launches, survivor fraction (points evaluated / points examined), dense_repeats
(launches re-run in pieces because a list overflowed) and phaserot_sweep_device + phaserot_peaks on the same
data in the same run.  Then the card's name and power limit.  The input (1.4 GB) is far larger than L2.

    python tools/overs_probe.py [--seconds 3600] [--steps 3] [--out profiles/overs_probe.jsonl]
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

    def legs(name, x, oversample, ceilings):
        h = capi.Phaserot(n_channels=2, blksiz=bench.BLKSIZ, subsample=bench.SUBSAMPLE, device=0, oversample=oversample)
        h.set_stream(torch.cuda.current_stream().cuda_stream)

        def sweep():
            h.reset()
            h.sweep_device(x.data_ptr(), frames)
            h.peaks()

        sweep_ms = timed(torch, sweep, a.steps)
        pk = h.peaks()
        cmax, cmin = float(pk.max()), float(pk.min())
        for label, T in ceilings(cmax, cmin):
            T = float(np.float32(T))
            ms = timed(torch, lambda: h.overs_device(x.data_ptr(), frames, T), a.steps)
            h.reset_stats()
            cnt, _ = h.overs_device(x.data_ptr(), frames, T)
            st = h.stats()
            emit({"leg": name, "detector": "true-peak 4x" if oversample else "digital", "ceiling": label, "ceiling_dbfs": round(20 * math.log10(T), 3),
                  "ms": round(ms, 3), "sweep_ms": round(sweep_ms, 3), "kernel_launches": st["kernel_launches"],
                  "survivor_fraction": st["points_evaluated"] / max(1, st["points_total"]), "dense_repeats": st["dense_repeats"],
                  "fewest_overs": [int(cnt[c].min()) for c in range(2)], "overs_at_angle0": [int(cnt[c, 0]) for c in range(2)]})
        h.close()

    def programme_ceilings(cmax, cmin):
        return [("min_peak", cmin)] + [(f"max_minus_{d}dB", cmax * 10 ** (-d / 20)) for d in (1, 3, 6, 12)]

    x = bench.gen_range_torch(torch, 0, frames, dev).contiguous()
    for os_ in (0, 4):
        legs("programme", x, os_, programme_ceilings)
    del x
    for name, freqs, amp in (("two_sine", (997.0, 3000.0), 0.45), ("sine", (997.0,), 0.8)):
        x = tones(torch, frames, dev, freqs, amp)
        legs(name, x, 0, lambda cmax, cmin: [("max_minus_3dB", cmax * 10 ** (-3 / 20))])
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
