"""Cost of the per-section sweep (phaserot_sweep_sections_device) against the plain sweep and against the
per-section shard loop it replaces.

Device-resident stereo 48 kHz, 1 h, 0.1 degree grid, blksiz 8192; programme material from bench.py's
generator and the config-1 two-sine material of tools/input_legs.py.  Per material: the plain
phaserot_sweep_device, the sections sweep at 10 s and 1 s sections, and the loop of one
phaserot_sweep_shard_device per 10 s section (history = the blksiz frames before it).  Every timing is
a host clock around a device synchronise, after two warm-up calls, mean of `--steps` calls; the input
(1.4 GB per material) is far larger than L2.  One JSON line per case, then the card.

    python tools/sections_probe.py [--seconds 3600] [--steps 3] [--out profiles/sections_probe.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


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
    import input_legs as IL
    from phaserotate.lv2_b200 import capi

    dev = torch.device("cuda", 0)
    frames = int(a.seconds * bench.SR)
    prog = bench.gen_range_torch(torch, 0, frames, dev)
    mats = {
        "programme": prog,
        "two_sine": IL.tone_chunks(torch, dev, frames, bench.SR, [(0.5, 110.0, [0.0, 1.0]), (0.25, 1760.3, [0.0, 0.0])]),
    }
    lines = []
    for name, x in mats.items():
        x = x.contiguous()
        h = capi.Phaserot(n_channels=2, blksiz=bench.BLKSIZ, subsample=bench.SUBSAMPLE, device=0)
        al = h.shard_align()
        sec = lambda s: (int(s * bench.SR) + al - 1) // al * al   # rounded up like the CLI's --sections

        def plain():
            h.reset()
            h.sweep_device(x.data_ptr(), frames)
            return h.peaks()

        def sections(S):
            h.sweep_sections_device(x.data_ptr(), frames, S)

        def shard_loop(S):
            n = (frames + S - 1) // S
            for k in range(n):
                f0, f1 = k * S, min(frames, (k + 1) * S)
                h.reset()
                h.sweep_shard_device(x[f0:].data_ptr(), f1 - f0, x[f0 - bench.BLKSIZ:f0].data_ptr() if k else None, k == 0, k == n - 1)
                h.peaks()

        cases = [("plain", None, plain)] + [(f"sections_{s:g}s", sec(s), (lambda S: lambda: sections(S))(sec(s))) for s in (10.0, 1.0)]
        cases.append(("shard_loop_10s", sec(10.0), lambda: shard_loop(sec(10.0))))
        for case, S, fn in cases:
            ms = timed(torch, fn, a.steps)
            h.reset_stats()
            fn()
            st = h.stats()
            r = {"material": name, "case": case, "ms": round(ms, 3), "section_frames": S,
                 "n_sections": None if S is None else (frames + S - 1) // S,
                 "survivor_fraction": st["points_evaluated"] / max(1, st["points_total"]),
                 "kernel_launches": st["kernel_launches"], "overflow_reruns": st["dense_repeats"]}
            if case == "sections_10s":
                plain_max = plain()
                h.sweep_sections_device(x.data_ptr(), frames, S)
                r["max_over_sections_equals_plain"] = bool((torch.from_numpy(h.section_peaks().max(0)) == torch.from_numpy(plain_max)).all())
            print(json.dumps(r), flush=True)
            lines.append(r)
        h.close()
        del x
    info = {"card": card(), "seconds": a.seconds, "channels": 2, "blksiz": bench.BLKSIZ, "subsample": bench.SUBSAMPLE,
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
