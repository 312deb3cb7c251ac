"""Cost of per-frame signal-quality capture (dabstar_decoder_set_frame_quality) on bench.py's headline workload.

96 recordings x 104 frames, u8, FIC only (scan mode), inputs resident in HBM, max_window 128: the same decoder runs steps with
capture off and on, alternating, so that both see the same clocks and neighbours. Per step: device time (CUDA events around
the run), stage [5] (demap, which holds k_frame_quality when capture is on) from dabstar_decoder_stage_ms. A separate,
untimed torch.profiler pass splits stage [5] into k_demap5 and k_frame_quality. Prints one JSON line (and writes it to --out).

    python tools/bench_frame_quality.py --steps 20 --warmup 3 [--out result.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LEAD, T_F, TAIL = 60000, 196608, 4096


def card():
    """Name and power limit of GPU 0 (read only)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        name, limit = (s.strip() for s in out.split(","))
        return name, limit
    except Exception as e:  # the figure is reported, not needed
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--recordings", type=int, default=96)
    ap.add_argument("--frames", type=int, default=104)
    ap.add_argument("--steps", type=int, default=20, help="timed steps per setting (capture off and on alternate)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--seed", type=int, default=2)
    ap.add_argument("--snr", type=float, default=15.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from dabstar_b200 import api, synth
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: the decode path has no CPU fallback")
    R, F = args.recordings, args.frames
    n = LEAD + F * T_F + TAIL
    host = np.empty((R, n, 2), np.uint8)
    for r in range(R):
        synth.generate(F, seed=args.seed + r, snr_db=args.snr, fmt=synth.FMT_U8, out=host[r])
    dev = torch.from_numpy(host).cuda()
    stream = torch.cuda.Stream()
    ctx = api.Context(0, stream=stream)
    dp = api.DabProcessor(R, input_format=api.FMT_U8, scan_mode=True, max_window=128, ctx=ctx)
    step = dp.prepared([dev[r].data_ptr() for r in range(R)], [n] * R, api.MEM_DEVICE)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {False: [], True: []}
    demap = {False: [], True: []}
    with torch.cuda.stream(stream):
        for on in (False, True):
            dp.set_frame_quality(on)
            for _ in range(args.warmup):
                step()
        for i in range(2 * args.steps):
            on = i % 2 == 1
            dp.set_frame_quality(on)
            e0.record(stream)
            step()
            e1.record(stream)
            e1.synchronize()
            res[on].append(e0.elapsed_time(e1))
            demap[on].append(dp.stage_ms()["demap"][0])
        frames = int(sum(dp.counters(r)[6] for r in range(R)))
        # kernel split of stage [5] with capture on (a run of its own: tracing slows the host)
        from torch.profiler import ProfilerActivity, profile
        dp.set_frame_quality(True)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                step()
            torch.cuda.synchronize()
    k_ms = {"k_demap5": 0.0, "k_frame_quality": 0.0}
    for ev in prof.key_averages():
        for k in k_ms:
            if k in ev.key:
                k_ms[k] += ev.device_time_total / 1000.0 / 3  # us over 3 steps -> ms per step
    name, limit = card()
    med = {on: float(np.median(res[on])) for on in res}
    out = {
        "workload": f"{R} recordings x {F} frames, u8, FIC only, inputs in HBM, max_window 128", "frames_per_step": frames,
        "gpu": name, "power_limit": limit, "steps_per_setting": args.steps,
        "step_ms_off": {"median": med[False], "min": min(res[False]), "max": max(res[False])},
        "step_ms_on": {"median": med[True], "min": min(res[True]), "max": max(res[True])},
        "step_overhead_pct": 100.0 * (med[True] / med[False] - 1.0),
        "demap_stage_ms_off": float(np.median(demap[False])), "demap_stage_ms_on": float(np.median(demap[True])),
        "profiler_ms_per_step_capture_on": k_ms,
        "k_frame_quality_share_of_demap_stage_pct": 100.0 * k_ms["k_frame_quality"] / max(1e-9, k_ms["k_demap5"] + k_ms["k_frame_quality"]),
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
