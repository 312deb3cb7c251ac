#!/usr/bin/env python
"""The DAB+ outer code inside the decoder (dabstar_decoder_set_dabplus) on the full-ensemble workload of
tools/bench_full_ensemble.py: R recordings of F frames, u8 IQ resident in HBM, the same 18 sub-channels, whose 14 EEP
sub-channels carry real super-frames at 15 dB. Steps alternate between a decoder without and one with DAB+ (same inputs, one
process), then the same with random payload (no super-frames: the Fire-code scan alone) and one long recording (the walk's
least parallel case). Prints one JSON line. Usage: python tools/bench_dabplus.py [--recordings 96] [--frames 104] [--steps 20]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        return out.strip().splitlines()[0]
    except Exception as e:  # the timing does not depend on it
        return f"unknown ({e})"


def main():
    import torch
    import helpers
    from bench_full_ensemble import SPEC
    from dabstar_b200 import api, synth
    from oracle_api import Oracle
    ap = argparse.ArgumentParser()
    ap.add_argument("--recordings", type=int, default=96)
    ap.add_argument("--frames", type=int, default=104)
    ap.add_argument("--unique", type=int, default=4)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--long-frames", type=int, default=3744)
    args = ap.parse_args()
    oracle = Oracle("dabo")
    subch, cu = [], 0
    for i, (sf, lvl, br, size) in enumerate(SPEC):
        subch.append(synth.SubChannel(i + 1, cu, size, sf, lvl, br))
        cu += size
    eep = [s for s in subch if s.short_form == 0]
    # 80 super-frames (400 logical frames) per EEP sub-channel, tiled: a tile boundary keeps the five-frame stride
    rng = np.random.default_rng(5)
    tiles = {s.sub_ch_id: np.concatenate([helpers.dabplus_superframe(s.bit_rate, rng, oracle.rs_encode, dac_rate=i % 2, sbr_flag=(i // 2) % 2)[0] for i in range(80)])
             for s in eep}

    def payload(n_frames, lead):
        out = []
        for s in subch:
            if s.short_form:
                out.append(None)
                continue
            t = tiles[s.sub_ch_id]
            reps = (4 * n_frames + lead) // t.shape[0] + 1
            out.append(np.ascontiguousarray(np.tile(t, (reps, 1))[lead:lead + 4 * n_frames]))
        return out

    stream = torch.cuda.Stream()
    ctx = api.Context(0, stream=stream)

    def decoders(n_rec, on):
        dp = api.DabProcessor(n_rec, input_format=api.FMT_U8, max_window=128, ctx=ctx)
        for r in range(n_rec):
            dp.set_audio_channel(r, subch)
            if on:
                for s in eep:
                    dp.set_dabplus(r, s.sub_ch_id)
        return dp

    def resident(recs, n_rec):
        host = torch.from_numpy(np.stack([recs[r % len(recs)].iq for r in range(n_rec)]))
        return host.cuda(), host.shape[1]

    def timed(dp, ptrs, ns):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        dp.run_ptrs(ptrs, ns, api.MEM_DEVICE)
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1)

    def dabplus_figures(dp):
        ms, rounds = dp.dabplus_ms()
        scanned, decoded = dp.dabplus_windows()
        return {"dabplus_ms": ms, "rounds": rounds, "windows_decoded": decoded, "windows_scanned": scanned}

    result = {"workload": "full ensemble (tools/bench_full_ensemble.py) + DAB+ outer code on its 14 EEP sub-channels", "card": card(),
              "recordings": args.recordings, "frames": args.frames, "steps_per_arm": args.steps}
    with torch.cuda.stream(stream):
        sf_recs = [synth.generate(args.frames, seed=900 + i, snr_db=15.0, subch=subch, fmt=synth.FMT_U8, msc_payload=payload(args.frames, 7 * i))
                   for i in range(args.unique)]
        dev, n = resident(sf_recs, args.recordings)
        ptrs, ns = [dev[r].data_ptr() for r in range(args.recordings)], [n] * args.recordings
        off, on = decoders(args.recordings, False), decoders(args.recordings, True)
        for dp in (off, on):  # warm-up
            dp.run_ptrs(ptrs, ns, api.MEM_DEVICE)
        t_off, t_on = [], []
        for _ in range(args.steps):
            t_off.append(timed(off, ptrs, ns))
            t_on.append(timed(on, ptrs, ns))
        good = bad = 0
        for r in range(min(args.recordings, args.unique)):
            for s in eep:
                rec, pay = on.superframes(r, s.sub_ch_id)
                for x, p in zip(rec, pay):
                    good += sum(1 for u in range(x.num_aus) if x.ok and x.au_state[u] == 1)
                    bad += sum(1 for u in range(x.num_aus) if not (x.ok and x.au_state[u] == 1))
        result.update({"step_ms_dabplus_off": float(np.median(t_off)), "step_ms_dabplus_on": float(np.median(t_on)),
                       "superframes": dabplus_figures(on), "aus_good_bad_first_recordings": [good, bad]})
        del dev
        rnd = [synth.generate(args.frames, seed=900 + i, snr_db=15.0, subch=subch, fmt=synth.FMT_U8) for i in range(args.unique)]
        dev, n = resident(rnd, args.recordings)
        ptrs = [dev[r].data_ptr() for r in range(args.recordings)]
        on.run_ptrs(ptrs, ns, api.MEM_DEVICE)
        t_rnd = [timed(on, ptrs, ns) for _ in range(3)]
        result["random_payload"] = dict(dabplus_figures(on), step_ms=float(np.median(t_rnd)))
        del dev, on, off
        long_rec = synth.generate(args.long_frames, seed=77, snr_db=15.0, subch=subch, fmt=synth.FMT_U8, msc_payload=payload(args.long_frames, 3))
        dev, n = resident([long_rec], 1)
        lp = decoders(1, True)
        lp.run_ptrs([dev[0].data_ptr()], [n], api.MEM_DEVICE)
        t_long = [timed(lp, [dev[0].data_ptr()], [n]) for _ in range(3)]
        result["long_recording"] = dict(dabplus_figures(lp), frames=args.long_frames, step_ms=float(np.median(t_long)))
    result["card_after"] = card()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
