#!/usr/bin/env python
"""Packet-mode FEC inside the decoder (dabstar_decoder_set_packet_fec) on the packet workload of tools/bench_packet.py: R recordings of
F frames of the full ensemble, u8 IQ resident in HBM, whose first four EEP sub-channels carry packet streams (three addresses each)
in FEC frames (tests/pfec_support.py) at 15 dB. Steps alternate between a decoder with the packet pass alone and one with the FEC
pass in front of it (same inputs, one process); one profiled run of its own splits the FEC pass into its kernels. Prints one JSON
line (--out: also writes it there).
Usage: python tools/bench_packet_fec.py [--recordings 96] [--frames 104] [--steps 20] [--out file]"""
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
    import packet_support as ps
    import pfec_support as fs
    from bench_full_ensemble import SPEC
    from dabstar_b200 import api, synth
    ap = argparse.ArgumentParser()
    ap.add_argument("--recordings", type=int, default=96)
    ap.add_argument("--frames", type=int, default=104)
    ap.add_argument("--unique", type=int, default=4)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    subch, cu = [], 0
    for i, (sf, lvl, br, size) in enumerate(SPEC):
        subch.append(synth.SubChannel(i + 1, cu, size, sf, lvl, br))
        cu += size
    pk = [s for s in subch if s.short_form == 0 and s.bit_rate % 8 == 0][:4]
    addrs = (1, 2, 1000)
    # 400 logical frames of packets per packet-mode sub-channel (three addresses, groups of up to 2 KB), tiled
    rng = np.random.default_rng(5)
    tiles = {s.sub_ch_id: fs.build_fec_stream(s.bit_rate, 412, {a: ps.random_groups(rng, 400 * s.bit_rate // 200 + 4, (0, 2048)) for a in addrs}, rng)[0]
             for s in pk}  # 412 logical frames hold whole FEC frames at every rate used (412 * bit_rate / 8 slots, a multiple of 103)

    def payload(n_frames, lead):
        out = []
        for s in subch:
            if s.sub_ch_id not in tiles:
                out.append(None)
                continue
            t = tiles[s.sub_ch_id]
            reps = (4 * n_frames + lead) // t.shape[0] + 1
            out.append(np.ascontiguousarray(np.tile(t, (reps, 1))[lead:lead + 4 * n_frames]))
        return out

    stream = torch.cuda.Stream()
    ctx = api.Context(0, stream=stream)

    def decoders(n_rec, fec):
        dp = api.DabProcessor(n_rec, input_format=api.FMT_U8, max_window=128, ctx=ctx)
        for r in range(n_rec):
            dp.set_audio_channel(r, subch)
            for s in pk:
                for a in addrs:
                    dp.set_packet(r, s.sub_ch_id, a)
                if fec:
                    dp.set_packet_fec(r, s.sub_ch_id)
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

    def kernel_ms(dp, ptrs, ns):
        """Device time of each FEC and packet kernel in one run, from a profiled run of its own (the timed steps run without the profiler)."""
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            dp.run_ptrs(ptrs, ns, api.MEM_DEVICE)
            torch.cuda.synchronize()
        out = {"k_pfec_code": 0.0, "k_pfec_start": 0.0, "k_pfec_list": 0.0, "k_pfec_correct": 0.0, "k_packet_scan": 0.0, "k_packet_walk": 0.0,
               "k_packet_compact": 0.0}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) / 1000.0
            for k in list(out):
                if k in e.key:
                    out[k] += t
            if e.key.startswith(("Memcpy", "Memset")):  # copies and fills of the whole run, the FEC pass's among them
                out["run: " + e.key] = out.get("run: " + e.key, 0.0) + t
        return out

    def figures(dp, n_rec):
        status = [0] * 5
        payload_bytes = packets = crc_errors = 0
        for r in range(n_rec):
            for s in pk:
                for a in addrs:
                    rec, pay = dp.data_groups(r, s.sub_ch_id, a)
                    for x in rec:
                        status[x.status] += 1
                    payload_bytes += pay.size
                    st = dp.packet_stats(r, s.sub_ch_id, a)
                    packets += st.packets
                    crc_errors += st.crc_errors
        frames = [0] * 4
        rows = [0, 0]
        for r in range(n_rec):
            for s in pk:
                for f in dp.fec_frames(r, s.sub_ch_id):
                    frames[f.status] += 1
                    rows[0] += f.rows_corrected
                    rows[1] += f.rows_failed
        return {"packet_ms": dp.packet_ms(), "packet_fec_ms": dp.packet_fec_ms(), "fec_frames_per_status": frames, "fec_rows_corrected_failed": rows,
                "logical_frames": sum(dp.result(r).msc[s.sub_ch_id].shape[0] for r in range(n_rec) for s in pk),
                "packets_of_selected_addresses": packets, "packet_crc_errors": crc_errors, "groups_per_status": status, "payload_bytes": payload_bytes}

    result = {"workload": "full ensemble (tools/bench_full_ensemble.py) + packet-mode data groups on 4 EEP sub-channels x 3 addresses, in FEC frames",
              "packet_subchannels": [(s.sub_ch_id, s.bit_rate) for s in pk], "card": card(),
              "recordings": args.recordings, "frames": args.frames, "steps_per_arm": args.steps}
    with torch.cuda.stream(stream):
        recs = [synth.generate(args.frames, seed=900 + i, snr_db=15.0, subch=subch, fmt=synth.FMT_U8, msc_payload=payload(args.frames, 7 * i))
                for i in range(args.unique)]
        dev, n = resident(recs, args.recordings)
        ptrs, ns = [dev[r].data_ptr() for r in range(args.recordings)], [n] * args.recordings
        off, on = decoders(args.recordings, False), decoders(args.recordings, True)
        for dp in (off, on):  # warm-up
            dp.run_ptrs(ptrs, ns, api.MEM_DEVICE)
        t_off, t_on, fec_ms, pk_ms = [], [], [], []
        for _ in range(args.steps):
            t_off.append(timed(off, ptrs, ns))
            t_on.append(timed(on, ptrs, ns))
            fec_ms.append(on.packet_fec_ms())
            pk_ms.append(on.packet_ms())
        result.update({"step_ms_fec_off": float(np.median(t_off)), "step_ms_fec_on": float(np.median(t_on)),
                       "packet_fec_ms_median": float(np.median(fec_ms)), "packet_ms_median_fec_on": float(np.median(pk_ms)),
                       "fec_on": figures(on, args.recordings), "kernel_ms": kernel_ms(on, ptrs, ns)})
    result["card_after"] = card()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
