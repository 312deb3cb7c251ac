#!/usr/bin/env python
"""bench.py — Mode-I frames/s decoded (IQ -> Viterbi) on N B200s, one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Headline workload (BASELINE.json configs[1]): FIC-only decode of a ~10 000-frame synthetic Mode-I batch per GPU (PRS sync,
ingest + FFT, DQPSK demap of all 75 data symbols, FIC Viterbi, FIB CRC). The batch is 96 INDEPENDENT recordings of 104 frames
(10 s each, the length of configs[0]) of u8 IQ at 15 dB SNR. A step = one pass of the whole path over the batch.
  value : whole-job frames/s, inputs resident in HBM, CUDA-event time, max over ranks
  e2e   : the same through the public API with pinned HOST buffers (H2D of the IQ and D2H of the FIB bits inside)
  roofline / stages : per kernel family, algorithmic bytes (DESIGN.md) over the CUDA-event time of its launches
  cpu_baseline : the reference's own CPU chain (oracle/_ref) or its C restatement on a bounded sample, rank 0, N=1
The other configs of BASELINE.json, each timed for a few steps after the headline (own keys in the same line):
  single_stream : ONE long recording (1 h = 37 440 frames, FIC only) decoded as parallel segments with a warm-up prefix; under
                  torchrun the SAME recording is split over the ranks by sample range (strong scaling), configs[2]'s sharding
  config0       : configs[0], one DAB+ EEP 3-A 72 kbit/s sub-channel + FIC, 96 recordings x 104 frames
  full_ensemble : configs[2]'s ensemble, 18 mixed EEP / UEP sub-channels (864 CU), 96 recordings x 104 frames
  snr_cfo_batch : configs[4], 256 recordings over all ranks, SNR 3..30 dB, carrier offset +-10 kHz
  viterbi_sweep : configs[3], Protection::deconvolve per protection level on reference-generated soft bits, every rank
  h2d_control   : a bare pinned-memory H2D copy of the headline input on every rank at the same time (what bounds e2e)
Scaling of the headline is weak: every rank decodes its own batch, no data-path collective (SURVEY.md section 8e).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_F = 196608
LEAD = 60000   # filler in front of the first null symbol of a synthetic recording (synth.generate's default)
TAIL = 4096
METRIC = "Mode I DAB frames/s decoded (IQ->Viterbi)"
UNIT = "frames/s"
# algorithmic bytes per frame of each kernel family (DESIGN.md section "Kernels")
BYTES_PER_FRAME = {
    "ingest_fft": 77 * 2048 * 2 + 77 * 1536 * 8,   # u8 IQ of the 77 useful parts in, nominal-carrier spectra out
    "demap": 77 * 1536 * 8 + 75 * 3072 * 2,        # spectra in, int16 soft bits out
    "cp_corr": 75 * 2 * 504 * 2,                   # both ends of every cyclic prefix
    "prs_corr": 2048 * 2,
}
KERNEL_NAMES = {"ingest_fft": "k_fft_frames", "demap": "k_demap5", "cp_corr": "k_cp_corr", "prs_corr": "k_prs_corr"}
ACS_PER_FRAME_FIC = 4 * 774 * 64
CPU_CORE_CAP = 64   # the same cap in the native arm's cpu_baseline and in --impl reference


def env_int(name, default):
    return int(os.environ.get(name, default))


def workload_config(args):
    """The `config` object: what is decoded, identical in both arms (everything measured goes into `run`)."""
    return {"workload": f"configs[1] FIC-only decode of a 10k-frame batch: {args.recordings} independent recordings x {args.frames} frames per GPU",
            "recordings_per_gpu": args.recordings, "frames_per_recording": args.frames, "input": "u8 IQ 2.048 MS/s", "snr_db": args.snr,
            "l2": f"no flush between steps: the inputs of a step ({args.recordings * args.frames * 196608 * 2 / 1e9:.1f} GB per GPU) and its intermediates exceed the 126 MB L2"}


# ---------------------------------------------------------------------------------------------- CPU arms
def cpu_worker(args):
    """One process = one recording through the CPU chain (the reference keeps file-scope state: one process each)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from dabstar_b200 import synth
    from oracle_api import Oracle
    o = Oracle(args.cpu_lib)
    rec = synth.generate(args.frames, seed=args.seed, snr_db=args.snr, fmt=synth.FMT_U8)
    iq = o.to_cf32(rec.iq)  # file reader conversion is not part of the timed chain (the reference does it in another thread)
    times, frames = [], 0
    for it in range(args.warmup + args.steps):
        r = o.chain_run(iq, scan_mode=1)
        if it >= args.warmup:
            times.append(r.seconds)
            frames += r.n_frames
        r.close()
    print(json.dumps({"frames": frames, "seconds": sum(times)}))


def run_cpu_chain(kind_lib: str, procs: int, frames: int, steps: int, warmup: int, snr: float, seed0: int = 1000):
    cmds = [[sys.executable, os.path.abspath(__file__), "--cpu-worker", "--cpu-lib", kind_lib, "--frames", str(frames), "--seed", str(seed0 + i),
             "--steps", str(steps), "--warmup", str(warmup), "--snr", str(snr)] for i in range(procs)]
    ps = [subprocess.Popen(c, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for c in cmds]
    tot_frames, max_s = 0, 0.0
    for p in ps:
        out, err = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("cpu worker failed: " + err[-400:])
        d = json.loads(out.strip().splitlines()[-1])
        tot_frames += d["frames"]
        max_s = max(max_s, d["seconds"])
    return tot_frames, max_s


def cpu_libs():
    """[(kind, oracle prefix, description)], fastest first. oracle/_ref travels to the GPU box prebuilt; where it is missing the C
    restatement (oracle/dab_oracle.c) is the CPU arm."""
    from dabstar_b200 import build
    out = []
    if os.path.exists(build.LIB_REF_FAST):
        out.append(("reference", "dabref_fast", "the reference's own sources, fastest configuration that builds here: -O3 -march=x86-64-v3, -DHAVE_VITERBI_AVX2 "
                    "(viterbi_16way.h, not bit exact with the scalar decoder), single-precision radix-4 FFT shim in place of FFTW3f (not installed), scalar OfdmDecoder (the SIMD one needs VOLK)"))
    if os.path.exists(build.LIB_REF):
        out.append(("reference", "dabref", "the reference's own sources, default configuration (scalar Viterbi + scalar OfdmDecoder, -O3), the build the parity tests use"))
    if not out:
        build.build_oracle()
        out.append(("port", "dabo", "C restatement of the reference chain (oracle/dab_oracle.c), scalar"))
    return out


def host_cores():
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return max(1, min(n, CPU_CORE_CAP))


def reference_arm(args, rank, world):
    """The reference's CPU implementation of the same workload on the box's host cores: one process per recording (the reference
    is one thread per stream), as many recordings at a time as there are cores; a step = `cores` of the batch's recordings."""
    if rank != 0:
        return
    kind, lib, what = cpu_libs()[0]
    cores = host_cores()
    t0 = time.time()
    tot, sec = run_cpu_chain(lib, cores, args.frames, args.steps, args.warmup, args.snr, seed0=args.seed)
    value = tot / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * sec / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (random FIB payloads, AWGN)", "gpu_launches": 0, "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "build": what,
                         "sample": f"bounded sample of the batch: {cores} of its recordings per step (one process per recording on {cores} cores, {args.frames} frames each, "
                                   f"the same synthetic generator, seeds and SNR), {args.steps} steps after {args.warmup} warm-up passes ({time.time() - t0:.0f} s wall)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                try:
                    r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------- native arm: helpers
# SURVEY.md section 8(d) config 4: (name, short_form, prot_level, bit_rate, size_cu) — the order of tests/golden/sweep_softbits.npz
SWEEP_PROFILES = [("EEP 1-A 72k", 0, 0, 72, 108), ("EEP 2-A 72k", 0, 1, 72, 72), ("EEP 3-A 72k", 0, 2, 72, 54), ("EEP 4-A 72k", 0, 3, 72, 36),
                  ("EEP 1-B 64k", 0, 4, 64, 54), ("EEP 2-B 64k", 0, 5, 64, 42), ("EEP 3-B 64k", 0, 6, 64, 36), ("EEP 4-B 64k", 0, 7, 64, 30),
                  ("UEP 1 128k", 1, 1, 128, 140), ("UEP 2 128k", 1, 2, 128, 116), ("UEP 3 128k", 1, 3, 128, 96), ("UEP 4 128k", 1, 4, 128, 84),
                  ("UEP 5 128k", 1, 5, 128, 64)]
# configs[2]: 18 mixed EEP / UEP sub-channels filling the 864 CU of a CIF: (short_form, prot_level, bit_rate, size_cu)
FULL_ENSEMBLE = [(0, 0, 72, 108), (0, 1, 72, 72), (0, 2, 72, 54), (0, 3, 72, 36), (0, 4, 64, 54), (0, 5, 64, 42), (0, 6, 64, 36), (0, 7, 64, 30),
                 (1, 3, 128, 96), (1, 4, 128, 84), (1, 5, 128, 64), (0, 2, 48, 36), (0, 2, 32, 24), (0, 6, 32, 18), (1, 5, 32, 16), (0, 3, 32, 16),
                 (0, 2, 8, 6), (1, 4, 64, 42)]


def int_alu_peak_acs(sm_mhz):
    """Integer-ALU issue roofline of the Viterbi kernels: 148 SMs x 128 lanes x f_clk / 4 lane-ops per add-compare-select (SURVEY.md 8d)."""
    return 148 * 128 * sm_mhz * 1e6 / 4.0


def load_sweep_softbits():
    """tests/golden/sweep_softbits.npz with its soft bits decoded: every soft_<level> is stored as an xz stream of little-endian
    int16 (16 logical frames x size_cu * 64), which keeps the file under 1 MB; the other arrays are stored as they are."""
    import lzma
    g = np.load(os.path.join(ROOT, "tests", "golden", "sweep_softbits.npz"))
    out = {k: g[k] for k in g.files}
    for li, (_, _, _, _, cu) in enumerate(SWEEP_PROFILES):
        out[f"soft_{li}"] = np.frombuffer(lzma.decompress(out[f"soft_{li}"].tobytes()), "<i2").astype(np.int16).reshape(-1, cu * 64)
    return out


def prbs_bits(n):
    """Energy-dispersal sequence x^9 + x^5 + 1, all-ones start (backend.cpp:72-83)."""
    reg = [1] * 9
    out = np.zeros(n, np.uint8)
    for i in range(n):
        b = reg[8] ^ reg[4]
        reg = [b] + reg[:8]
        out[i] = b
    return out


def viterbi_sweep(ctx, stream, n_frames, sm_mhz):
    """configs[3]: Protection::deconvolve (depuncture + K=7 Viterbi) over n_frames logical frames per protection level. The soft bits
    are the reference's own (tests/golden/sweep_softbits.npz: its OfdmDecoder output at 12 dB, time de-interleaved, 16 logical frames
    per level; tools/make_sweep_softbits.py), tiled to n_frames and resident in HBM. 3 timed launches after 1 warm-up, CUDA events;
    the decoded bits of the first tile are compared with the reference's Backend output."""
    import ctypes
    import torch
    from dabstar_b200 import api
    gold = load_sweep_softbits()
    out = {"logical_frames_per_level": n_frames, "levels": {}, "input": "reference-generated soft bits (oracle/_ref chain at 12 dB SNR, 16 logical frames per level tiled), resident in HBM",
           "bits_equal_reference": True}
    tot_bits, tot_ms = 0.0, 0.0
    for li, (name, sf, lvl, br, cu) in enumerate(SWEEP_PROFILES):
        tile = torch.from_numpy(np.ascontiguousarray(gold[f"soft_{li}"])).cuda()
        assert tile.shape[1] == cu * 64
        soft = tile.repeat((n_frames + tile.shape[0] - 1) // tile.shape[0], 1)[:n_frames].contiguous()
        bits = torch.empty((n_frames, 24 * br), dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()

        def run():
            ctx.check(ctx.lib.dabstar_protection_deconvolve(ctx.h, sf, br, lvl, cu, ctypes.c_void_p(soft.data_ptr()), n_frames,
                                                            ctypes.c_void_p(bits.data_ptr()), api.MEM_DEVICE), "dabstar_protection_deconvolve")
        run()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(3):
            run()
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 3
        want = np.unpackbits(gold[f"bits_{li}"], axis=1)[:, :24 * br] ^ prbs_bits(24 * br)[None, :]   # Backend output with the energy dispersal put back
        got = bits[-tile.shape[0]:].cpu().numpy() if n_frames % tile.shape[0] == 0 else bits[:tile.shape[0]].cpu().numpy()
        if not np.array_equal(got, want):
            out["bits_equal_reference"] = False
        info_bits = n_frames * 24 * br
        acs = n_frames * 64 * (24 * br + 6)
        out["levels"][name] = {"ms": ms, "mbit_s": info_bits / ms / 1e3, "gacs": acs / ms / 1e6, "frac_int_alu": (acs / ms * 1e3) / int_alu_peak_acs(sm_mhz)}
        tot_bits += info_bits
        tot_ms += ms
        del soft, bits
    out["mbit_s_overall"] = tot_bits / tot_ms / 1e3
    return out


def pin_to_gpu_cpus(local_rank, world):
    """One host control loop per GPU: keep each rank on the CPUs NVML reports as local to its GPU (its NUMA node), and inside
    that set on its own share, so that the ranks do not migrate across sockets or onto each other."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        local = [c for c in range(n_cpu) if (words[c // 64] >> (c % 64)) & 1]
        allowed = sorted(set(local) & set(os.sched_getaffinity(0))) or sorted(os.sched_getaffinity(0))
        # ranks whose GPUs share this CPU set split it evenly
        same = [r for r in range(world) if list(pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(r), (n_cpu + 63) // 64)) == list(words)]
        k, i = max(1, len(allowed) // max(1, len(same))), same.index(local_rank) if local_rank in same else 0
        mine = allowed[i * k:(i + 1) * k] or allowed
        os.sched_setaffinity(0, mine)
        return len(mine)
    except Exception:
        return None


class Timed:
    """A few timed runs of one DabProcessor over device-resident recordings: CUDA events on the context's stream around the
    steps, barrier + synchronize on both sides, max over ranks; stage and MSC-kernel times summed over the steps."""

    def __init__(self, stream, world, dist):
        self.stream, self.world, self.dist = stream, world, dist

    def barrier(self):
        import torch
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def reduce(self, ms, frames):
        import torch
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        f = torch.tensor([float(frames)], dtype=torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            self.dist.all_reduce(f, op=self.dist.ReduceOp.SUM)
        return t.item(), f.item()

    def run(self, dp, ptrs, ns, steps, warmup=1):
        import torch
        from dabstar_b200 import api
        step = dp.prepared(ptrs, ns, api.MEM_DEVICE)
        for _ in range(warmup):
            step()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record(self.stream)
        for _ in range(steps):
            step()
        e1.record(self.stream)
        self.barrier()
        ms = e0.elapsed_time(e1) / steps
        # the last of the timed runs gives the per-kernel-family times (they are read back outside the timed region)
        stages = {k: v[0] for k, v in dp.stage_ms().items() if v[0] > 0}
        msc = list(dp.msc_kernel_ms())
        return ms, stages, msc


FRAME_INFO_FIELDS = ("sym0_pos", "start_index", "fbb_sym0", "fbb_data", "fbb_null", "fsync", "phase_cp", "clock_err", "fic_ratio_before", "fic_ratio_after")
DUMP_RECORDING_BYTES = 40 << 20   # budget of the per-recording arrays; beyond it a seeded subset of the recordings is written
DUMP_SOFT_FRAMES = 16             # (recording, frame) pairs of soft_bits_sample.npy (14 MB), drawn with a fixed seed


def dump_outputs(dp, R, F, out_dir):
    """Writes what the headline decode returned to its caller for the batch's last run, as float32 / float64 .npy files under
    out_dir (30 MB at the default sizes, at most 54 MB): for the recordings listed in recordings.npy (all of them unless that
    would pass the budget) the frame count, the FrameInfo fields of every frame (last axis of frame_info.npy in the order of
    FRAME_INFO_FIELDS), the FIC CRC flags, the packed FIB bytes and the counters; and the soft bits of a seeded sample of frames
    (soft_bits_sample_index.npy: recording, frame). Frames a recording did not decode are NaN, so two builds can be compared
    array for array even where their frame counts differ."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    per_recording = F * (12 * 32 * 4 + len(FRAME_INFO_FIELDS) * 8 + 4 * 4) + 8 * 8 + 8
    rows = np.arange(R)
    if R * per_recording > DUMP_RECORDING_BYTES:
        rows = np.sort(rng.choice(R, max(1, DUMP_RECORDING_BYTES // per_recording), replace=False))
    res = [dp.result(int(r)) for r in rows]
    nf = np.array([x.n_frames for x in res], np.float64)
    n_max = max(1, int(nf.max()))
    info = np.full((len(rows), n_max, len(FRAME_INFO_FIELDS)), np.nan, np.float64)
    valid = np.full((len(rows), n_max, 4), np.nan, np.float32)
    fib = np.full((len(rows), n_max, 12, 32), np.nan, np.float32)
    for j, (r, x) in enumerate(zip(rows, res)):
        if not x.n_frames:   # a recording without a decoded frame stays NaN
            continue
        info[j, :x.n_frames] = [[getattr(i, k) for k in FRAME_INFO_FIELDS] for i in x.info]
        valid[j, :x.n_frames] = x.fic_valid
        fib[j, :x.n_frames] = dp.fib_packed(int(r))
    pick = np.stack([rng.integers(0, R, DUMP_SOFT_FRAMES), rng.integers(0, F, DUMP_SOFT_FRAMES)], axis=1)
    soft = np.full((DUMP_SOFT_FRAMES, 75, 3072), np.nan, np.float32)
    for j, (r, f) in enumerate(pick):
        if f < dp.n_frames(int(r)):
            soft[j] = dp.soft_bits(int(r), int(f))
    arrays = {"recordings": rows.astype(np.float64), "n_frames": nf, "frame_info": info, "fic_valid": valid, "fib_packed": fib,
              "counters": np.stack([x.counters for x in res]).astype(np.float64), "soft_bits_sample_index": pick.astype(np.float64),
              "soft_bits_sample": soft}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def replicated_recordings(uniq, copies):
    """[len(uniq) * copies, n, 2] u8 on the device: physical copies, so that the inputs exceed the L2 as independent recordings do."""
    import torch
    host = torch.from_numpy(np.stack([u.iq for u in uniq]))
    return host.cuda().repeat(copies, 1, 1).contiguous()


def msc_workload(T, ctx, args, subch, name, sm_mhz, seed0):
    """R recordings x F frames with the sub-channels `subch`, every sub-channel of every CIF decoded (configs[0] / configs[2])."""
    import torch
    from dabstar_b200 import api, synth
    R, F, U = args.recordings, args.frames, 4
    uniq = [synth.generate(F, seed=seed0 + i, snr_db=args.snr, subch=subch, fmt=synth.FMT_U8) for i in range(U)]
    dev = replicated_recordings(uniq, (R + U - 1) // U)[:R]
    dp = api.DabProcessor(R, input_format=api.FMT_U8, max_window=args.window, ctx=ctx)
    for r in range(R):
        dp.set_audio_channel(r, subch)
    ptrs, ns = [dev[r].data_ptr() for r in range(R)], [dev.shape[1]] * R
    ms, stages, msc = T.run(dp, ptrs, ns, args.extra_steps)
    frames = sum(dp.n_frames(r) for r in range(R))
    res = dp.result(1)
    ok = all(np.array_equal(res.msc[s.sub_ch_id], uniq[1].msc_truth[j][:res.msc[s.sub_ch_id].shape[0]]) for j, s in enumerate(subch))
    ms, tot_frames = T.reduce(ms, frames)
    info_bits = frames * (3072 + 4 * 24 * sum(s.bit_rate for s in subch))
    acs_msc = frames * 4 * sum(64 * (24 * s.bit_rate + 6) for s in subch)
    out = {"workload": name, "recordings_per_gpu": R, "frames_per_recording": F, "unique_recordings": U, "frames_per_step_all_gpus": tot_frames, "steps": args.extra_steps,
           "ms_per_step": ms, "frames_per_s": tot_frames / ms * 1e3, "decoded_mbit_s_per_gpu": info_bits / ms / 1e3, "payload_equals_transmitted": bool(ok),
           "stages_ms": stages, "msc_gather_ms": msc[0], "msc_trellis_ms": msc[1]}
    if msc[1] > 0:
        out["msc_trellis_gacs"] = acs_msc / msc[1] / 1e6
        out["msc_trellis_frac_int_alu"] = (acs_msc / msc[1] * 1e3) / int_alu_peak_acs(sm_mhz)
    if msc[0] > 0:
        # the gather reads every soft bit of the sub-channels once (2 B) and writes one byte per kept symbol position (4 per trellis step)
        gb = frames * 4 * sum(s.size_cu * 64 * 2 + 4 * (24 * s.bit_rate + 6) for s in subch)
        out["msc_gather_gbs"] = gb / msc[0] / 1e6
    del dp, dev
    torch.cuda.empty_cache()
    return out


def snr_cfo_workload(T, ctx, args, rank, world):
    """configs[4]: 256 independent recordings over all ranks, SNR 3..30 dB, carrier offset within +-10 kHz: time sync, coarse AFC,
    re-synchronisation after FIC failures (dab_processor.cpp:144-182) under load."""
    import torch
    from dabstar_b200 import api, synth
    total, F = 256, args.snr_cfo_frames
    R = max(1, total // world)
    U = min(R, 64)
    snr = np.linspace(3.0, 30.0, U)
    cfo = np.array([((-1) ** i) * (250.0 + 9750.0 * ((i * 7) % U) / max(U - 1, 1)) for i in range(U)])
    uniq = [synth.generate(F, seed=5000 + 97 * rank + i, snr_db=float(snr[i]), cfo_hz=float(cfo[i]), fmt=synth.FMT_U8) for i in range(U)]
    dev = replicated_recordings(uniq, (R + U - 1) // U)[:R]
    dp = api.DabProcessor(R, input_format=api.FMT_U8, scan_mode=True, max_window=args.window, ctx=ctx)
    ptrs, ns = [dev[r].data_ptr() for r in range(R)], [dev.shape[1]] * R
    ms, stages, _ = T.run(dp, ptrs, ns, args.extra_steps)
    cnt = np.stack([dp.counters(r) for r in range(R)])
    frames = int(cnt[:, 6].sum())
    hi = [r for r in range(R) if snr[r % U] >= 10.0]
    ms, tot_frames = T.reduce(ms, frames)
    out = {"workload": "configs[4] batch of 256 independent recordings, SNR 3..30 dB, carrier offset +-10 kHz, FIC decode", "recordings_all_gpus": R * world,
           "recordings_per_gpu": R, "unique_recordings_per_gpu": U, "frames_per_recording": F, "frames_decoded_all_gpus": tot_frames, "steps": args.extra_steps,
           "ms_per_step": ms, "frames_per_s": tot_frames / ms * 1e3,
           "rank0": {"fib_crc_pass": float(cnt[:, 0].sum()) / max(1.0, 12.0 * frames),
                     "fib_crc_pass_snr_ge_10db": float(cnt[hi, 0].sum()) / max(1.0, 12.0 * float(cnt[hi, 6].sum())),
                     "time_syncs": int(cnt[:, 1].sum()), "time_sync_failures": int(cnt[:, 2].sum()), "windows_run": int(cnt[:, 4].sum()),
                     "windows_cut_by_verification": int(cnt[:, 5].sum()), "frames_through_heavy_pass": int(cnt[:, 7].sum())},
           "stages_ms": stages}
    del dp, dev
    torch.cuda.empty_cache()
    return out


def two_batches_workload(T, args, local_rank, dp, d_ptrs, ns, frames_per_step, good_fibs):
    """configs[1] as a stream of batches: a second decoder (own context, own stream, own host thread) decodes the same resident
    recordings while the first one runs, so one batch's time sync, layout passes and host control fall into the other batch's
    FFT / demapper time. Not the headline (`value` stays one batch at a time); wall clock around the synchronous calls."""
    import threading
    import torch
    from dabstar_b200 import api
    R = len(d_ptrs)
    stream2 = torch.cuda.Stream()
    ctx2 = api.Context(local_rank, stream=stream2)
    dp2 = api.DabProcessor(R, input_format=api.FMT_U8, scan_mode=True, max_window=args.window, ctx=ctx2)
    calls = [dp.prepared(d_ptrs, ns, api.MEM_DEVICE), dp2.prepared(d_ptrs, ns, api.MEM_DEVICE)]
    for _ in range(2):
        calls[1]()
    n = max(2, args.extra_steps)
    err = []

    def work(i):
        try:
            for _ in range(n):
                calls[i]()
        except Exception as e:  # noqa: BLE001 - reported in the bench line
            err.append(repr(e))

    torch.cuda.synchronize()
    T.barrier()
    t0 = time.perf_counter()
    th = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    torch.cuda.synchronize()
    ms, _ = T.reduce((time.perf_counter() - t0) * 1e3, 0)
    good2 = int(np.sum([dp2.counters(r) for r in range(R)], axis=0)[0])
    out = {"workload": "configs[1], two batches of the same recordings in flight (two decoders, streams and host threads)", "batches": 2 * n,
           "ms_per_batch": ms / (2 * n), "frames_per_s_per_gpu": 2 * n * frames_per_step / (ms / 1e3), "good_fibs_equal": good2 == good_fibs,
           "timing": "wall clock around the synchronous decode calls, max over ranks"}
    if err:
        out["error"] = err[0]
    del dp2
    return out


def single_stream_workload(T, ctx, args, rank, world, uniq_dev):
    """configs[1] read as ONE stream / configs[2]'s sharding: a 1 h recording (args.stream_frames frames, FIC only) whose frames are
    the tiled frames of the first recordings of rank 0's batch (every rank synthesises the same ones). One GPU demaps each verified
    window as parallel segments with a warm-up prefix (dabstar_decoder_set_segmentation); N ranks split the SAME stream by sample
    range (parallel.stream_shard: cold start + warm-up frames in front of each range), so the total work is fixed: strong scaling.
    Redundant frames (segment warm-ups, the ranks' lead-in) are reported and NOT counted as decoded."""
    import torch
    from dabstar_b200 import api, parallel
    F = args.frames
    L = F * T_F
    U = uniq_dev.shape[0]
    tiles = max(1, args.stream_frames // F)
    n_total = LEAD + tiles * L + TAIL
    sh = parallel.stream_shard(n_total, rank, world, warmup_frames=args.segment_warmup)

    def piece(lo, hi):   # samples [lo, hi) of the stream
        parts = []
        s = lo
        while s < hi:
            if s < LEAD:
                e = min(hi, LEAD)
                parts.append(uniq_dev[0, s:e])
            elif s < LEAD + tiles * L:
                t, o = divmod(s - LEAD, L)
                e = min(hi, LEAD + (t + 1) * L)
                parts.append(uniq_dev[t % U, LEAD + o:LEAD + o + (e - s)])
            else:
                e = hi
                o = s - (LEAD + tiles * L)
                parts.append(uniq_dev[0, LEAD + L + o:LEAD + L + o + (e - s)])
            s = e
        return torch.cat(parts).contiguous()

    dev = piece(sh.in_lo, sh.in_hi)
    dp = api.DabProcessor(1, input_format=api.FMT_U8, scan_mode=True, max_window=args.stream_window, ctx=ctx)
    # segments per window: about 96 (288 demapper CTAs fill the 148 SMs twice); a rank whose share is shorter than a full
    # window takes shorter segments (more warm-up frames per decoded frame, reported as redundant) instead of leaving SMs empty
    seg_frames = args.stream_segment_frames
    if seg_frames <= 0:
        share = min(args.stream_window, (tiles * F + world - 1) // world)
        seg_frames = max(32, min(104, (share + 95) // 96))
    dp.set_segmentation(seg_frames, args.segment_warmup)
    ptrs, ns = [dev.data_ptr()], [dev.shape[0]]
    ms, stages, _ = T.run(dp, ptrs, ns, args.extra_steps)
    first, last = parallel.owned_frames(dp.frame_positions(0), sh)
    cnt = dp.counters(0)
    decoded, warm = dp.n_frames(0), dp.warmup_frames(0)
    ms, owned = T.reduce(ms, last - first)
    _, redundant = T.reduce(0.0, decoded - (last - first) + warm)
    _, good = T.reduce(0.0, float(cnt[0]))
    _, dec_all = T.reduce(0.0, decoded)
    out = {"workload": f"one {tiles * F}-frame recording ({tiles * F * 0.096 / 60:.0f} min), FIC only, decoded as frame batches with a warm-up prefix",
           "scaling": "strong", "frames": owned, "frames_expected": tiles * F, "steps": args.extra_steps, "ms_per_step": ms, "frames_per_s": owned / ms * 1e3,
           "x_real_time": owned / ms * 1e3 / (2048000 / T_F),
           "segment_frames": seg_frames, "segment_warmup_frames": args.segment_warmup, "window": args.stream_window,
           "redundant_frames": redundant, "redundant_fraction": redundant / max(1.0, owned),
           "fib_crc_pass_incl_lead_in": min(1.0, good / max(1.0, 12.0 * dec_all)),   # (FIBs of a trailing incomplete frame count as good, not as a frame)
           "rank0": {"samples": int(dev.shape[0]), "frames_decoded": int(decoded), "frames_owned": int(last - first), "segment_warmup_frames_demapped": int(warm),
                     "windows_run": int(cnt[4]), "windows_cut_by_verification": int(cnt[5])},
           "stages_ms": stages,
           "note": "soft bits of warm-started segments are approximations (tests/test_long_recordings.py: FIB / MSC bytes identical to the sequential oracle run, "
                   "soft bits beyond 1 LSB 4e-2 / 5e-8 / 0 for warm-up 4 / 18 / 32 frames)"}
    del dp, dev
    torch.cuda.empty_cache()
    return out


def h2d_control(T, host, world):
    """A bare cudaMemcpyAsync of the headline's pinned input on every rank at the same time: the host -> device ceiling of the box
    at N ranks, which is what bounds `e2e`."""
    import torch
    dst = torch.empty_like(host, device="cuda")
    dst.copy_(host, non_blocking=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    T.barrier()
    e0.record()
    for _ in range(2):
        dst.copy_(host, non_blocking=True)
    e1.record()
    T.barrier()
    ms = e0.elapsed_time(e1) / 2
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        T.dist.all_reduce(t, op=T.dist.ReduceOp.MAX)
    nbytes = host.numel() * host.element_size()
    del dst
    return {"bytes_per_rank": int(nbytes), "ms_max_over_ranks": t.item(), "gbs_per_rank": nbytes / t.item() / 1e6, "gbs_all_ranks": world * nbytes / t.item() / 1e6,
            "what": "torch copy_ from pinned host memory (one contiguous cudaMemcpyAsync), all ranks concurrently, 2 repetitions"}


# ---------------------------------------------------------------------------------------------- native arm
def native_arm(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from dabstar_b200 import api, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the decode path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pinned_cpus = pin_to_gpu_cpus(local_rank, world) if world > 1 and not args.no_cpu_affinity else None
    R, F = args.recordings, args.frames
    n_samples = LEAD + F * T_F + TAIL
    S_UNIQ = min(8, R)   # recordings with rank-independent seeds: the frames of the shared single stream

    # ---- synthetic recordings in pinned host memory, every one from its own seed: the same arguments give the same input
    host = torch.empty((R, n_samples, 2), dtype=torch.uint8, pin_memory=True)
    hnp = host.numpy()
    for r in range(R):
        seed = args.seed + r if r < S_UNIQ else args.seed + 7919 * rank + r
        synth.generate(F, seed=seed, snr_db=args.snr, fmt=synth.FMT_U8, out=hnp[r])
    dev = host.cuda(non_blocking=False)
    stream = torch.cuda.Stream()
    ctx = api.Context(local_rank, stream=stream)
    dp = api.DabProcessor(R, input_format=api.FMT_U8, scan_mode=True, max_window=args.window, ctx=ctx)
    if args.segment_frames > 0:
        dp.set_segmentation(args.segment_frames, args.segment_warmup)
    d_ptrs = [dev[r].data_ptr() for r in range(R)]
    h_ptrs = [host[r].data_ptr() for r in range(R)]
    ns = [n_samples] * R
    T = Timed(stream, world, dist)
    extras = {}

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            dp.run_ptrs(d_ptrs, ns, api.MEM_DEVICE)
        # ---- timed: inputs resident in HBM
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clocks = ClockSampler(local_rank)
        T.barrier()
        clocks.start()
        launches0 = ctx.kernel_launches
        step_dev = dp.prepared(d_ptrs, ns, api.MEM_DEVICE)   # the ctypes argument arrays are built once, outside the timed region
        e0.record(stream)
        for _ in range(args.steps):
            step_dev()
        e1.record(stream)
        T.barrier()
        clk = clocks.stop()
        ms_total = e0.elapsed_time(e1)
        launches = ctx.kernel_launches - launches0
        cnt = np.sum([dp.counters(r) for r in range(R)], axis=0)   # of the last timed step
        frames_per_step = int(cnt[6])
        good_fibs = int(cnt[0])
        if args.dump_outputs and rank == 0:
            dump_outputs(dp, R, F, args.dump_outputs)
        # ---- the same steps again, untimed, for the per-kernel-family CUDA-event times (reading them back after every run costs
        #      host time that is not part of the decode)
        stage_acc = {}
        heavy_acc = [0.0, 0.0]
        for _ in range(args.steps):
            step_dev()
            heavy_acc[0] += dp.heavy_ms(False)
            heavy_acc[1] += dp.heavy_ms(True)
            for k, (ms, ln) in dp.stage_ms().items():
                a = stage_acc.setdefault(k, [0.0, 0])
                a[0] += ms
                a[1] += ln
        # ---- timed: end to end from pinned host memory (H2D of the IQ and D2H of the FIB bits inside the call)
        step_host = dp.prepared(h_ptrs, ns, api.MEM_HOST)
        step_host()
        T.barrier()
        e0.record(stream)
        for _ in range(args.steps):
            step_host()
            _ = dp.fib_packed(0)
        e1.record(stream)
        T.barrier()
        ms_e2e = e0.elapsed_time(e1)
        sm_mhz = clk.get("sm_mhz") or clk.get("sm_max_mhz") or 1965.0
        if not args.no_extras:
            extras["two_batches_in_flight"] = two_batches_workload(T, args, local_rank, dp, d_ptrs, ns, frames_per_step, good_fibs)
        del dp

        # ---- the other configs (a few steps each)
        if not args.no_extras:
            extras["h2d_control"] = h2d_control(T, host, world)
            extras["single_stream"] = single_stream_workload(T, ctx, args, rank, world, dev[:S_UNIQ])
            del dev
            torch.cuda.empty_cache()
            extras["snr_cfo_batch"] = snr_cfo_workload(T, ctx, args, rank, world)
            extras["config0"] = msc_workload(T, ctx, args, [synth.SubChannel(3, 100, 54, 0, 2, 72)],
                                             "configs[0] one DAB+ EEP 3-A 72 kbit/s sub-channel + FIC, every CIF decoded", sm_mhz, 300)
            fe, cu = [], 0
            for i, (sf, lvl, br, size) in enumerate(FULL_ENSEMBLE):
                fe.append(synth.SubChannel(i + 1, cu, size, sf, lvl, br))
                cu += size
            extras["full_ensemble"] = msc_workload(T, ctx, args, fe, "configs[2] full ensemble: 18 mixed EEP / UEP sub-channels (864 CU), every sub-channel of every CIF decoded", sm_mhz, 900)
        # ---- configs[3]: Viterbi-only throughput per protection level on every rank (the "Viterbi Mbit/s" half of the metric)
        vit_sweep = None
        if not args.no_viterbi_sweep:
            vit_sweep = viterbi_sweep(ctx, stream, args.viterbi_frames, sm_mhz)
            if world > 1:
                t = torch.tensor([vit_sweep["mbit_s_overall"]], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.SUM)
                vit_sweep["mbit_s_overall_all_gpus"] = t.item()
                vit_sweep["note"] = "levels: rank 0's GPU; mbit_s_overall_all_gpus: sum over the ranks, every rank runs the sweep on its own GPU at the same time"

    t = torch.tensor([ms_total, ms_e2e], dtype=torch.float64, device="cuda")
    fr = torch.tensor([frames_per_step], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(fr, op=dist.ReduceOp.SUM)
    ms_total, ms_e2e = t.tolist()
    total_frames = fr.item()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    value = total_frames * args.steps / (ms_total / 1e3)
    e2e_value = total_frames * args.steps / (ms_e2e / 1e3)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (of fallback)"
    stages = {}
    for k, (ms, ln) in stage_acc.items():
        if ln == 0:
            continue
        d = {"ms_per_step": ms / args.steps, "launches_per_step": ln / args.steps}
        if k in BYTES_PER_FRAME:
            gbs = BYTES_PER_FRAME[k] * frames_per_step * args.steps / (ms / 1e3) / 1e9
            d.update({"achieved_gbs": gbs, "frac_hbm": gbs / hbm_peak})
        if k == "fic_viterbi":
            acs = ACS_PER_FRAME_FIC * frames_per_step * args.steps / (ms / 1e3)
            d.update({"achieved_gacs": acs / 1e9, "frac_int_alu": acs / int_alu_peak_acs(sm_mhz), "mbit_s": 3072 * frames_per_step * args.steps / (ms / 1e3) / 1e6})
        stages[k] = d
    # the FFT + demap STAGE as one span (its chunks may overlap on two streams), against SURVEY.md 8(d)'s stage bytes: 76 symbols +
    # null symbol of spectra in, soft bits out = 1 722 368 B per frame
    stage_bytes = 77 * 2048 * 8 + 75 * 3072 * 2
    gbs = stage_bytes * frames_per_step * args.steps / (max(heavy_acc[0], 1e-9) / 1e3) / 1e9
    stages["fft_demap_stage"] = {"ms_per_step": heavy_acc[0] / args.steps, "with_fic_ms_per_step": heavy_acc[1] / args.steps, "algorithmic_bytes_per_frame": stage_bytes,
                                 "achieved_gbs_stage": gbs, "frac_hbm_stage": gbs / hbm_peak,
                                 "note": "first FFT launch to last demap launch of every window, CUDA events; the per-kernel times above may overlap"}
    kernel_ms = sum(v["ms_per_step"] for k, v in stages.items() if k != "fft_demap_stage")
    hbm_stages = {k: v for k, v in stages.items() if "achieved_gbs" in v}
    dom = max(hbm_stages, key=lambda k: hbm_stages[k]["ms_per_step"])
    roofline = {"kernel": KERNEL_NAMES[dom], "bound": "hbm",
                "achieved": hbm_stages[dom]["achieved_gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": hbm_stages[dom]["frac_hbm"], "traffic": None,
                "peak_source": peak_src, "algorithmic_bytes_per_frame": BYTES_PER_FRAME[dom]}
    # achieved / traffic are per launch: algorithmic bytes of one launch over its average CUDA-event duration
    n_launch = max(1.0, hbm_stages[dom]["launches_per_step"])
    roofline["algorithmic_bytes_per_launch"] = BYTES_PER_FRAME[dom] * frames_per_step / n_launch
    roofline["ms_per_launch"] = hbm_stages[dom]["ms_per_step"] / n_launch
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        k = tr["kernels"].get(roofline["kernel"])
        if k and n_launch == 1.0 and int(tr["frames_per_launch"]) == int(frames_per_step):
            roofline["traffic"] = k["dram_read_bytes"] + k["dram_write_bytes"]
            roofline["traffic_source"] = tr["source"] + " (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum, same workload)"
    except Exception:
        pass

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        libs = cpu_libs()
        cores = host_cores()
        t0 = time.time()
        kind, lib, what = libs[0]
        tot, sec = run_cpu_chain(lib, cores, F, 2, 1, args.snr, seed0=args.seed)
        cpu = {"value": tot / sec, "unit": UNIT, "cores": cores, "kind": kind, "build": what,
               "sample": f"bounded sample of the batch: {cores} of its recordings (one process per recording on {cores} cores, {F} frames each, same seeds and SNR), 2 passes after 1 warm-up"}
        if len(libs) > 1:   # second column: the default (scalar, parity) build of the same sources
            kind2, lib2, what2 = libs[1]
            tot2, sec2 = run_cpu_chain(lib2, cores, F, 1, 1, args.snr, seed0=args.seed)
            cpu["default_build"] = {"value": tot2 / sec2, "unit": UNIT, "cores": cores, "kind": kind2, "build": what2, "sample": "the same recordings, 1 pass after 1 warm-up"}
        cpu["sample"] += f" ({time.time() - t0:.0f} s wall for both builds)"

    cfg = workload_config(args)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": f"synthetic ({R} unique recordings per GPU of {R}, random FIB payloads, AWGN {args.snr} dB)",
        "config": cfg,
        "run": {"frames_per_step_all_gpus": total_frames, "input_bytes_per_gpu": int(R * n_samples * 2),
                "l2": "inputs (3.9 GB) and intermediates far exceed the 126 MB L2", "window": args.window, "cpus_per_rank": pinned_cpus,
                "fib_crc_pass": good_fibs / max(1.0, 12.0 * frames_per_step), "windows_per_recording": float(cnt[4]) / R,
                "frames_through_heavy_pass": int(cnt[7]), "x_real_time": value / world / (2048000 / T_F),
                "kernel_ms_per_step": kernel_ms, "host_control_ms_per_step": ms_total / args.steps - kernel_ms},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(R * n_samples * 2), "d2h_bytes_per_step": int(frames_per_step * 384),
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches), "clocks": clk, "roofline": roofline, "stages": stages, "viterbi_sweep": vit_sweep, "cpu_baseline": cpu,
    }
    line.update(extras)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--recordings", type=int, default=96)
    ap.add_argument("--frames", type=int, default=104)
    ap.add_argument("--window", type=int, default=128)
    ap.add_argument("--seed", type=int, default=2)
    ap.add_argument("--snr", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-viterbi-sweep", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="only the headline workload (configs[1]) and the Viterbi sweep")
    ap.add_argument("--no-cpu-affinity", action="store_true", help="N > 1: do not pin each rank to the CPUs local to its GPU")
    ap.add_argument("--viterbi-frames", type=int, default=1048576, help="logical frames per protection level in the Viterbi-only sweep")
    ap.add_argument("--extra-steps", type=int, default=3, help="timed steps of each of the other configs")
    ap.add_argument("--segment-frames", type=int, default=0, help="headline: demap a recording's window as parallel segments of this many frames (0 = off)")
    ap.add_argument("--segment-warmup", type=int, default=18)
    ap.add_argument("--stream-frames", type=int, default=37440, help="single_stream: frames of the one long recording (1 h)")
    ap.add_argument("--stream-window", type=int, default=9984)
    ap.add_argument("--stream-segment-frames", type=int, default=0, help="single_stream: frames per demapper segment (0 = about 96 segments per window, 32..104 frames)")
    ap.add_argument("--snr-cfo-frames", type=int, default=13)
    ap.add_argument("--dump-outputs", metavar="DIR", help="native arm only: after the timed headline steps, write what the last step decoded (rank 0) as .npy files to DIR")
    ap.add_argument("--cpu-worker", action="store_true")
    ap.add_argument("--cpu-lib", default="dabo")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the native arm's decoded outputs; --impl reference has none to write")
    if args.cpu_worker:
        return cpu_worker(args)
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    if args.impl == "reference":
        return reference_arm(args, rank, world)
    if world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun as the driver does
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    native_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
