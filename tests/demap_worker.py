"""One demapper configuration in a process of its own (used by test_gpu_demap_shapes.py; not collected as tests).

The demapper's output lag (k_demap5<SOFT, LAG>) is read from DABSTAR_DEMAP_LAG once per process, on the first launch, and
DABSTAR_TRACE prints the engine's round lines to stderr: both need a fresh process with the environment set. The caller
sets them, runs

    python demap_worker.py MODE IN_DIR OUT_DIR

and reads OUT_DIR/out.npz (plus OUT_DIR/soft.npy for the batch and the segment modes). MODE:

* tap      OfdmDecoder.decode_frames on IN_DIR/in.npz (fft, clock_err, tii) for soft_bit_type 0 / 1 / 2: six frames with one
           TII null symbol, a one-frame call, and the six frames as a continuation over two calls on the same state;
* batch    DabProcessor over the 256 copies of the batch_source() recordings, then every source decoded alone;
* segments DabProcessor with set_segmentation over segment_recording(); IN_DIR/in.npz holds segment_frames, warmup and
           max_window.
"""
from __future__ import annotations

import contextlib
import hashlib
import os
import re
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from dabstar_b200 import synth  # noqa: E402

# ---- the batch: 256 recordings past one wave of demapper CTAs (768 CTAs; 2 / 3 / 4 per SM at lag 15 / 7 / 3 on 148 SMs)
N_SRC, N_COPIES, N_FULL = 32, 256, 6
K_CUT = (1, 2, 3, 4, 7, 8, 15, 16, 40, 74)  # data symbols the recording's last frame still holds
LEAD = 60000                                # synth.generate's default lead_samples
F_MAX = N_FULL + 2                          # padding of the per-frame arrays


def batch_source(i: int) -> tuple[np.ndarray, int]:
    """Source i of the batch: N_FULL complete frames and a last frame cut after K_CUT[i % 10] data symbols (plus half a symbol),
    SNR 12..30 dB, carrier offset within +-5 kHz. Returns (uint8[n, 2] samples, k)."""
    snr = 12.0 + 18.0 * i / (N_SRC - 1)
    cfo = (-1) ** i * (150.0 + 4850.0 * ((i * 11) % N_SRC) / (N_SRC - 1))
    k = K_CUT[i % len(K_CUT)]
    rec = synth.generate(N_FULL + 1, seed=7000 + i, snr_db=snr, cfo_hz=cfo, fmt=synth.FMT_U8, lead_samples=LEAD)
    # frame f: null symbol (2656 samples) at LEAD + f * T_FRAME, then symbol 0 and the data symbols (2552 samples each)
    cut = LEAD + N_FULL * synth.T_FRAME + 2656 + 2552 + k * 2552 + 1276
    return np.ascontiguousarray(rec.iq[:cut]), k


def segment_recording() -> np.ndarray:
    """The clean long recording of the segmented-decode checks: 400 frames, 15 dB, no carrier offset."""
    return synth.generate(400, seed=31, snr_db=15.0, fmt=synth.FMT_U8).iq


ROUND_RE = re.compile(r"\[dabstar\] round (\d+) t=[0-9.]+ ms: (\d+) recordings, (\d+) frames")


def parse_rounds(text: str) -> np.ndarray:
    """(recordings, frames) of every round line DABSTAR_TRACE printed."""
    return np.array([(int(m.group(2)), int(m.group(3))) for m in ROUND_RE.finditer(text)], np.int64).reshape(-1, 2)


@contextlib.contextmanager
def stderr_to(path: str):
    """File descriptor 2 (where the library prints its trace) into `path` for the duration."""
    sys.stderr.flush()
    saved = os.dup(2)
    fd = os.open(path, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644)
    os.dup2(fd, 2)
    os.close(fd)
    try:
        yield
    finally:
        sys.stderr.flush()
        os.dup2(saved, 2)
        os.close(saved)


def traced(path: str, fn):
    with stderr_to(path):
        fn()
    with open(path) as f:
        text = f.read()
    sys.stderr.write(text)
    return parse_rounds(text)


def result_arrays(dp, r: int) -> dict:
    """What a recording's result holds, as fixed-shape arrays (frames beyond n_frames are -1 / 0)."""
    res = dp.result(r)
    n = res.n_frames
    assert n <= F_MAX, n
    pos = np.full((F_MAX, 2), -1, np.int64)
    fbb = np.zeros((F_MAX, 2), np.float32)
    ce = np.zeros(F_MAX, np.float32)
    valid = np.zeros((F_MAX, 4), np.uint8)
    fib = np.zeros((F_MAX, 3072), np.uint8)
    for f, i in enumerate(res.info):
        pos[f] = (i.sym0_pos, i.start_index)
        fbb[f] = (i.fbb_data, i.fbb_null)
        ce[f] = i.clock_err
    valid[:n] = res.fic_valid
    fib[:n] = res.fib_bits
    return dict(n_frames=n, pos=pos, fbb=fbb, clock_err=ce, fic_valid=valid, fib=fib, counters=res.counters)


def batch_results(dp) -> dict:
    """result_arrays of every recording of a batch, stacked."""
    per = [result_arrays(dp, r) for r in range(dp.n)]
    return {k: np.stack([p[k] for p in per]) for k in per[0]}


def digest(a: np.ndarray) -> np.ndarray:
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def decode_batch(ctx, srcs: list[np.ndarray], soft_bit_type: int, trace_path: str | None = None):
    """The 256 copies (copy i from source i % N_SRC, physical copies on the device) in one DabProcessor, scan mode.
    Returns (processor, round table or None, device buffers)."""
    import torch
    from dabstar_b200 import api
    dev = [torch.from_numpy(srcs[i % N_SRC]).cuda() for i in range(N_COPIES)]
    torch.cuda.synchronize()
    dp = api.DabProcessor(N_COPIES, input_format=api.FMT_U8, soft_bit_type=soft_bit_type, scan_mode=True, ctx=ctx)

    def run():
        dp.run_ptrs([t.data_ptr() for t in dev], [t.shape[0] for t in dev], api.MEM_DEVICE)
    rounds = None
    if trace_path:
        rounds = traced(trace_path, run)
    else:
        run()
    return dp, rounds, dev


def soft_of(dp, r: int) -> np.ndarray:
    n = dp.n_frames(r)
    return np.stack([dp.soft_bits(r, f) for f in range(n)]) if n else np.zeros((0, 75, 3072), np.int16)


def mode_tap(ctx, inp, out_dir):
    from dabstar_b200 import api
    fft, ce, tii = inp["fft"], inp["clock_err"], inp["tii"]
    out = {}
    for st in (0, 1, 2):
        dec = api.OfdmDecoder(st, ctx)
        out[f"full_soft_{st}"] = dec.decode_frames(fft, ce, tii)
        out[f"full_state_{st}"] = np.concatenate([dec.state(w) for w in range(6)])
        out[f"full_quality_{st}"] = np.array([dec.quality()[k] for k in api.OfdmDecoder.QUALITY], np.float32)
        dec = api.OfdmDecoder(st, ctx)
        out[f"one_soft_{st}"] = dec.decode_frames(fft[:1], ce[:1])
        out[f"one_state_{st}"] = np.concatenate([dec.state(w) for w in range(6)])
        dec = api.OfdmDecoder(st, ctx)
        a = dec.decode_frames(fft[:3], ce[:3], tii[:3])
        b = dec.decode_frames(fft[3:], ce[3:], tii[3:])
        out[f"cont_soft_{st}"] = np.concatenate([a, b])
        out[f"cont_state_{st}"] = np.concatenate([dec.state(w) for w in range(6)])
    np.savez(os.path.join(out_dir, "out.npz"), **out)


def mode_batch(ctx, inp, out_dir):
    from dabstar_b200 import api
    srcs = [batch_source(i)[0] for i in range(N_SRC)]
    dp, rounds, dev = decode_batch(ctx, srcs, 0, os.path.join(out_dir, "trace.txt"))
    out = batch_results(dp)
    out["rounds"] = rounds
    # soft bits of the first copy of every source; a digest per frame of every copy
    soft = np.zeros((N_SRC, F_MAX, 75, 3072), np.int16)
    dig = np.zeros((N_COPIES, F_MAX, 32), np.uint8)
    for r in range(N_COPIES):
        s = soft_of(dp, r)
        for f in range(s.shape[0]):
            dig[r, f] = digest(s[f])
        if r < N_SRC:
            soft[r, :s.shape[0]] = s
    out["digest"] = dig
    del dp, dev
    # every source decoded alone: its digests, its result and its own rounds; its soft bits where a frame differs from the batch
    single = [[] for _ in range(6)]
    diff_at, diff_soft = [], []
    import torch
    for i in range(N_SRC):
        t = torch.from_numpy(srcs[i]).cuda()
        dp1 = api.DabProcessor(1, input_format=api.FMT_U8, scan_mode=True, ctx=ctx)
        rounds1 = traced(os.path.join(out_dir, "trace1.txt"), lambda: dp1.run_ptrs([t.data_ptr()], [t.shape[0]], api.MEM_DEVICE))
        s = soft_of(dp1, 0)
        d = np.zeros((F_MAX, 32), np.uint8)
        for f in range(s.shape[0]):
            d[f] = digest(s[f])
            if not np.array_equal(d[f], dig[i, f]):
                diff_at.append((i, f))
                diff_soft.append(s[f] - soft[i, f])
        ra = result_arrays(dp1, 0)
        starts = np.zeros(F_MAX, np.uint8)  # frames that begin a window of this decode
        starts[np.cumsum(np.concatenate([[0], rounds1[:, 1]]))[:-1].clip(max=F_MAX - 1)] = 1
        for lst, v in zip(single, (d, ra["n_frames"], ra["pos"], ra["fbb"], ra["fic_valid"], starts)):
            lst.append(v)
    for name, lst in zip(("digest", "n_frames", "pos", "fbb", "fic_valid", "window_start"), single):
        out["single_" + name] = np.stack(lst)
    # (source, frame) where the lone decode differs from the batch, and the difference (lone - batch)
    out["single_diff_at"] = np.array(diff_at, np.int64).reshape(-1, 2)
    out["single_diff"] = np.array(diff_soft, np.int16).reshape(-1, 75, 3072)
    np.save(os.path.join(out_dir, "soft.npy"), soft)
    np.savez(os.path.join(out_dir, "out.npz"), **out)


def mode_segments(ctx, inp, out_dir):
    from dabstar_b200 import api
    seg_frames, warmup, max_window = int(inp["segment_frames"]), int(inp["warmup"]), int(inp["max_window"])
    iq = segment_recording()
    dp = api.DabProcessor(1, input_format=api.FMT_U8, scan_mode=True, max_window=max_window, ctx=ctx)
    dp.set_segmentation(seg_frames, warmup)
    rounds = traced(os.path.join(out_dir, "trace.txt"), lambda: dp.run([iq]))
    out = result_arrays_long(dp)
    out["rounds"] = rounds
    out["warmup_frames"] = dp.warmup_frames(0)
    np.save(os.path.join(out_dir, "soft.npy"), soft_of(dp, 0))
    np.savez(os.path.join(out_dir, "out.npz"), **out)


def result_arrays_long(dp) -> dict:
    res = dp.result(0)
    return dict(n_frames=res.n_frames, pos=np.array([(i.sym0_pos, i.start_index) for i in res.info], np.int64).reshape(-1, 2),
                fic_valid=res.fic_valid, counters=res.counters)


def main():
    mode, in_dir, out_dir = sys.argv[1:4]
    from dabstar_b200 import api
    ctx = api.Context(0)
    path = os.path.join(in_dir, "in.npz")
    inp = dict(np.load(path)) if os.path.exists(path) else {}
    {"tap": mode_tap, "batch": mode_batch, "segments": mode_segments}[mode](ctx, inp, out_dir)


if __name__ == "__main__":
    main()
