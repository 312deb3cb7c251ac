"""What the demapper-shape and frame-quality GPU tests share (not collected as tests): the batch past one wave of demapper CTAs
and the long recording of the segmented decode, fixed-shape views of a run's results, the engine's round trace, a forced
demapper lag, and the engine's segment layout with the oracle replay that walks it.

DABSTAR_DEMAP_LAG is read on every demapper launch and DABSTAR_TRACE once per run, so both are set around the runs that need
them (forced_lag, traced) and the tests run in the test process."""
from __future__ import annotations

import contextlib
import hashlib
import os
import re
import sys
import tempfile
from collections import Counter

import numpy as np

from dabstar_b200 import synth

# ---- the batch: 256 recordings past one wave of demapper CTAs (768 CTAs; 2 / 3 / 4 per SM at lag 15 / 7 / 3 on 148 SMs)
N_SRC, N_COPIES, N_FULL = 32, 256, 6
K_CUT = (1, 2, 3, 4, 7, 8, 15, 16, 40, 74)  # data symbols the recording's last frame still holds
LEAD = 60000                                # synth.generate's default lead_samples
F_MAX = N_FULL + 2                          # padding of the per-frame arrays
N_LONG = 400                                # frames of segment_recording()


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
    """The clean long recording of the segmented-decode checks: N_LONG frames, 15 dB, no carrier offset."""
    return synth.generate(N_LONG, seed=31, snr_db=15.0, fmt=synth.FMT_U8).iq


# ---- the environment switches
@contextlib.contextmanager
def _env(name: str, value: str | None):
    old = os.environ.get(name)
    if value is None:
        os.environ.pop(name, None)
    else:
        os.environ[name] = value
    try:
        yield
    finally:
        if old is None:
            os.environ.pop(name, None)
        else:
            os.environ[name] = old


def forced_lag(lag: int | None):
    """DABSTAR_DEMAP_LAG = lag for the body (None: unset, the launcher's choice), the previous value afterwards."""
    return _env("DABSTAR_DEMAP_LAG", None if lag is None else str(lag))


ROUND_RE = re.compile(r"\[dabstar\] round (\d+) t=[0-9.]+ ms: (\d+) recordings, (\d+) frames")


def parse_rounds(text: str) -> np.ndarray:
    """(recordings, frames) of every round line DABSTAR_TRACE printed."""
    return np.array([(int(m.group(2)), int(m.group(3))) for m in ROUND_RE.finditer(text)], np.int64).reshape(-1, 2)


@contextlib.contextmanager
def stderr_to(f):
    """File descriptor 2 (where the library prints its trace) into the open file `f` for the duration."""
    sys.stderr.flush()
    saved = os.dup(2)
    os.dup2(f.fileno(), 2)
    try:
        yield
    finally:
        sys.stderr.flush()
        os.dup2(saved, 2)
        os.close(saved)


def traced(fn) -> np.ndarray:
    """fn() with DABSTAR_TRACE set: the round table of its runs (the trace itself goes on to stderr)."""
    with tempfile.TemporaryFile("w+") as f:
        with _env("DABSTAR_TRACE", "1"), stderr_to(f):
            fn()
        f.seek(0)
        text = f.read()
    sys.stderr.write(text)
    return parse_rounds(text)


# ---- results
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


def soft_of(dp, r: int) -> np.ndarray:
    n = dp.n_frames(r)
    return np.stack([dp.soft_bits(r, f) for f in range(n)]) if n else np.zeros((0, 75, 3072), np.int16)


def decode_batch(ctx, srcs: list[np.ndarray], soft_bit_type: int, trace: bool = False, frame_quality: bool = False):
    """The 256 copies (copy i from source i % N_SRC, physical copies on the device) in one DabProcessor, scan mode, with the
    round trace and per-frame quality if asked. Returns (processor, round table or None, device buffers)."""
    import torch
    from dabstar_b200 import api
    dev = [torch.from_numpy(srcs[i % N_SRC]).cuda() for i in range(N_COPIES)]
    torch.cuda.synchronize()
    dp = api.DabProcessor(N_COPIES, input_format=api.FMT_U8, soft_bit_type=soft_bit_type, scan_mode=True, ctx=ctx)
    if frame_quality:
        dp.set_frame_quality(True)

    def run():
        dp.run_ptrs([t.data_ptr() for t in dev], [t.shape[0] for t in dev], api.MEM_DEVICE)
    rounds = None
    if trace:
        rounds = traced(run)
    else:
        run()
    return dp, rounds, dev


# ---- the engine's segment layout and the oracle replay of it
def engine_segments(windows, seg_frames, seg_warmup):
    """The engine's demapper runs over a recording's windows (decoder.cu, heavy pass: 'demapper runs'), as replay segments.

    A window of n >= 2 seg_frames frames is cut into n_seg = n // seg_frames segments; segment sg covers [b, e) with
    b = n sg / n_seg and starts w = min(warm-up, b) frames early (w = 0 for sg = 0). A segment that reaches back to the window's
    first frame continues from the recording's state (reset() in the first window after the time sync), the others start
    from reset() and discard their w warm-up frames; the window's last segment hands its state to the next window.
    Returns (segments, sum of w)."""
    segs, f0, total_w, prev = [], 0, 0, -1
    for n in windows:
        n_seg = n // seg_frames if seg_frames > 0 and n >= 2 * seg_frames else 1
        for sg in range(n_seg):
            b, e = n * sg // n_seg, n * (sg + 1) // n_seg
            w = 0 if sg == 0 else min(seg_warmup, b)
            total_w += w
            segs.append((f0 + b - w, f0 + e - 1, w, prev if b - w == 0 else -1))
        prev = len(segs) - 1
        f0 += n
    return segs, total_w


def replay_segments(oracle, fft, clock_err, segments, soft_bit_type, kept):
    """The oracle's OfdmDecoder over `segments`, from the given spectra; kept(f, h, soft) after every kept frame.

    fft(f): complex64[77, 2048] of frame f (symbol 0, symbols 1..75, null symbol), clock_err[f] its clock error;
    segments: [(first, last, warmup, parent)]: frames first..last are decoded, first + warmup..last are kept; parent -1 starts
    from a fresh (reset) decoder, parent j >= 0 continues from the state after segment j (which ends at frame first - 1 and
    comes earlier in the list). kept gets the frame, the decoder handle after the frame's null symbol and the frame's soft bits
    (int16[75, 3072]). The chain passes its CP phase as phase_corr; that only feeds the frequency-correction statistics, not
    the soft bits, so 0 is passed."""

    def run(h, seg, keep):
        first, last, warmup, _ = seg
        for f in range(first, last + 1):
            x = fft(f)
            soft = np.zeros((75, 3072), np.int16)
            oracle.ofdm_store_reference(h, x[0])
            for s in range(1, 76):
                soft[s - 1] = oracle.ofdm_decode_symbol(h, x[s], s, 0.0, float(clock_err[f]))
            oracle.ofdm_store_null(h, x[76])
            if keep and f >= first + warmup:
                kept(f, h, soft)

    def state_after(j):
        """A new decoder in the state after segment j (replayed again from its own start)."""
        p = segments[j][3]
        h = oracle.ofdm_new(soft_bit_type) if p < 0 else state_after(p)
        run(h, segments[j], False)
        return h

    children = Counter(s[3] for s in segments if s[3] >= 0)
    handles = {}
    for i, seg in enumerate(segments):
        p = seg[3]
        assert p < i and (p < 0 or segments[p][1] == seg[0] - 1), (i, seg)
        if p < 0:
            h = oracle.ofdm_new(soft_bit_type)
        else:
            children[p] -= 1
            h = handles.pop(p) if children[p] == 0 else state_after(p)
        run(h, seg, True)
        if children[i] > 0:
            handles[i] = h
        else:
            oracle.ofdm_free(h)
    for h in handles.values():
        oracle.ofdm_free(h)
