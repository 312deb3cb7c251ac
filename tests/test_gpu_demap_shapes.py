"""The DQPSK demapper (k_demap5 in ofdm_kernels.cu) in every compiled form and in the launch shapes the engine uses.

launch_demap picks the output lag from the grid: 15 up to 2 CTAs per SM, 7 up to 3, 3 above (DESIGN.md section 2). Each lag is its
own template instance with its own stash depth, output-row ring and drain loop, and each soft_bit_type another. Here:

* the oracle replay model (CPU): soft bits rebuilt from the oracle chain's own FFT rows and clock errors with the oracle's
  OfdmDecoder, over any list of segments (first frame, last frame, warm-up, reset or continue). Unsegmented it reproduces the
  chain bit for bit; it is the checker of the segmented decode below;
* the stage tap (OfdmDecoder.decode_frames) at lag 3 / 7 / 15 x soft_bit_type 0 / 1 / 2: a TII null symbol, a one-frame
  call, a continuation over two calls. The three lags must agree bit for bit: the scale of a symbol (sum |r| of the previous
  one) is built both by the shuffle chain and by dm5_total's polling path, which one runs depends on timing, and the two
  agree exactly (DESIGN.md section 5); an error of one ulp there moves soft bits by less than one LSB;
* a batch of 256 recordings (768 CTAs, more than are resident at any lag) at each lag, every recording cut inside its last
  frame, against the oracle chain; all copies of a source and the source decoded alone bit identical;
* the segmented decode of a 400-frame recording against the replay of the engine's own segment layout, frame by frame.

The lag is read from DABSTAR_DEMAP_LAG once per process, so each configuration runs in a fresh process (demap_worker.py).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from collections import Counter

import numpy as np
import pytest

import demap_worker as W
from dabstar_b200 import synth

LAGS = (3, 7, 15)
N_SM, CTAS_PER_RUN = 148, 3
RESIDENT = {15: 2 * N_SM, 7: 3 * N_SM, 3: 4 * N_SM}  # demap5_smem_bytes: (LAG + 1 + 8) x 4 KB per CTA
TAP_TII = np.array([0, 0, 1, 0, 0, 0], np.uint8)     # frame 2's null symbol carries TII: it leaves the null power alone
QUALITY = ("mer_db", "snr_db", "mean_value", "mean_power_overall", "noise_power", "sigma_freq_corr")  # OfdmDecoder.QUALITY


# ------------------------------------------------------------------------------------------------ oracle replay model
def replay(oracle, fft, clock_err, segments, soft_bit_type):
    """Soft bits of the kept frames of `segments`, decoded by the oracle's OfdmDecoder from the given spectra.

    fft(f): complex64[77, 2048] of frame f (symbol 0, symbols 1..75, null symbol), clock_err[f] its clock error;
    segments: [(first, last, warmup, parent)]: frames first..last are decoded, the soft bits of first + warmup..last are kept;
    parent -1 starts from a fresh (reset) decoder, parent j >= 0 continues from the state after segment j (which ends at
    frame first - 1 and comes earlier in the list).
    The chain passes its CP phase as phase_corr; that only feeds the frequency-correction statistics, not the soft bits (the
    self-check pins it), so 0 is passed. Returns {frame: int16[75, 3072]}."""

    def run(h, seg, out):
        first, last, warmup, _ = seg
        for f in range(first, last + 1):
            x = fft(f)
            soft = np.zeros((75, 3072), np.int16)
            oracle.ofdm_store_reference(h, x[0])
            for s in range(1, 76):
                soft[s - 1] = oracle.ofdm_decode_symbol(h, x[s], s, 0.0, float(clock_err[f]))
            oracle.ofdm_store_null(h, x[76])
            if out is not None and f >= first + warmup:
                out[f] = soft

    def state_after(j):
        """A new decoder in the state after segment j (replayed again from its own start)."""
        p = segments[j][3]
        h = oracle.ofdm_new(soft_bit_type) if p < 0 else state_after(p)
        run(h, segments[j], None)
        return h

    children = Counter(s[3] for s in segments if s[3] >= 0)
    kept, out = {}, {}
    for i, seg in enumerate(segments):
        p = seg[3]
        assert p < i and (p < 0 or segments[p][1] == seg[0] - 1), (i, seg)
        if p < 0:
            h = oracle.ofdm_new(soft_bit_type)
        else:
            children[p] -= 1
            h = kept.pop(p) if children[p] == 0 else state_after(p)
        run(h, seg, out)
        if children[i] > 0:
            kept[i] = h
        else:
            oracle.ofdm_free(h)
    for h in kept.values():
        oracle.ofdm_free(h)
    return out


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


def _chain_with_taps(oracle, iq, soft_bit_type=0):
    return oracle.chain_run(oracle.to_cf32(iq), scan_mode=1, soft_bit_type=soft_bit_type, tap_fft=True, tap_soft=True)


@pytest.mark.parametrize("soft_bit_type,cut", [(0, False), (1, False), (2, False), (0, True)])
def test_replay_reproduces_the_chain(oracle, soft_bit_type, cut):
    """Replaying the chain's own FFT rows and clock errors through one unsegmented run gives the chain's soft bits bit for bit
    (cut: the recording ends 10 data symbols into its last frame; the chain drops that frame, the complete ones stay exact)."""
    rec = synth.generate(7, seed=30 + soft_bit_type, snr_db=18.0, cfo_hz=1500.0, fmt=synth.FMT_U8)
    iq = rec.iq[:W.LEAD + 6 * synth.T_FRAME + 2656 + 2552 + 10 * 2552 + 1000] if cut else rec.iq
    r = _chain_with_taps(oracle, iq, soft_bit_type)
    assert r.n_frames == (6 if cut else 7)
    ce = [i.clock_err for i in r.info]
    got = replay(oracle, r.fft, ce, [(0, r.n_frames - 1, 0, -1)], soft_bit_type)
    assert sorted(got) == list(range(r.n_frames))
    for f in range(r.n_frames):
        assert np.array_equal(got[f], r.soft_bits(f)), f
    r.close()


def test_replay_continuation_and_warmup(oracle):
    """A continuation is exact: segments that continue the state after an earlier one (also two continuing the same state,
    one of them with a warm-up frame) reproduce the chain; a segment from reset() with a warm-up differs, and keeps only the
    frames after its warm-up."""
    rec = synth.generate(7, seed=33, snr_db=18.0, fmt=synth.FMT_U8)
    r = _chain_with_taps(oracle, rec.iq)
    ce = [i.clock_err for i in r.info]
    got = replay(oracle, r.fft, ce, [(0, 2, 0, -1), (3, 4, 0, 0), (3, 6, 1, 0), (5, 6, 0, 1)], 0)
    assert sorted(got) == list(range(7))
    for f in range(7):
        assert np.array_equal(got[f], r.soft_bits(f)), f
    warm = replay(oracle, r.fft, ce, [(2, 6, 2, -1)], 0)
    assert sorted(warm) == [4, 5, 6] and not np.array_equal(warm[4], r.soft_bits(4))
    r.close()


def test_engine_segment_layout():
    segs, w = engine_segments([1, 399], 48, 4)
    assert segs[0] == (0, 0, 0, -1) and segs[1] == (1, 49, 0, 0) and len(segs) == 1 + 8
    assert segs[2] == (1 + 49 - 4, 1 + 99 - 1, 4, -1) and w == 7 * 4
    segs, w = engine_segments([1, 399], 2, 4)
    assert len(segs) == 1 + 199 and segs[2] == (1, 4, 2, 0) and segs[3] == (1, 6, 4, 0) and segs[4] == (3, 8, 4, -1)
    assert w == 2 + 4 * 197
    assert engine_segments([5, 7], 4, 2) == ([(0, 4, 0, -1), (5, 11, 0, 0)], 0)  # windows < 2 segments: one run each


# ------------------------------------------------------------------------------------------------ worker processes
def run_worker(mode, lag, out_dir, inputs=None, timeout=900):
    """demap_worker.py MODE in a fresh process with DABSTAR_DEMAP_LAG = lag (None: the launcher's choice) and DABSTAR_TRACE."""
    os.makedirs(out_dir, exist_ok=True)
    if inputs is not None:
        np.savez(os.path.join(out_dir, "in.npz"), **inputs)
    env = dict(os.environ, DABSTAR_TRACE="1")
    env.pop("DABSTAR_DEMAP_LAG", None)
    if lag is not None:
        env["DABSTAR_DEMAP_LAG"] = str(lag)
    flags = (["-s"] if sys.flags.no_user_site else []) + (["-E"] if sys.flags.ignore_environment else [])
    r = subprocess.run([sys.executable] + flags + [W.__file__, mode, str(out_dir), str(out_dir)], env=env, capture_output=True,
                       text=True, timeout=timeout)
    assert r.returncode == 0, f"worker {mode} lag {lag} exited {r.returncode}:\n{r.stderr[-4000:]}"
    return dict(np.load(os.path.join(out_dir, "out.npz")))


def _check_soft(got, want, where):
    """Soft bits of one frame against the oracle: <= 1e-4 of them more than one LSB apart (the parity bar), and <= 1 % apart at
    all. The float arithmetic differs from the oracle's only in its last bits, so a value truncates to another integer rarely;
    a conversion that rounds the wrong way moves half of all values by one and fails the second bar, not the first."""
    d = np.abs(np.asarray(got).astype(np.int32) - np.asarray(want).astype(np.int32))
    beyond, differ = float((d > 1).mean()), float((d > 0).mean())
    assert beyond <= 1e-4 and differ <= 1e-2, (where, f"beyond 1 LSB {beyond:.2e}, differing {differ:.2e}, max {d.max()}")


@pytest.fixture(scope="module")
def work_dir(tmp_path_factory):
    d = tmp_path_factory.mktemp("demap_shapes")
    yield d
    shutil.rmtree(d, ignore_errors=True)  # the soft-bit dumps are some hundred MB


# ------------------------------------------------------------------------------------------------ B: the tap at every lag
@pytest.fixture(scope="module")
def tap_inputs(oracle):
    """FFT rows of 6 frames at 18 dB with clock error, as the oracle chain produced them (the rows of test_gpu_stages)."""
    rec = synth.generate(7, seed=30, snr_db=18.0, fmt=synth.FMT_CF32)
    r = oracle.chain_run(rec.iq, scan_mode=1, tap_fft=True)
    assert r.n_frames >= 6
    fft = np.stack([r.fft(f) for f in range(6)])
    ce = np.array([r.info[f].clock_err for f in range(6)], np.float32)
    r.close()
    assert np.abs(ce).max() > 1.0
    return fft, ce


@pytest.fixture(scope="module")
def tap_runs(tap_inputs, work_dir):
    cache = {}

    def get(lag):
        if lag not in cache:
            fft, ce = tap_inputs
            cache[lag] = run_worker("tap", lag, work_dir / f"tap{lag}", dict(fft=fft, clock_err=ce, tii=TAP_TII), timeout=600)
        return cache[lag]
    return get


def _oracle_tap(oracle, fft, ce, st, frames, calls_tii):
    """The oracle decoder over `frames` in order (one object), TII flags per frame: soft bits, state vectors, quality."""
    h = oracle.ofdm_new(st)
    soft = np.zeros((len(frames), 75, 3072), np.int16)
    for i, f in enumerate(frames):
        oracle.ofdm_store_reference(h, fft[f, 0])
        for s in range(1, 76):
            soft[i, s - 1] = oracle.ofdm_decode_symbol(h, fft[f, s], s, 0.0, float(ce[f]))
        if not calls_tii[i]:
            oracle.ofdm_store_null(h, fft[f, 76])
    states = [oracle.ofdm_state(h, w) for w in range(6)]
    q = oracle.ofdm_quality(h)
    oracle.ofdm_free(h)
    return soft, states, q


def _null_pow_order(oracle):
    """Index of each carrier's FFT bin: the device keeps the null power per carrier, the oracle per bin."""
    bins = oracle.freq_interleaver().astype(np.int64)
    return np.where(bins < 0, bins + 2048, bins)


def _check_tap_state(got_flat, want, order):
    got = np.split(got_flat, np.cumsum([1536] * 5))
    for which, tol in ((0, 1e-4), (1, 1e-3), (2, 1e-3), (3, 1e-3)):
        assert np.allclose(got[which], want[which], rtol=tol, atol=1e-6), which
    assert np.allclose(got[4], want[4][order], rtol=1e-4, atol=1e-12)
    assert np.isclose(got[5][0], want[5][0], rtol=1e-4) and np.isclose(got[5][1], want[5][1], rtol=1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("lag", LAGS)
@pytest.mark.parametrize("soft_bit_type", [0, 1, 2])
def test_tap_every_lag_against_oracle(oracle, tap_inputs, tap_runs, lag, soft_bit_type):
    """OfdmDecoder.decode_frames at each lag: six frames with a TII null symbol in frame 2, one frame alone, and the six frames
    as two calls on one state, against the oracle decoder: <= 1e-4 of the soft bits beyond one LSB, state vectors and quality
    figures as in test_gpu_stages.test_ofdm_decoder_soft_bits."""
    fft, ce = tap_inputs
    out = tap_runs(lag)
    st = soft_bit_type
    order = _null_pow_order(oracle)
    for case, frames in (("full", range(6)), ("one", range(1)), ("cont", range(6))):
        tii = np.zeros(6, np.uint8) if case == "one" else TAP_TII
        want, states, q = _oracle_tap(oracle, fft, ce, st, list(frames), tii[list(frames)])
        got = out[f"{case}_soft_{st}"]
        assert got.shape == want.shape
        for f in range(got.shape[0]):
            _check_soft(got[f], want[f], (case, f))
        _check_tap_state(out[f"{case}_state_{st}"], states, order)
        if case == "full":
            gq = dict(zip(QUALITY, (float(v) for v in out[f"full_quality_{st}"])))
            assert abs(gq["mer_db"] - q["mer_db"]) < 0.01 and abs(gq["snr_db"] - q["snr_db"]) < 0.01, (gq, q)
            assert np.isclose(gq["noise_power"], q["noise_power"], rtol=1e-4) and np.isclose(gq["mean_power_overall"], q["mean_power_overall"], rtol=1e-4)
    # the TII flag reached the kernel: the null power is not what storing every null symbol gives
    _, states_all, _ = _oracle_tap(oracle, fft, ce, st, list(range(6)), np.zeros(6, np.uint8))
    assert not np.allclose(out[f"full_state_{st}"][4 * 1536:5 * 1536], states_all[4][order], rtol=1e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("soft_bit_type", [0, 1, 2])
def test_tap_lags_bit_identical(tap_runs, soft_bit_type):
    """Lag 3, 7 and 15 give the same soft bits and states bit for bit: every symbol's scale is the same float whichever
    path (shuffle chain, ring poll, drain) produced it."""
    outs = [tap_runs(lag) for lag in LAGS]
    for case in ("full", "one", "cont"):
        for kind in ("soft", "state"):
            key = f"{case}_{kind}_{soft_bit_type}"
            for lag, o in zip(LAGS[1:], outs[1:]):
                a, b = outs[0][key], o[key]
                assert np.array_equal(a, b), f"{key}: lag {LAGS[0]} vs {lag}: {int((a != b).sum())} values differ"


# ------------------------------------------------------------------------------------------------ C: a batch past one wave
@pytest.fixture(scope="module")
def batch_want(oracle):
    """The oracle chain of each of the 32 sources (soft_bit_type 0)."""
    want = []
    for i in range(W.N_SRC):
        iq, k = W.batch_source(i)
        want.append((oracle.chain_run(oracle.to_cf32(iq), scan_mode=1, tap_soft=True), k))
    yield want
    for r, _ in want:
        r.close()


@pytest.fixture(scope="module")
def batch_runs(work_dir):
    cache = {}

    def get(lag):
        if lag not in cache:
            d = work_dir / f"batch{lag}"
            out = run_worker("batch", lag, d, timeout=1200)
            out["soft"] = np.load(d / "soft.npy", mmap_mode="r")
            cache[lag] = out
        return cache[lag]
    return get


def _check_copy_against_chain(got, r, want, k, soft=None):
    """Recording r of a batch result (worker arrays) against the chain of its source. The chain drops the cut frame and the
    decoder's result holds complete frames only, so the cut frame is seen through the good-FIB count (its FIC blocks count in
    both) and through the last complete frame, whose trailing rows the drain writes when the cut frame holds fewer than LAG
    symbols."""
    n = int(got["n_frames"][r])
    assert n == want.n_frames == W.N_FULL, (r, n, want.n_frames)
    assert [tuple(p) for p in got["pos"][r, :n]] == [(i.sym0_pos, i.start_index) for i in want.info], r
    assert [(round(float(a)), round(float(b))) for a, b in got["fbb"][r, :n]] == [(round(i.fbb_data), round(i.fbb_null)) for i in want.info], r
    assert np.array_equal(got["fic_valid"][r, :n], want.fic_valid), r
    ok = want.fic_valid.astype(bool).repeat(768, axis=1)
    assert np.array_equal(got["fib"][r, :n][ok], want.fib_bits[ok]), r
    assert got["counters"][r, 0] == want.n_good_fibs, (r, k, got["counters"][r, 0], want.n_good_fibs)
    if soft is not None:
        for f in range(n):
            _check_soft(soft[f], want.soft_bits(f), (r, k, f))


@pytest.mark.gpu
@pytest.mark.parametrize("lag", LAGS)
def test_batch_past_one_wave(batch_runs, batch_want, lag):
    """256 recordings (32 sources, copy i from source i % 32) at a forced lag: 768 CTAs, more than are resident at any lag,
    so later CTAs take their work from the ticket counter as earlier ones finish. Every copy equals the oracle chain of its
    source (positions, AFC, CRC flags, FIB bits, good FIBs, soft bits of every frame within one LSB); the copies of a source
    are bit identical to each other and to the source decoded alone."""
    out = batch_runs(lag)
    rounds = out["rounds"]
    heavy = rounds[rounds[:, 0] == W.N_COPIES]
    assert heavy.shape[0] >= 1, rounds   # a heavy round ran every recording in one demapper launch
    assert W.N_COPIES * CTAS_PER_RUN > RESIDENT[lag]
    for r in range(W.N_COPIES):
        s = r % W.N_SRC
        want, k = batch_want[s]
        _check_copy_against_chain(out, r, want, k, out["soft"][s] if r < W.N_SRC else None)
        assert np.array_equal(out["digest"][r], out["digest"][s]), (r, s)
        for key in ("n_frames", "pos", "fbb", "fic_valid", "fib", "counters"):
            assert np.array_equal(out[key][r], out[key][s]), (r, key)
    # the same source decoded alone. Were its windows cut differently from the batch's, the first symbol of a window could
    # move by one (the scale of a window's first symbol is mMeanValue, stored as total / 1536): allowed there and nowhere else
    for (s, f), d in zip(out["single_diff_at"], out["single_diff"]):
        assert out["single_window_start"][s, f] and np.abs(d[1:]).max() == 0 and np.abs(d[0]).max() <= 1, (s, f)
    differing = {(int(s), int(f)) for s, f in out["single_diff_at"]}
    for s in range(W.N_SRC):
        for f in range(int(out["n_frames"][s])):
            if (s, f) not in differing:
                assert np.array_equal(out["single_digest"][s, f], out["digest"][s, f]), (s, f)
        assert out["single_n_frames"][s] == out["n_frames"][s]
        for key in ("pos", "fbb", "fic_valid"):
            assert np.array_equal(out["single_" + key][s], out[key][s]), (s, key)


@pytest.mark.gpu
def test_batch_lags_bit_identical(batch_runs):
    """The batch at lag 3, 7 and 15: the same results and soft bits, bit for bit."""
    outs = [batch_runs(lag) for lag in LAGS]
    for lag, o in zip(LAGS[1:], outs[1:]):
        for key in ("n_frames", "pos", "fbb", "clock_err", "fic_valid", "fib", "counters", "digest"):
            assert np.array_equal(outs[0][key], o[key]), (key, LAGS[0], lag)


@pytest.mark.gpu
@pytest.mark.parametrize("soft_bit_type", [1, 2])
def test_batch_soft_bit_types(ctx, oracle, soft_bit_type):
    """soft_bit_type 1 and 2 through DabProcessor: the 256-recording batch with the launcher's own lag choice (3 for 768
    CTAs) against chain_run with the same soft-bit type."""
    srcs = [W.batch_source(i) for i in range(W.N_SRC)]
    dp, _, dev = W.decode_batch(ctx, [s for s, _ in srcs], soft_bit_type)
    got = W.batch_results(dp)
    for s, (iq, k) in enumerate(srcs):
        want = oracle.chain_run(oracle.to_cf32(iq), scan_mode=1, soft_bit_type=soft_bit_type, tap_soft=True)
        soft = W.soft_of(dp, s)
        for r in range(s, W.N_COPIES, W.N_SRC):
            _check_copy_against_chain(got, r, want, k, soft if r == s else None)
            if r != s:
                assert np.array_equal(W.soft_of(dp, r), soft), r
        want.close()
    del dp, dev


# ------------------------------------------------------------------------------------------------ D: segmented decode
N_LONG = 400


@pytest.fixture(scope="module")
def long_chain(oracle):
    r = _chain_with_taps(oracle, W.segment_recording())
    assert r.n_frames == N_LONG
    yield r
    r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("seg_frames,warmup,lag,max_window", [(48, 4, 15, 200), (48, 18, 15, 200), (2, 4, 3, 512)])
def test_segmented_decode_matches_exact_model(oracle, long_chain, work_dir, seg_frames, warmup, lag, max_window):
    """set_segmentation over a clean 400-frame recording, frame by frame against the oracle replay of the engine's own layout:
    the windows from the round trace, each cut into segments that warm up from reset() or continue the recording's state.
    Every frame within one LSB on <= 1e-4 of its soft bits, and warmup_frames() the sum of the warm-ups. (2, 4) is ~200
    segments in one launch: ~600 CTAs at lag 3, past one wave. With windows of at most 200 frames the last window starts from
    a state adapted over 200 frames, far from reset(): a segment that continued from it instead of warming up from reset()
    would not match."""
    d = work_dir / f"seg{seg_frames}_{warmup}"
    out = run_worker("segments", lag, d, dict(segment_frames=seg_frames, warmup=warmup, max_window=max_window), timeout=900)
    soft = np.load(d / "soft.npy", mmap_mode="r")
    rounds = out["rounds"]
    assert (rounds[:, 0] == 1).all() and rounds[:, 1].sum() == int(out["n_frames"]) == N_LONG, rounds  # no replayed window
    windows = [int(n) for n in rounds[:, 1]]
    segs, total_w = engine_segments(windows, seg_frames, warmup)
    assert int(out["warmup_frames"]) == total_w
    n_runs = max(n // seg_frames if n >= 2 * seg_frames else 1 for n in windows)
    if seg_frames == 2:
        assert n_runs * CTAS_PER_RUN > RESIDENT[lag], windows
    else:
        assert len(windows) >= 2 and windows[0] >= 100 and windows[-1] >= 4 * seg_frames and len(segs) >= 8, windows
    r = long_chain
    assert [tuple(p) for p in out["pos"]] == [(i.sym0_pos, i.start_index) for i in r.info]
    assert np.array_equal(out["fic_valid"], r.fic_valid)
    want = replay(oracle, r.fft, [i.clock_err for i in r.info], segs, 0)
    assert sorted(want) == list(range(N_LONG))
    for f in range(N_LONG):
        _check_soft(soft[f], want[f], f)
