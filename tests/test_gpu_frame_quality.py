"""Per-frame signal quality: dabstar_decoder_set_frame_quality / dabstar_decoder_frame_quality and the stage tap
dabstar_ofdm_decode_frames_quality (OfdmDecoder.decode_frames(..., quality=True)).

Record f of a recording is what dabstar_decoder_quality would return had the recording ended after frame f: { MER dB, SNR dB,
mMeanValue, mMeanPowerOvrAll, noise power, sqrt(mMeanSigmaSqFreqCorr) } of the OFDM state after frame f's null symbol.
The capture instance of the demapper (k_demap5<.., QUAL = true>) snapshots that state and k_frame_quality sums it in the order
and precision of the host's quality_from_state, so:

* the last record equals dabstar_decoder_quality bit for bit when no cut trailing frame was demapped after it, and the tap's
  last row equals dabstar_ofdm_state_quality after the call;
* against the oracle's per-frame figures (chain_records: the chain's OfdmDecoder replayed on its own FFT rows, pinned to the
  chain's end-of-run figures at every frame by the CPU tests) the bars are
  those of the end-of-run figures: MER / SNR within 0.01 dB, mMeanValue, mMeanPowerOvrAll and noise within 1e-4 relative,
  field 5 within 1e-4 (absolute, or relative for figures above 1 Hz). mMeanPowerOvrAll is the reference's serial IIR in the
  oracle and its per-carrier form on the GPU (DESIGN.md section 8, row D4): equal up to float rounding, not bit for bit;
* field 5 is replayed on the host from the frames' cyclic-prefix phases: bit for bit the float recurrence below.

The CPU tests pin the oracle's records themselves. Forced demapper lags and traced segment layouts use demap_support.
"""
from __future__ import annotations

import ctypes

import numpy as np
import pytest

import demap_support as S
from dabstar_b200 import api, synth
from demap_support import N_LONG, engine_segments

T_U, T_S, T_N = 2048, 2552, 2656
LEAD = 60000
SC_3A = synth.SubChannel(3, 100, 54, 0, 2, 72)
LAGS = (3, 7, 15)


# ------------------------------------------------------------------------------------------------ helpers
def tii_flags(oracle, res) -> list[bool]:
    """The chain's TII null symbols with track_cif: after each frame the CIF counter of the last FIG 0/0 in its CRC-good FIBs
    (scan_cif_count in dab_oracle.c, the counter kept across frames from 0, 0) marks the null symbol as TII when
    (count & 7) >= 4."""
    hi = lo = 0
    out = []
    for f in range(res.n_frames):
        for k in range(12):
            fib = res.fib_bits[f, (k // 3) * 768 + (k % 3) * 256:][:256]
            if not oracle.check_crc_bits(np.ascontiguousarray(fib)):
                continue
            done = 0
            while done < 30:
                d = fib[8 * done:]
                bits = lambda a, b: int("".join(str(int(x)) for x in d[a:b]), 2)
                typ, ln = bits(0, 3), bits(3, 8)
                if (typ == 7 and ln == 31) or done + ln + 1 > 30:
                    break
                if typ == 0 and bits(11, 16) == 0 and ln >= 5:
                    hi, lo = bits(35, 40), bits(40, 48)
                done += ln + 1
        out.append(((hi * 250 + lo) & 7) >= 4)
    return out


def chain_records(oracle, res, track_cif=False) -> np.ndarray:
    """The oracle's records: the chain's OfdmDecoder replayed through dabo_ofdm_* on the chain's own FFT rows (tap_fft), clock
    errors and CP phases, with dabo_ofdm_quality after every listed frame's null symbol. The chain resets the decoder at every
    time-sync search: a frame that does not begin where the previous one's null symbol ended plus its PRS offset follows one.
    The CP phase handed to symbol 1 is the previous frame's, across resets too (the chain keeps it; reset() keeps the sigma).
    The CPU tests below pin this replay to the chain's own end-of-run figures at every frame."""
    tii = tii_flags(oracle, res) if track_cif else [False] * res.n_frames
    h = oracle.ofdm_new(0)
    q = np.zeros((res.n_frames, 6), np.float32)
    for f in range(res.n_frames):
        a, x = res.info[f], res.fft(f)
        if f > 0:
            b = res.info[f - 1]
            if a.sym0_pos != b.sym0_pos + T_U + 75 * T_S + T_N + a.start_index:
                oracle.ofdm_reset(h)
        phase = res.info[f - 1].phase_cp if f > 0 else 0.0
        oracle.ofdm_store_reference(h, x[0])
        for s_ in range(1, 76):
            oracle.ofdm_decode_symbol(h, x[s_], s_, phase, float(a.clock_err))
        if not tii[f]:
            oracle.ofdm_store_null(h, x[76])
        q[f] = oracle_quality(oracle, h)
    oracle.ofdm_free(h)
    return q


def chain_quality(oracle, res) -> np.ndarray:
    q = np.zeros(6, np.float32)
    oracle.f("chain_quality")(res.h, q.ctypes.data_as(ctypes.c_void_p))
    return q


def oracle_quality(oracle, h) -> np.ndarray:
    q = np.zeros(6, np.float32)
    oracle.f("ofdm_quality")(h, q.ctypes.data_as(ctypes.c_void_p))
    return q


def sigma_replay(phase_cp) -> np.ndarray:
    """Field 5 of every record: dabstar_decoder_quality's float recurrence over the frames' cyclic-prefix phases."""
    two_pi, k, a = np.float32(6.28318530717958647692), np.float32(1000.0), np.float32(0.2)
    sigma, phase, out = np.float32(0.0), np.float32(0.0), []
    for p in phase_cp:
        fc = np.float32(np.float32(phase / two_pi) * k)
        sigma = np.float32(sigma + np.float32(a * np.float32(np.float32(fc * fc) - sigma)))
        phase = np.float32(p)
        out.append(np.sqrt(sigma))
    return np.array(out, np.float32)


def check_records(got, want, where):
    """The bars of the end-of-run figures, over all records at once (the message shows the worst of each field)."""
    assert got.shape == want.shape, (where, got.shape, want.shape)
    d_db = np.abs(got[:, :2].astype(np.float64) - want[:, :2])
    rel = np.abs(got[:, 2:5].astype(np.float64) / want[:, 2:5] - 1.0)
    d5 = np.abs(got[:, 5].astype(np.float64) - want[:, 5])
    bar5 = 1e-4 * np.maximum(1.0, np.abs(want[:, 5]))
    msg = f"{where}: MER/SNR max {d_db.max(axis=0)} dB, fields 2-4 max rel {rel.max(axis=0)}, field 5 max {d5.max()}"
    assert (d_db <= 0.01).all() and (rel <= 1e-4).all() and (d5 <= bar5).all(), msg


def chain(oracle, iq, tap_fft=True, **kw):
    return oracle.chain_run(oracle.to_cf32(iq), scan_mode=1, tap_fft=tap_fft, **kw)


def gpu(ctx, iqs, fmt=synth.FMT_U8, quality=True, subch=None, **kw):
    dp = api.DabProcessor(len(iqs), input_format=fmt, scan_mode=subch is None, ctx=ctx, **kw)
    for r in range(len(iqs)):
        if subch:
            dp.set_audio_channel(r, subch)
    dp.set_frame_quality(quality)
    dp.run(iqs)
    return dp


def ends_on_frame_boundary(iq, res, frame=-1):
    """The recording cut right after the null symbol of the chain's frame `frame`: too short for another phase reference."""
    end = res.info[frame].sym0_pos + T_U + 75 * T_S + T_N + 1000
    return np.ascontiguousarray(iq[:end])


def sync_loss_recording(fmt, seed=43):
    """Six frames, then a splice into another transmission: the time sync is lost and re-established, OfdmDecoder resets."""
    a = synth.generate(6, seed=seed, snr_db=18.0, cfo_hz=900.0, fmt=fmt)
    b = synth.generate(6, seed=seed + 1, snr_db=16.0, cfo_hz=-1700.0, fmt=fmt, lead_samples=20000)
    return np.ascontiguousarray(np.concatenate([a.iq[:LEAD + 4 * synth.T_FRAME + 100_000], b.iq]))


WORKLOADS = {
    "clean": lambda fmt: synth.generate(8, seed=41, snr_db=20.0, fmt=fmt).iq,
    "carrier_offset": lambda fmt: synth.generate(8, seed=42, snr_db=15.0, cfo_hz=-4300.0, fmt=fmt, lead_samples=77777).iq,
    "low_snr": lambda fmt: synth.generate(10, seed=11, snr_db=6.0, fmt=fmt).iq,
    "sync_loss": sync_loss_recording,
}
CASES = [("clean", synth.FMT_U8), ("carrier_offset", synth.FMT_U8), ("low_snr", synth.FMT_U8),
         ("sync_loss", synth.FMT_U8), ("sync_loss", synth.FMT_I16), ("sync_loss", synth.FMT_CF32)]


# ------------------------------------------------------------------------------------------------ the oracle's records (CPU)
@pytest.mark.parametrize("name", ["carrier_offset", "sync_loss", "tii_nulls"])
def test_oracle_records_are_chain_quality_at_every_frame(oracle, name):
    """Record f of the replay is dabo_chain_quality of the chain run over the recording cut right after frame f, bit for bit,
    at every frame: with a carrier offset, across a lost and re-established time sync (the decoder reset), and with track_cif
    (TII null symbols leave the noise power alone)."""
    track = name == "tii_nulls"
    if name == "carrier_offset":
        iq = synth.generate(7, seed=62, snr_db=14.0, cfo_hz=-2500.0, fmt=synth.FMT_U8).iq
    elif name == "sync_loss":
        iq = sync_loss_recording(synth.FMT_U8, seed=61)
    else:
        iq = synth.generate(8, seed=63, snr_db=16.0, subch=[SC_3A], fmt=synth.FMT_U8, fig_mode=1, tii=(5, 3)).iq
    r = chain(oracle, iq, track_cif=track)
    q = chain_records(oracle, r, track_cif=track)
    assert len({tuple(x) for x in q}) == r.n_frames  # one figure set per frame
    if name == "sync_loss":
        resets = [f for f in range(1, r.n_frames)
                  if r.info[f].sym0_pos != r.info[f - 1].sym0_pos + T_U + 75 * T_S + T_N + r.info[f].start_index]
        assert len(resets) == 1 and r.n_frames >= 9, resets
    if track:
        assert 3 <= sum(tii_flags(oracle, r)) <= (r.n_frames + 1) // 2
    for f in range(r.n_frames):
        c = chain(oracle, ends_on_frame_boundary(iq, r, f), tap_fft=False, track_cif=track)
        assert c.n_frames == f + 1
        assert np.array_equal(q[f].view(np.uint32), chain_quality(oracle, c).view(np.uint32)), (name, f)
        c.close()
    r.close()


def test_oracle_tii_null_keeps_noise(oracle):
    """With track_cif, a frame whose null symbol carries TII leaves the noise power where the previous frame left it (every
    second frame once FIG 0/0 is read: the CIF counter advances by 4 per frame); without it, every frame moves the noise."""
    rec = synth.generate(10, seed=63, snr_db=16.0, subch=[SC_3A], fmt=synth.FMT_U8, fig_mode=1, tii=(5, 3))
    r = chain(oracle, rec.iq, track_cif=True)
    q, p = chain_records(oracle, r, track_cif=True), chain_records(oracle, r)
    same = [f for f in range(1, r.n_frames) if q[f, 4] == q[f - 1, 4]]
    assert same == [f for f, t in enumerate(tii_flags(oracle, r)) if t and f > 0] and len(same) >= 3, same
    assert all(p[f, 4] != p[f - 1, 4] for f in range(1, r.n_frames))
    r.close()


def test_sigma_replay_matches_the_oracle_recurrence(oracle):
    """sigma_replay (the check of field 5) is the oracle's own recurrence on the chain's CP phases, bit for bit."""
    r = chain(oracle, synth.generate(6, seed=64, snr_db=14.0, cfo_hz=3300.0, fmt=synth.FMT_U8).iq)
    assert np.array_equal(sigma_replay([i.phase_cp for i in r.info]).view(np.uint32), chain_records(oracle, r)[:, 5].view(np.uint32))
    r.close()


# ------------------------------------------------------------------------------------------------ GPU: against the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("name,fmt", CASES)
def test_records_against_oracle_chain(ctx, oracle, name, fmt):
    """Every frame's record against the oracle chain's; field 5 bit for bit against the replay of the decoder's own CP phases.
    (The recordings end in a 4096-sample tail, so whether a cut frame follows the last record is not fixed here: the bit-exact
    tie to the end-of-run figures is test_last_record_is_end_of_run_quality's.)"""
    iq = WORKLOADS[name](fmt)
    r = chain(oracle, iq)
    dp = gpu(ctx, [iq], fmt)
    res = dp.result(0)
    assert [(i.sym0_pos, i.start_index) for i in res.info] == [(i.sym0_pos, i.start_index) for i in r.info]
    if name == "sync_loss":
        assert res.counters[1] >= 2  # the time sync was established again after the splice
    q = dp.frame_quality(0)
    assert q.shape == (res.n_frames, 6) and np.isfinite(q).all()
    check_records(q, chain_records(oracle, r), f"{name} fmt {fmt}")
    assert np.array_equal(q[:, 5].view(np.uint32), sigma_replay([i.phase_cp for i in res.info]).view(np.uint32))
    r.close()


@pytest.mark.gpu
def test_last_record_is_end_of_run_quality(ctx, oracle):
    """Ending on a frame boundary: the last record is dabstar_decoder_quality bit for bit. Ending 10 symbols into a frame: that
    frame is demapped but not listed, so it has no record and the end-of-run figures (which include its symbols) differ from
    the last record, while the records still match the oracle."""
    rec = synth.generate(9, seed=65, snr_db=17.0, cfo_hz=1200.0, fmt=synth.FMT_U8)
    full = chain(oracle, rec.iq)
    iq = ends_on_frame_boundary(rec.iq, full)
    dp = gpu(ctx, [iq])
    q = dp.frame_quality(0)
    assert q.shape[0] == full.n_frames
    assert np.array_equal(q[-1].view(np.uint32), np.array(list(dp.quality(0).values()), np.float32).view(np.uint32))
    cut = np.ascontiguousarray(rec.iq[:full.info[-1].sym0_pos + T_U + 10 * T_S + 1000])
    r = chain(oracle, cut)
    dpc = gpu(ctx, [cut])
    qc = dpc.frame_quality(0)
    assert qc.shape[0] == r.n_frames == full.n_frames - 1
    assert not np.array_equal(qc[-1], np.array(list(dpc.quality(0).values()), np.float32))
    check_records(qc, chain_records(oracle, r), "cut trailing frame")
    assert np.array_equal(qc.view(np.uint32), q[:-1].view(np.uint32))  # a frame's record does not depend on what follows it
    full.close()
    r.close()


@pytest.mark.gpu
def test_frame_quality_needs_capture(ctx):
    dp = api.DabProcessor(1, input_format=synth.FMT_U8, scan_mode=True, ctx=ctx)
    with pytest.raises(api.DabstarError):
        dp.frame_quality(0)  # no run yet
    dp.run([synth.generate(3, seed=66, fmt=synth.FMT_U8).iq])
    with pytest.raises(api.DabstarError):
        dp.frame_quality(0)  # the run did not capture


@pytest.mark.gpu
def test_capture_changes_nothing_else(ctx):
    """With capture on, soft bits, FIB bits, CRC flags, frame info, MSC bytes and counters are bit identical to capture off."""
    iq = sync_loss_recording(synth.FMT_U8, seed=71)
    runs = [gpu(ctx, [iq], quality=on, subch=[SC_3A]) for on in (False, True)]
    a, b = (dp.result(0) for dp in runs)
    assert a.n_frames == b.n_frames > 6
    assert np.array_equal(a.fib_bits, b.fib_bits) and np.array_equal(a.fic_valid, b.fic_valid)
    assert np.array_equal(a.counters, b.counters) and np.array_equal(a.msc[3], b.msc[3]) and a.msc[3].size > 0
    assert [bytes(i) for i in a.info] == [bytes(i) for i in b.info]
    for f in range(a.n_frames):
        assert np.array_equal(runs[0].soft_bits(0, f), runs[1].soft_bits(0, f)), f
    assert np.array_equal(np.array(list(runs[0].quality(0).values())), np.array(list(runs[1].quality(0).values())))


# ------------------------------------------------------------------------------------------------ GPU: stage tap
@pytest.mark.gpu
def test_tap_rows_against_oracle_and_state_quality(ctx, oracle):
    """decode_frames(quality=True): soft bits equal the plain call's; row f against the oracle OfdmDecoder's figures after
    frame f (one TII null symbol, a continuation over two calls); the last row equals quality() after the call bit for bit."""
    r = chain(oracle, synth.generate(7, seed=67, snr_db=15.0, cfo_hz=800.0, fmt=synth.FMT_U8).iq, tap_fft=True)
    n = 6
    fft = np.stack([r.fft(f) for f in range(n)])
    ce = np.array([r.info[f].clock_err for f in range(n)], np.float32)
    tii = np.array([0, 0, 1, 0, 0, 0], np.uint8)
    h = oracle.ofdm_new(0)
    want = []
    for f in range(n):
        oracle.ofdm_store_reference(h, fft[f, 0])
        for s in range(1, 76):
            oracle.ofdm_decode_symbol(h, fft[f, s], s, 0.0, float(ce[f]))
        if not tii[f]:
            oracle.ofdm_store_null(h, fft[f, 76])
        want.append(oracle_quality(oracle, h))
    oracle.ofdm_free(h)
    want = np.stack(want)
    plain = api.OfdmDecoder(0, ctx=ctx).decode_frames(fft, ce, tii)
    dec = api.OfdmDecoder(0, ctx=ctx)
    soft, q = dec.decode_frames(fft, ce, tii, quality=True)
    assert np.array_equal(soft, plain) and q.shape == (n, 6)
    check_records(q, want, "tap")
    assert (q[:, 5] == 0).all() and q[2, 4] == q[1, 4]  # a bare state has no CP phases; the TII null keeps the noise
    assert np.array_equal(q[-1].view(np.uint32), np.array(list(dec.quality().values()), np.float32).view(np.uint32))
    dec2 = api.OfdmDecoder(0, ctx=ctx)
    _, q1 = dec2.decode_frames(fft[:2], ce[:2], tii[:2], quality=True)
    _, q2 = dec2.decode_frames(fft[2:], ce[2:], tii[2:], quality=True)
    assert np.array_equal(np.concatenate([q1, q2]).view(np.uint32), q.view(np.uint32))
    r.close()


# ------------------------------------------------------------------------------------------------ GPU: determinism
@pytest.mark.gpu
def test_cut_windows(ctx):
    """max_window 4 against 128 on recordings whose FIC fails (low SNR, a lost time sync): windows are cut by verification and
    replayed, and each frame keeps the record of the pass that committed it."""
    iqs = [synth.generate(12, seed=90 + i, snr_db=5.0 + i, fmt=synth.FMT_U8).iq for i in range(4)] + [sync_loss_recording(synth.FMT_U8, seed=95)]
    big, small = gpu(ctx, iqs, max_window=128), gpu(ctx, iqs, max_window=4)
    assert sum(int(small.counters(r)[5]) for r in range(len(iqs))) > 0
    for r in range(len(iqs)):
        assert small.n_frames(r) == big.n_frames(r)
        assert np.array_equal(small.frame_quality(r).view(np.uint32), big.frame_quality(r).view(np.uint32)), r


def quality_records(dp, r: int, n_max: int) -> np.ndarray:
    """frame_quality of recording r padded with NaN to n_max rows."""
    q = dp.frame_quality(r)
    out = np.full((n_max, 6), np.nan, np.float32)
    out[:q.shape[0]] = q
    return out


def batch_quality(ctx) -> dict:
    """Records of the 256 copies of the batch sources in one DabProcessor (traced), then of every source decoded alone."""
    srcs = [S.batch_source(i)[0] for i in range(S.N_SRC)]
    dp, rounds, dev = S.decode_batch(ctx, srcs, 0, trace=True, frame_quality=True)
    out = dict(rounds=rounds,
               n_frames=np.array([dp.n_frames(r) for r in range(S.N_COPIES)], np.int64),
               quality=np.stack([quality_records(dp, r, S.F_MAX) for r in range(S.N_COPIES)]))
    del dp, dev
    single_n, single_q = [], []
    for i in range(S.N_SRC):
        dp1 = gpu(ctx, [srcs[i]])
        single_n.append(dp1.n_frames(0))
        single_q.append(quality_records(dp1, 0, S.F_MAX))
    out["single_n_frames"] = np.array(single_n, np.int64)
    out["single_quality"] = np.stack(single_q)
    return out


@pytest.mark.gpu
def test_batch_every_lag_bit_identical(ctx, oracle):
    """256 recordings (768 demapper CTAs, past one wave at every lag), every one ending inside a cut frame: at lag 3 / 7 / 15
    every copy's records equal its source decoded alone and the other lags' bit for bit, and the oracle chain's."""
    outs = {}
    for lag in LAGS:
        with S.forced_lag(lag):
            outs[lag] = batch_quality(ctx)
    ref = outs[LAGS[0]]
    n = ref["single_n_frames"]
    assert (n == S.N_FULL).all()
    for lag, o in outs.items():
        assert o["rounds"][0, 0] == S.N_COPIES
        assert np.array_equal(o["n_frames"], np.tile(n, S.N_COPIES // S.N_SRC)), lag
        q = o["quality"].view(np.uint32)
        for c in range(S.N_COPIES):
            assert np.array_equal(q[c], o["single_quality"][c % S.N_SRC].view(np.uint32)), (lag, c)
        assert np.array_equal(o["single_quality"].view(np.uint32), ref["single_quality"].view(np.uint32)), lag
    for i in range(0, S.N_SRC, 4):
        r = chain(oracle, S.batch_source(i)[0])
        assert r.n_frames == S.N_FULL
        check_records(ref["single_quality"][i, :S.N_FULL], chain_records(oracle, r), f"source {i}")
        r.close()


# ------------------------------------------------------------------------------------------------ GPU: segments, streaming, TII
@pytest.fixture(scope="module")
def long_chain(oracle):
    r = oracle.chain_run(oracle.to_cf32(S.segment_recording()), scan_mode=1, tap_fft=True)
    assert r.n_frames == N_LONG
    yield r
    r.close()


def replay_quality(oracle, r, segments):
    """Records of the kept frames of `segments` (demap_support.replay_segments: (first, last, warmup, parent)), from the
    chain's FFT rows and clock errors; field 5 from the chain's CP phases."""
    out = {}
    S.replay_segments(oracle, r.fft, [i.clock_err for i in r.info], segments, 0,
                      lambda f, h, soft: out.__setitem__(f, oracle_quality(oracle, h)))
    q = np.stack([out[f] for f in range(len(out))])
    q[:, 5] = sigma_replay([i.phase_cp for i in r.info])
    return q


def segment_quality(ctx, seg_frames, warmup, max_window) -> dict:
    """DabProcessor with set_segmentation and set_frame_quality over segment_recording() (traced)."""
    dp = api.DabProcessor(1, input_format=api.FMT_U8, scan_mode=True, max_window=max_window, ctx=ctx)
    dp.set_segmentation(seg_frames, warmup)
    dp.set_frame_quality(True)
    rounds = S.traced(lambda: dp.run([S.segment_recording()]))
    res = dp.result(0)
    return dict(rounds=rounds, warmup_frames=dp.warmup_frames(0), quality=dp.frame_quality(0),
                pos=np.array([(i.sym0_pos, i.start_index) for i in res.info], np.int64).reshape(-1, 2),
                phase_cp=np.array([i.phase_cp for i in res.info], np.float32))


@pytest.mark.gpu
@pytest.mark.parametrize("seg_frames,warmup,lag,max_window", [(48, 4, 15, 200), (48, 18, 15, 200), (2, 4, 3, 512)])
def test_segmented_records_match_replay(ctx, oracle, long_chain, seg_frames, warmup, lag, max_window):
    """set_segmentation over 400 frames: every record against the oracle replaying the engine's own segment layout (segments
    that warm up from reset() carry that state, as their soft bits do). (2, 4) is ~600 CTAs at lag 3, past one wave."""
    with S.forced_lag(lag):
        out = segment_quality(ctx, seg_frames, warmup, max_window)
    rounds = out["rounds"]
    assert (rounds[:, 0] == 1).all() and rounds[:, 1].sum() == N_LONG, rounds
    segs, total_w = engine_segments([int(n) for n in rounds[:, 1]], seg_frames, warmup)
    assert int(out["warmup_frames"]) == total_w > 0
    assert [tuple(p) for p in out["pos"]] == [(i.sym0_pos, i.start_index) for i in long_chain.info]
    want = replay_quality(oracle, long_chain, segs)
    check_records(out["quality"], want, f"segments {seg_frames}x{warmup}")
    assert np.array_equal(out["quality"][:, 5].view(np.uint32), sigma_replay(out["phase_cp"]).view(np.uint32))


@pytest.mark.gpu
def test_streaming_chunks(ctx):
    """A recording in 3 chunks with export / import: fields 0-4 bit identical to the one-run records (the OFDM state crosses
    the chunks in the state blob); field 5 is replayed from each run's own frames, so it starts again at every chunk."""
    rec = synth.generate(30, seed=101, snr_db=14.0, cfo_hz=1234.0, fmt=synth.FMT_U8)
    one = gpu(ctx, [rec.iq])
    want = one.frame_quality(0)
    ends = [2_000_001, 4_123_457, rec.iq.shape[0]]
    got, phases, blob, pos = [], [], None, 0
    for ci, end in enumerate(ends):
        dp = api.DabProcessor(1, input_format=synth.FMT_U8, scan_mode=True, ctx=ctx)
        dp.set_streaming(ci + 1 < len(ends))
        dp.set_frame_quality(True)
        start = pos
        if blob is not None:
            ld = min(1 << 21, pos)
            start = pos - ld
            dp.import_state(0, blob, ld)
        dp.run([rec.iq[start:end]])
        q = dp.frame_quality(0)
        assert q.shape[0] == dp.n_frames(0) > 0
        assert np.array_equal(q[:, 5].view(np.uint32), sigma_replay([i.phase_cp for i in dp.result(0).info]).view(np.uint32))
        got.append(q)
        if ci + 1 < len(ends):
            pos = dp.consumed(0)
            blob = dp.export_state(0)
    got = np.concatenate(got)
    assert got.shape == want.shape
    assert np.array_equal(got[:, :5].view(np.uint32), want[:, :5].view(np.uint32))
    assert not np.array_equal(got[:, 5], want[:, 5])


@pytest.mark.gpu
def test_self_configuration_tii_nulls(ctx, oracle):
    """Self-configuration level 2: the null symbols the recording's own CIF counter marks as TII leave the noise alone; the
    records (those of the final pass) match the oracle chain with track_cif."""
    rec = synth.generate(12, seed=102, snr_db=16.0, subch=[SC_3A], fmt=synth.FMT_U8, fig_mode=1, tii=(5, 3))
    r = chain(oracle, rec.iq, track_cif=True)
    dp = api.DabProcessor(1, input_format=synth.FMT_U8, ctx=ctx)
    dp.set_auto_config(0, True, tii_null_symbols=True)
    dp.set_frame_quality(True)
    dp.run([rec.iq])
    q = dp.frame_quality(0)
    want = chain_records(oracle, r, track_cif=True)
    check_records(q, want, "auto config 2")
    same = [f for f in range(1, q.shape[0]) if q[f, 4] == q[f - 1, 4]]
    assert same == [f for f in range(1, want.shape[0]) if want[f, 4] == want[f - 1, 4]] and len(same) >= 3
    r.close()
