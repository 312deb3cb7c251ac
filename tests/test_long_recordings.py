"""-m gpu: long recordings (SURVEY.md 8e, second half): one stream decoded as parallel segments with a warm-up prefix, and
as chunks across runs / decoders through export_state / import_state. The checker is the CPU oracle's SEQUENTIAL run
(ofdm_decoder.cpp:182-251, backend.cpp:129-161 and dab_processor.cpp:191-265 carry state across all frames)."""
import json

import numpy as np
import pytest

from dabstar_b200 import api, synth

pytestmark = pytest.mark.gpu

SC = [synth.SubChannel(3, 100, 54, 0, 2, 72), synth.SubChannel(7, 200, 96, 1, 3, 128)]
N_LONG = 400


@pytest.fixture(scope="module")
def long_rec():
    return synth.generate(N_LONG, seed=31, snr_db=15.0, subch=SC, fmt=synth.FMT_U8)


@pytest.fixture(scope="module")
def long_want(oracle, long_rec):
    return oracle.chain_run(oracle.to_cf32(long_rec.iq), synth.subch_table(SC), len(SC), tap_soft=True)


def _check_decoded(got, want, rec):
    assert got.n_frames == want.n_frames == N_LONG
    assert [(i.sym0_pos, i.start_index) for i in got.info] == [(i.sym0_pos, i.start_index) for i in want.info]
    assert [(round(i.fbb_data), round(i.fbb_null)) for i in got.info] == [(round(i.fbb_data), round(i.fbb_null)) for i in want.info]
    assert np.array_equal(got.fic_valid, want.fic_valid) and want.fic_valid.all()
    assert np.array_equal(got.fib_bits, want.fib_bits) and np.array_equal(got.fib_bits, rec.fib_truth)
    assert got.n_good_fibs == want.n_good_fibs == 12 * N_LONG
    for i, s in enumerate(SC):
        assert np.array_equal(got.msc[s.sub_ch_id], want.msc[s.sub_ch_id]), s
        assert np.array_equal(got.msc[s.sub_ch_id], rec.msc_truth[i][:got.msc[s.sub_ch_id].shape[0]])


def _soft_diff(dp, want, frames):
    over, n, worst = 0, 0, 0
    for f in frames:
        d = np.abs(dp.soft_bits(0, f).astype(np.int32) - want.soft_bits(f).astype(np.int32))
        over += int((d > 1).sum())
        n += d.size
        worst = max(worst, int(d.max()))
    return over / n, worst


def test_long_recording_sequential_parity(ctx, long_rec, long_want):
    """The unsegmented path over the whole stream: decoded bytes identical, soft bits within one LSB up to the LAST frame."""
    dp = api.DabProcessor(1, input_format=synth.FMT_U8, max_window=512, ctx=ctx)
    dp.set_audio_channel(0, SC)
    dp.run([long_rec.iq])
    _check_decoded(dp.result(0), long_want, long_rec)
    frac, worst = _soft_diff(dp, long_want, [0, 1, N_LONG // 2, N_LONG - 2, N_LONG - 1])
    assert frac <= 1e-4, (frac, worst)
    assert dp.warmup_frames(0) == 0


@pytest.mark.parametrize("warmup", [4, 18, 32])
def test_segmented_decode_identical_bytes(ctx, long_rec, long_want, warmup, record_property):
    """400 frames as >= 8 parallel segments: FIB / MSC bytes, CRC flags, positions and AFC identical to the sequential oracle
    run at 15 dB; the soft bits are approximated by the warm-up, the fraction beyond one LSB is reported per warm-up length."""
    dp = api.DabProcessor(1, input_format=synth.FMT_U8, max_window=512, ctx=ctx)
    dp.set_audio_channel(0, SC)
    dp.set_segmentation(48, warmup)
    dp.run([long_rec.iq])
    got = dp.result(0)
    _check_decoded(got, long_want, long_rec)
    n_warm = dp.warmup_frames(0)
    assert n_warm >= 7 * warmup and n_warm % warmup == 0, n_warm   # at least 8 segments, 7 of them warm-started
    frac_all, worst = _soft_diff(dp, long_want, range(0, N_LONG))
    # frames right after a segment start carry most of the difference
    report = {"frames": N_LONG, "segment_frames": 48, "warmup_frames": warmup, "segments_warm_started": n_warm // warmup,
              "soft_bits_beyond_1_lsb": frac_all, "max_abs_diff": worst, "fib_msc_identical": True, "snr_db": 15.0}
    print("segment parity:", json.dumps(report))
    record_property("segment_parity", json.dumps(report))   # (pytest --junitxml keeps it with the test result)
    assert frac_all < (0.2 if warmup < 18 else 0.05)


def test_segment_count_does_not_change_bytes(ctx, long_rec, long_want):
    """Short segments (16 frames) with the default warm-up: more redundancy, same bytes."""
    dp = api.DabProcessor(1, input_format=synth.FMT_U8, max_window=512, ctx=ctx)
    dp.set_audio_channel(0, SC)
    dp.set_segmentation(16, 18)
    dp.run([long_rec.iq])
    _check_decoded(dp.result(0), long_want, long_rec)


def _chunked_run(ctx, rec, cuts, lead, subch, new_decoder_per_chunk=True):
    """Decodes rec.iq as chunks [.., cuts[0]), [.., cuts[1]), ... each starting `lead` samples before the consumed position."""
    n_total = rec.iq.shape[0]
    ends = list(cuts) + [n_total]
    dp, blob = None, None
    pos = 0
    out = {"fib": [], "valid": [], "pos": [], "msc": {s.sub_ch_id: [] for s in subch}, "soft_last": None, "frames": 0}
    for ci, end in enumerate(ends):
        if dp is None or new_decoder_per_chunk:
            dp = api.DabProcessor(1, input_format=synth.FMT_U8, ctx=ctx)
            dp.set_audio_channel(0, subch)
        dp.set_streaming(ci + 1 < len(ends))  # the last chunk ends the stream: a cut frame is decoded as far as it goes
        start = pos
        if blob is not None:
            ld = min(lead, pos)
            start = pos - ld
            dp.import_state(0, blob, ld)
        dp.run([rec.iq[start:end]])
        got = dp.result(0)
        out["fib"].append(got.fib_bits)
        out["valid"].append(got.fic_valid)
        out["pos"] += [(i.sym0_pos, i.start_index, round(i.fbb_data), i.fic_ratio_after) for i in got.info]
        for s in subch:
            out["msc"][s.sub_ch_id].append(got.msc[s.sub_ch_id])
        if got.n_frames:
            out["soft_last"] = dp.soft_bits(0, got.n_frames - 1)
        out["frames"] += got.n_frames
        if ci + 1 < len(ends):
            pos = dp.consumed(0)
            assert pos <= end
            blob = dp.export_state(0)
    out["fib"] = np.concatenate(out["fib"])
    out["valid"] = np.concatenate(out["valid"])
    for s in subch:
        out["msc"][s.sub_ch_id] = np.concatenate(out["msc"][s.sub_ch_id])
    return out


@pytest.mark.parametrize("cuts", [(5_000_000,), (2_000_001, 4_123_457, 9_000_000), (30_000, 250_000, 700_000, 1_300_000)])
def test_stream_in_chunks_is_bit_exact(ctx, cuts):
    """A recording decoded chunk by chunk on fresh decoders (export_state / import_state) equals one run over the whole
    recording: frame positions, AFC, FIB bits and flags, MSC bytes, and the soft bits of the last frame bit for bit.
    The cuts are not frame aligned; the third case cuts inside the level estimate, the time sync and the first frames."""
    rec = synth.generate(56, seed=41, snr_db=14.0, cfo_hz=1234.0, subch=SC, fmt=synth.FMT_U8)
    one = api.DabProcessor(1, input_format=synth.FMT_U8, ctx=ctx)
    one.set_audio_channel(0, SC)
    one.run([rec.iq])
    want = one.result(0)
    got = _chunked_run(ctx, rec, cuts, lead=1 << 21, subch=SC)
    assert got["frames"] == want.n_frames == 56
    assert got["pos"] == [(i.sym0_pos, i.start_index, round(i.fbb_data), i.fic_ratio_after) for i in want.info]
    assert np.array_equal(got["valid"], want.fic_valid) and np.array_equal(got["fib"], want.fib_bits)
    for s in SC:
        assert np.array_equal(got["msc"][s.sub_ch_id], want.msc[s.sub_ch_id]), s
    assert np.array_equal(got["soft_last"], one.soft_bits(0, want.n_frames - 1))


def test_stream_chunks_on_one_decoder_and_short_lead(ctx):
    """The same decoder object may continue its own stream; without lead samples the result is the same as long as no time
    re-synchronisation falls on a chunk boundary (the lead only feeds the level estimate of the null-symbol search)."""
    rec = synth.generate(30, seed=43, snr_db=18.0, subch=SC[:1], fmt=synth.FMT_U8)
    one = api.DabProcessor(1, input_format=synth.FMT_U8, ctx=ctx)
    one.set_audio_channel(0, SC[:1])
    one.run([rec.iq])
    want = one.result(0)
    got = _chunked_run(ctx, rec, (1_500_000, 3_100_000), lead=0, subch=SC[:1], new_decoder_per_chunk=False)
    assert got["frames"] == want.n_frames
    assert np.array_equal(got["fib"], want.fib_bits) and np.array_equal(got["msc"][3], want.msc[3])


def test_export_state_needs_streaming(ctx):
    rec = synth.generate(6, seed=44, snr_db=20.0, fmt=synth.FMT_U8)
    dp = api.DabProcessor(1, input_format=synth.FMT_U8, ctx=ctx)
    dp.run([rec.iq])
    with pytest.raises(api.DabstarError):
        dp.export_state(0)
    with pytest.raises(api.DabstarError):
        dp.import_state(0, np.zeros(100, np.uint8))


def test_stream_sharded_over_ranks_identical_bytes(ctx):
    """parallel.stream_shard: one recording as three sample ranges, each decoded from a cold start a few frames early (what three
    ranks do, here one after the other on one GPU): FIB bits, flags, positions and MSC bytes of the stitched result equal one run."""
    from dabstar_b200 import parallel
    rec = synth.generate(150, seed=47, snr_db=15.0, subch=SC, fmt=synth.FMT_U8)
    one = api.DabProcessor(1, input_format=synth.FMT_U8, max_window=256, ctx=ctx)
    one.set_audio_channel(0, SC)
    one.run([rec.iq])
    want = one.result(0)
    parts = []
    for rank in range(3):
        sh = parallel.stream_shard(rec.iq.shape[0], rank, 3, warmup_frames=18)
        dp = api.DabProcessor(1, input_format=synth.FMT_U8, max_window=256, ctx=ctx)
        dp.set_audio_channel(0, SC)
        dp.set_streaming(rank < 2)  # the last range ends the stream
        parts.append(parallel.decode_stream_shard(dp, rec.iq[sh.in_lo:sh.in_hi], sh, SC))
        assert parts[-1]["decoded_frames"] >= parts[-1]["frames"] + (25 if rank else 0) - 2
    got = parallel.stitch(parts)
    assert got["frames"] == want.n_frames == 150
    assert got["pos"] == [i.sym0_pos for i in want.info]
    assert np.array_equal(got["valid"], want.fic_valid) and np.array_equal(got["fib"], want.fib_bits)
    for s in SC:
        assert np.array_equal(got["msc"][s.sub_ch_id], want.msc[s.sub_ch_id]), s
