"""-m gpu: DAB+ super-frames and access units inside the whole-path decoder (dabstar_decoder_set_dabplus), and the stage tap
dabstar_dabplus_decode on the same batched device pass. Real super-frames travel through the RF chain (synth msc_payload);
every stream is compared, record for record and byte for byte, with the tap and the oracle's Mp4Processor run on the
decoder's own MSC bits."""
import numpy as np
import pytest

import helpers
from dabstar_b200 import api, synth
from dabstar_b200._lib import DabstarError
from test_dabplus_walk import SCENARIOS, scenario_stream

pytestmark = pytest.mark.gpu
E_INVALID, E_UNSUPPORTED = -1, -4

# (sub_ch_id, start_cu, size_cu, short_form, prot_level, bit_rate): DAB+ at 8 / 32 / 72 / 128 kbit/s (EEP-A and EEP-B), one UEP
# sub-channel (MPEG layer II in the synthetic FIG 0/2) and one EEP sub-channel that carries random bits
LAYOUT = [(1, 0, 6, 0, 2, 8), (2, 6, 18, 0, 6, 32), (3, 24, 54, 0, 2, 72), (4, 78, 96, 0, 2, 128), (5, 174, 96, 1, 3, 128), (6, 270, 30, 0, 7, 64)]
SUBCH = [synth.SubChannel(i, cu, size, sf, lvl, br) for i, cu, size, sf, lvl, br in LAYOUT]
DABPLUS = [1, 2, 3, 4]  # carry super-frames
EEP = [1, 2, 3, 4, 6]


def key(r):
    return (r.first_frame, r.ok, r.rs_errors, r.rs_corrections, r.fc_corrected, r.dac_rate, r.sbr_flag, r.aac_channel_mode, r.ps_flag, r.mpeg_surround,
            r.num_aus, tuple(r.au_start), tuple(r.au_state))


def superframe_payload(oracle, bit_rate, n_frames, seed, lead=3, junk=None, slip=None, byte_errors=0.0):
    """Logical frames of n_frames DAB frames (4 per frame) carrying super-frames from frame `lead` on: random bits in front,
    junk: (first, count) super-frames left as random bits, slip: one random frame inserted before super-frame `slip`,
    byte_errors: that share of all bytes corrupted. Returns (bits, {first_frame: access units})."""
    rng = np.random.default_rng(seed)
    n = 4 * n_frames
    bits = rng.integers(0, 2, (n, 24 * bit_rate), dtype=np.uint8)
    truth, f, i = {}, lead, 0
    while f + 5 <= n:
        if slip is not None and i == slip:
            f += 1
            slip = None
            continue
        # at 8 kbit/s, 110 bytes leave no room for 4 or 6 access units: SBR on (2 or 3)
        b, aus = helpers.dabplus_superframe(bit_rate, rng, oracle.rs_encode, dac_rate=i % 2, sbr_flag=1 if bit_rate < 32 else (i // 2) % 2)
        if junk is None or not junk[0] <= i < junk[0] + junk[1]:
            bits[f:f + 5] = b
            truth[f] = aus
        f += 5
        i += 1
    if byte_errors:
        by = np.packbits(bits.reshape(-1))
        pos = rng.choice(by.size, int(by.size * byte_errors), replace=False)
        by[pos] ^= rng.integers(1, 256, pos.size, dtype=np.uint8)
        bits = np.unpackbits(by).reshape(bits.shape)
    return bits, truth


def make_recording(oracle, n_frames, seed, fmt, snr_db=25.0, fig_mode=0, **damage):
    pays, truths = [], {}
    for s in SUBCH:
        if s.sub_ch_id in DABPLUS:
            bits, truth = superframe_payload(oracle, s.bit_rate, n_frames, seed * 100 + s.sub_ch_id, lead=1 + s.sub_ch_id, **damage)
            pays.append(bits)
            truths[s.sub_ch_id] = truth
        else:
            pays.append(None)
    rec = synth.generate(n_frames, seed=seed, snr_db=snr_db, subch=SUBCH, fmt=fmt, fig_mode=fig_mode, msc_payload=pays)
    return rec, truths


def check_stream(ctx, oracle, dp, r, sid, bit_rate, msc=None):
    """The decoder's records and payload of one stream equal the tap's and the oracle's on the decoder's own bits."""
    bits = dp.result(r).msc[sid] if msc is None else msc
    got_rec, got_pay = dp.superframes(r, sid)
    want_rec, want_pay = oracle.dabplus_run(bits, bit_rate)
    tap_rec, tap_pay = api.Mp4Processor(bit_rate, ctx).add_frames(bits)
    assert [key(g) for g in got_rec] == [w.key() for w in want_rec] == [key(t) for t in tap_rec], (r, sid)
    assert got_pay.shape == want_pay.shape and np.array_equal(got_pay, want_pay) and np.array_equal(tap_pay, want_pay), (r, sid)
    return got_rec, got_pay


def decoder(ctx, n, fmt, **kw):
    return api.DabProcessor(n, input_format=fmt, ctx=ctx, **kw)


@pytest.mark.parametrize("fmt", [synth.FMT_U8, synth.FMT_I16])
def test_chain_clean(ctx, oracle, fmt):
    recs = [make_recording(oracle, 40, seed=20 + k, fmt=fmt) for k in range(2)]
    dp = decoder(ctx, 2, fmt)
    for r in range(2):
        dp.set_audio_channel(r, SUBCH)
        for sid in EEP:
            dp.set_dabplus(r, sid)
    dp.run([rec.iq for rec, _ in recs])
    ms, rounds = dp.dabplus_ms()
    assert ms > 0 and 1 <= rounds <= 2
    for r, (rec, truths) in enumerate(recs):
        for s in SUBCH:
            if s.sub_ch_id not in EEP:
                with pytest.raises(DabstarError):
                    dp.superframes(r, s.sub_ch_id)
                continue
            got_rec, got_pay = check_stream(ctx, oracle, dp, r, s.sub_ch_id, s.bit_rate)
            if s.sub_ch_id == 6:
                continue  # random bits: whatever the oracle attempts (normally nothing)
            truth = truths[s.sub_ch_id]
            first = min(truth)
            assert got_rec and got_rec[0].first_frame == first
            assert len(got_rec) == len([f for f in truth if f + 5 <= dp.result(r).msc[s.sub_ch_id].shape[0]])
            for g, p in zip(got_rec, got_pay):
                assert g.ok and g.rs_corrections == 0 and g.rs_errors == 0
                assert api.Mp4Processor.access_units(g, p) == truth[g.first_frame]


@pytest.mark.parametrize("case", ["low_snr", "junk_and_slip"])
def test_chain_damaged(ctx, oracle, case):
    if case == "low_snr":
        # 6.2 dB is just above where this layout loses frame sync (the 32 kbit/s EEP-B sub-channel already needs RS corrections);
        # 3 % of the payload bytes corrupted on top make some code words uncorrectable
        rec, _ = make_recording(oracle, 40, seed=31, fmt=synth.FMT_U8, snr_db=6.2, byte_errors=0.03)
    else:
        rec, _ = make_recording(oracle, 48, seed=32, fmt=synth.FMT_U8, junk=(6, 6), slip=14)
    dp = decoder(ctx, 1, synth.FMT_U8)
    dp.set_audio_channel(0, SUBCH)
    for sid in EEP:
        dp.set_dabplus(0, sid)
    dp.run([rec.iq])
    _, rounds = dp.dabplus_ms()
    recs = {s.sub_ch_id: check_stream(ctx, oracle, dp, 0, s.sub_ch_id, s.bit_rate)[0] for s in SUBCH if s.sub_ch_id in EEP}
    dab = [r for sid in DABPLUS for r in recs[sid]]
    if case == "low_snr":
        assert sum(r.rs_corrections for r in dab) > 0 and any(r.rs_errors for r in dab)
    else:
        assert rounds > 2
        for sid in DABPLUS:  # lost at the junk, found again, and realigned after the slipped frame
            firsts = [r.first_frame for r in recs[sid] if r.ok]
            assert any((b - a) % 5 for a, b in zip(firsts, firsts[1:])) and any(not r.ok for r in recs[sid])


def test_batch_beyond_one_wave_and_segmentation(ctx, oracle):
    """Enough streams that the decode launch spans more than one wave; every stream equals its recording decoded alone, and
    (clean signal) the run with segmentation."""
    n_rec = 128
    uniq = [make_recording(oracle, 32, seed=40 + k, fmt=synth.FMT_U8) for k in range(3)]
    iqs = [uniq[r % 3][0].iq for r in range(n_rec)]
    runs = []
    for seg in (False, True):
        dp = decoder(ctx, n_rec, synth.FMT_U8)
        if seg:
            dp.set_segmentation(6, 18)
        for r in range(n_rec):
            dp.set_audio_channel(r, SUBCH)
            for sid in EEP:
                dp.set_dabplus(r, sid)
        dp.run(iqs)
        runs.append({(r, sid): dp.superframes(r, sid) for r in range(n_rec) for sid in EEP})
    # the first decode launch has a thread per (window, code word slot of 24): more blocks of 128 than the 148 SMs hold at once
    # (k_dabplus_rs: 48 registers, so 10 blocks per SM)
    windows = sum(len(v[0]) for v in runs[0].values())
    assert windows * 24 > 148 * 10 * 128, windows
    for u in range(3):
        alone = decoder(ctx, 1, synth.FMT_U8)
        alone.set_audio_channel(0, SUBCH)
        for sid in EEP:
            alone.set_dabplus(0, sid)
        alone.run([uniq[u][0].iq])
        for r in range(u, n_rec, 3):
            for sid in EEP:
                a_rec, a_pay = alone.superframes(0, sid)
                for run in runs:
                    g_rec, g_pay = run[(r, sid)]
                    assert [key(x) for x in g_rec] == [key(x) for x in a_rec] and np.array_equal(g_pay, a_pay), (r, sid)


def test_self_configuration(ctx, oracle):
    rec, _ = make_recording(oracle, 40, seed=51, fmt=synth.FMT_U8, fig_mode=1)
    runs = {}
    for mode in ("all", "explicit", "level2"):
        dp = decoder(ctx, 1, synth.FMT_U8)
        dp.set_auto_config(0, True, tii_null_symbols=mode == "level2")
        if mode == "level2":
            dp.set_tii_processing(0, True)
        for sid in ([-1] if mode != "explicit" else EEP):
            dp.set_dabplus(0, sid)
        dp.run([rec.iq])
        assert sorted(sid for sid in range(64) if _decoded(dp, 0, sid)) == EEP  # -1: exactly the sub-channels FIG 0/2 lists as DAB+
        # the components are what the FIB parser makes of the decoder's own CRC-good FIBs
        res = dp.result(0)
        fp = api.FibParser()
        for f in range(res.n_frames):
            for k in range(12):
                if res.fic_valid[f, k // 3]:
                    fp.process_FIB(res.fib_bits[f, 256 * k:256 * (k + 1)])
        assert dp.components(0) == fp.components()
        assert {c.sub_ch_id for c in dp.components(0) if c.tmid == 0 and c.type == 63} == set(EEP)
        runs[mode] = {}
        for s in SUBCH:
            if s.sub_ch_id in EEP:
                got_rec, got_pay = check_stream(ctx, oracle, dp, 0, s.sub_ch_id, s.bit_rate)
                runs[mode][s.sub_ch_id] = ([key(x) for x in got_rec], got_pay)
                if s.sub_ch_id in DABPLUS:
                    assert len(got_rec) >= 20 and all(r.ok for r in got_rec)
    for mode in ("explicit", "level2"):
        for sid in EEP:
            assert runs[mode][sid][0] == runs["all"][sid][0] and np.array_equal(runs[mode][sid][1], runs["all"][sid][1]), (mode, sid)
    plain = decoder(ctx, 1, synth.FMT_U8)
    plain.set_audio_channel(0, SUBCH)
    plain.run([rec.iq])
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        plain.components(0)  # not self-configured


def _decoded(dp, r, sid):
    try:
        dp.superframes(r, sid)
        return True
    except DabstarError:
        return False


def test_no_side_effects(ctx, oracle):
    rec, _ = make_recording(oracle, 30, seed=61, fmt=synth.FMT_U8)
    out = []
    for on in (False, True):
        dp = decoder(ctx, 1, synth.FMT_U8)
        dp.set_audio_channel(0, SUBCH)
        if on:
            for sid in EEP:
                dp.set_dabplus(0, sid)
        dp.run([rec.iq])
        res = dp.result(0)
        packed = {s.sub_ch_id: _msc_packed(dp, s) for s in SUBCH}
        info = [bytes(i) for i in res.info]
        out.append((res.fib_bits, res.fic_valid, packed, info, res.counters, dp.quality(0), dp.fib_packed(0)))
    a, b = out
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[3] == b[3] and np.array_equal(a[4], b[4]) and a[5] == b[5]
    assert np.array_equal(a[6], b[6])
    for sid in a[2]:
        assert np.array_equal(a[2][sid], b[2][sid])


def _msc_packed(dp, s):
    import ctypes
    n = int(dp.ctx.lib.dabstar_decoder_msc_size(dp.h, 0, s.sub_ch_id)) // 8
    out = np.zeros(max(n, 1), np.uint8)
    dp.ctx.lib.dabstar_decoder_msc_packed(dp.h, 0, s.sub_ch_id, out.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(n))
    return out[:n]


@pytest.mark.parametrize("bit_rate", [8, 32, 72, 96, 128])
@pytest.mark.parametrize("scenario", SCENARIOS)
def test_tap_on_the_batched_path(ctx, oracle, bit_rate, scenario):
    stream, _ = scenario_stream(oracle, bit_rate, scenario, seed=3)
    want_rec, want_pay = oracle.dabplus_run(stream, bit_rate)
    got_rec, got_pay = api.Mp4Processor(bit_rate, ctx).add_frames(stream)
    assert [key(g) for g in got_rec] == [w.key() for w in want_rec]
    assert np.array_equal(got_pay, want_pay)


def test_tap_one_by_one_equals_the_batch(ctx, oracle):
    """200 short streams of mixed bit rates through the decoder as one batch (the recordings' MSC payload) equal the tap run on
    each stream alone."""
    n_rec = 40  # x 5 EEP sub-channels = 200 streams
    uniq = [make_recording(oracle, 8, seed=70 + k, fmt=synth.FMT_U8, snr_db=9.0 + k) for k in range(4)]
    dp = decoder(ctx, n_rec, synth.FMT_U8)
    for r in range(n_rec):
        dp.set_audio_channel(r, SUBCH)
        for sid in EEP:
            dp.set_dabplus(r, sid)
    dp.run([uniq[r % 4][0].iq for r in range(n_rec)])
    n_streams = 0
    for r in range(n_rec):
        res = dp.result(r)
        for s in SUBCH:
            if s.sub_ch_id in EEP:
                got_rec, got_pay = dp.superframes(r, s.sub_ch_id)
                tap_rec, tap_pay = api.Mp4Processor(s.bit_rate, ctx).add_frames(res.msc[s.sub_ch_id])
                assert [key(g) for g in got_rec] == [key(t) for t in tap_rec] and np.array_equal(got_pay, tap_pay), (r, s.sub_ch_id)
                n_streams += 1
    assert n_streams == 200


def test_rejections(ctx, oracle):
    dp = decoder(ctx, 1, synth.FMT_U8)
    dp.set_audio_channel(0, SUBCH)
    for sid in (-1, 17):  # -1 without self-configuration; an unknown sub-channel
        with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
            dp.set_dabplus(0, sid)
    dp2 = decoder(ctx, 1, synth.FMT_U8)
    dp2.set_audio_channel(0, [synth.SubChannel(9, 0, 100, 0, 3, 200)])  # EEP 4-A at 200 kbit/s
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        dp2.set_dabplus(0, 9)  # outside 8..192 (every sub-channel profile has a multiple of 8)
    rec, _ = make_recording(oracle, 6, seed=81, fmt=synth.FMT_U8)
    st = decoder(ctx, 1, synth.FMT_U8)
    st.set_audio_channel(0, SUBCH)
    st.set_dabplus(0, 3)
    st.set_streaming(True)
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_UNSUPPORTED):
        st.run([rec.iq])
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_UNSUPPORTED):
        st.set_dabplus(0, 2)
    ok = decoder(ctx, 1, synth.FMT_U8)
    ok.set_audio_channel(0, SUBCH)
    ok.set_dabplus(0, 3)
    ok.run([rec.iq])
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        ok.superframes(0, 2)  # decoded, but not DAB+-decoded
    short = decoder(ctx, 1, synth.FMT_U8)  # a run too short for five logical frames: DAB+-decoded, no records
    short.set_audio_channel(0, SUBCH)
    short.set_dabplus(0, 3)
    short.run([rec.iq[:60000 + 5 * synth.T_FRAME]])
    assert short.result(0).msc[3].shape[0] < 5 and short.superframes(0, 3)[0] == []
    short = api.Mp4Processor(72, ctx).add_frames(np.zeros((4, 24 * 72), np.uint8))
    assert short[0] == []


def test_file_harness_prints_and_writes_the_access_units(ctx, oracle, tmp_path):
    import os
    import shutil
    import subprocess
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "dab_file_decode")
    subprocess.run(["g++", "-std=c++17", "-O2", os.path.join(root, "dabstar_b200", "host", "dab_file_decode.cpp"), "-I", os.path.join(root, "include"),
                    "-L", os.path.join(root, "dabstar_b200"), "-ldabstar_b200", "-Wl,-rpath," + os.path.join(root, "dabstar_b200"), "-o", exe], check=True)
    rec, truths = make_recording(oracle, 30, seed=91, fmt=synth.FMT_U8, fig_mode=1)
    path = str(tmp_path / "rec.iq")
    rec.iq.tofile(path)
    r = subprocess.run([exe, "-f", "u8", "-a", "-d", "all", "-o", str(tmp_path / "o_"), path], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lines = {int(l.split("DAB+ sub-channel ")[1].split(":")[0]): l for l in r.stdout.splitlines() if "DAB+ sub-channel" in l}
    assert sorted(lines) == EEP, r.stdout
    for sid in DABPLUS:
        good = int(lines[sid].split(" AUs good")[0].split(", ")[-1])
        assert good > 0, lines[sid]
        raw = open(str(tmp_path / f"o_0.subch{sid}.aus"), "rb").read()
        aus, o = [], 0
        while o < len(raw):
            n = (raw[o] << 8) | raw[o + 1]
            aus.append(raw[o + 2:o + 2 + n])
            o += 2 + n
        assert len(aus) == good
        sent = [au for f in sorted(truths[sid]) for au in truths[sid][f]]
        k = sent.index(aus[0])  # the self-configured Backend starts a frame after the FIC described the sub-channel
        assert aus == sent[k:k + len(aus)]
