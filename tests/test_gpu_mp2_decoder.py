"""-m gpu: MPEG layer II audio frames inside the whole-path decoder (dabstar_decoder_set_mp2), and the stage tap dabstar_mp2_frames
on the same batched device pass. Layer II frames travel through the RF chain (synth msc_payload) on UEP sub-channels (48 kHz) and
on explicitly selected EEP sub-channels (24 kHz); every stream is compared, record for record and byte for byte, with the tap and
the plain-C oracle run on the decoder's own MSC bits."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import mp2_support as ms
from dabstar_b200 import api, synth
from dabstar_b200._lib import DabstarError
from mp2_support import CRC_ERROR, NO_HEADER, OK

pytestmark = pytest.mark.gpu
E_INVALID, E_UNSUPPORTED = -1, -4

# (sub_ch_id, start_cu, size_cu, short_form, prot_level, bit_rate, sample_rate, mode): UEP rates of the full-ensemble layout
# (tools/bench_full_ensemble.py) as 48 kHz stereo, joint stereo (mode_extension 0..3 in turn), mono and dual channel (both
# Table B.2c: 32 kbit/s per channel), 24 kHz frames on two EEP sub-channels, and one EEP sub-channel at 72 kbit/s (no layer II
# rate) that carries random bits
LAYOUT = [(1, 0, 96, 1, 3, 128, 48000, 0), (2, 96, 84, 1, 4, 128, 48000, 1), (3, 180, 16, 1, 5, 32, 48000, 3), (4, 196, 42, 1, 4, 64, 48000, 2),
          (5, 238, 36, 0, 2, 48, 24000, 1), (6, 274, 54, 0, 4, 64, 24000, 3), (7, 328, 54, 0, 2, 72, None, None)]
SUBCH = [synth.SubChannel(i, cu, size, sf, lvl, br) for i, cu, size, sf, lvl, br, _, _ in LAYOUT]
MP2 = [1, 2, 3, 4, 5, 6]
UEP = [1, 2, 3, 4]  # FIG 0/2 of the synthetic transmitter: UEP -> ASCTy 0 (MPEG layer II), EEP -> ASCTy 63 (DAB+)
RATE = {x[0]: x[5] for x in LAYOUT}


def make_recording(n_frames, seed, fmt, snr_db=25.0, fig_mode=0, **damage):
    pays, truths = [], {}
    for sid, _, _, _, _, br, sr, mode in LAYOUT:
        if sr is None:
            pays.append(None)
            continue
        rng = np.random.default_rng(seed * 100 + sid)
        bits, truth = ms.mp2_stream(br, 4 * n_frames, rng, sample_rate=sr, mode=mode, lead=sid % 3, **damage)
        pays.append(bits)
        truths[sid] = truth
    rec = synth.generate(n_frames, seed=seed, snr_db=snr_db, subch=SUBCH, fmt=fmt, fig_mode=fig_mode, msc_payload=pays)
    return rec, truths


def decoder(ctx, n, fmt=synth.FMT_U8, **kw):
    return api.DabProcessor(n, input_format=fmt, ctx=ctx, **kw)


def check_stream(ctx, dp, r, sid):
    """The decoder's records and payload of one stream equal the tap's and the oracle's on the decoder's own bits."""
    bits = dp.result(r).msc[sid]
    got_rec, got_pay = dp.mp2_frames(r, sid)
    want_rec, want_pay = ms.oracle().run(bits, RATE[sid])
    tap_rec, tap_pay = api.Mp2Processor(RATE[sid], ctx).add_frames(bits)
    assert [ms.key(g) for g in got_rec] == [ms.key(w) for w in want_rec] == [ms.key(t) for t in tap_rec], (r, sid)
    assert np.array_equal(got_pay, want_pay) and np.array_equal(tap_pay, want_pay), (r, sid)
    return got_rec, got_pay


def selected(dp, r, sid):
    try:
        dp.mp2_frames(r, sid)
        return True
    except DabstarError:
        return False


@pytest.mark.parametrize("fmt", [synth.FMT_U8, synth.FMT_I16])
def test_chain_clean(ctx, fmt):
    recs = [make_recording(40, seed=20 + k, fmt=fmt) for k in range(2)]
    dp = decoder(ctx, 2, fmt)
    for r in range(2):
        dp.set_audio_channel(r, SUBCH)
        for sid in MP2:
            dp.set_mp2(r, sid)
    dp.run([rec.iq for rec, _ in recs])
    assert dp.mp2_ms() > 0
    for r, (rec, truths) in enumerate(recs):
        assert not selected(dp, r, 7)
        for sid in MP2:
            got_rec, got_pay = check_stream(ctx, dp, r, sid)
            n = dp.result(r).msc[sid].shape[0]
            sent = {f: t for f, t in truths[sid].items() if f + t.shape[0] <= n}
            frames = {rec.first_frame: fb for rec, fb in api.Mp2Processor.frames(got_rec, got_pay, RATE[sid])}
            assert sorted(frames) == sorted(sent), (r, sid)
            for f, t in sent.items():
                assert frames[f] == np.packbits(t.reshape(-1)).tobytes(), (r, sid, f)


@pytest.mark.parametrize("case", ["low_snr", "junk_and_slip"])
def test_chain_damaged(ctx, case):
    if case == "low_snr":
        # 6.2 dB is just above where this layout loses frame sync; 0.3 % of the payload bytes corrupted on top
        rec, _ = make_recording(40, seed=31, fmt=synth.FMT_U8, snr_db=6.2, byte_errors=0.003)
    else:
        rec, _ = make_recording(48, seed=32, fmt=synth.FMT_U8, junk=range(6, 12), slip=14, damage_header=(20, 21))
    dp = decoder(ctx, 1)
    dp.set_audio_channel(0, SUBCH)
    for sid in MP2:
        dp.set_mp2(0, sid)
    dp.run([rec.iq])
    recs = {sid: check_stream(ctx, dp, 0, sid)[0] for sid in MP2}
    st = [r.status for sid in MP2 for r in recs[sid]]
    assert st.count(OK) > 0
    if case == "low_snr":
        assert st.count(CRC_ERROR) > 0
    else:
        assert st.count(NO_HEADER) > 0
        for sid in MP2:  # found again after the junk and the slipped frame
            assert any(r.status == OK and r.first_frame > 4 * 16 for r in recs[sid]), sid


def test_batch_beyond_one_wave_and_segmentation(ctx):
    """64 recordings x 6 MP2 sub-channels: the compaction (one CTA of 128 threads per record) spans several waves of the 148 SMs at
    16 resident CTAs each, the scan (one thread per logical frame) more than two CTAs per SM. Every stream equals its recording
    decoded alone, and (clean signal) the run with segmentation."""
    n_rec = 64
    uniq = [make_recording(32, seed=40 + k, fmt=synth.FMT_U8) for k in range(3)]
    iqs = [uniq[r % 3][0].iq for r in range(n_rec)]
    runs = []
    for seg in (False, True):
        dp = decoder(ctx, n_rec)
        if seg:
            dp.set_segmentation(6, 18)
        for r in range(n_rec):
            dp.set_audio_channel(r, SUBCH)
            for sid in MP2:
                dp.set_mp2(r, sid)
        dp.run(iqs)
        runs.append({(r, sid): dp.mp2_frames(r, sid) for r in range(n_rec) for sid in MP2})
    records = sum(len(v[0]) for v in runs[0].values())
    slots = sum(sum(x.n_frames for x in v[0]) for v in runs[0].values())
    assert records > 3 * 148 * 16 and slots > 2 * 148 * 128, (records, slots)
    for u in range(3):
        alone = decoder(ctx, 1)
        alone.set_audio_channel(0, SUBCH)
        for sid in MP2:
            alone.set_mp2(0, sid)
        alone.run([uniq[u][0].iq])
        for r in range(u, n_rec, 3):
            for sid in MP2:
                a_rec, a_pay = alone.mp2_frames(0, sid)
                for run in runs:
                    g_rec, g_pay = run[(r, sid)]
                    assert [ms.key(x) for x in g_rec] == [ms.key(x) for x in a_rec] and np.array_equal(g_pay, a_pay), (r, sid)


def test_self_configuration(ctx):
    rec, _ = make_recording(40, seed=51, fmt=synth.FMT_U8, fig_mode=1)
    runs = {}
    for mode in ("all", "explicit", "level2", "with_dabplus"):
        dp = decoder(ctx, 1)
        dp.set_auto_config(0, True, tii_null_symbols=mode == "level2")
        if mode == "level2":
            dp.set_tii_processing(0, True)
        for sid in ([-1] if mode != "explicit" else UEP):
            dp.set_mp2(0, sid)
        if mode == "with_dabplus":
            dp.set_dabplus(0, -1)
        dp.run([rec.iq])
        assert sorted(sid for sid in range(64) if selected(dp, 0, sid)) == UEP, mode  # -1: exactly the ASCTy 0 sub-channels
        assert {c.sub_ch_id for c in dp.components(0) if c.tmid == 0 and c.type == 0} == set(UEP)
        runs[mode] = {sid: check_stream(ctx, dp, 0, sid) for sid in UEP}
        for sid in UEP:
            assert sum(r.status == OK for r in runs[mode][sid][0]) >= 20
        if mode == "with_dabplus":
            dab_both = {sid: dp.superframes(0, sid) for sid in (5, 6, 7)}
    for mode in ("explicit", "level2", "with_dabplus"):
        for sid in UEP:
            a, b = runs[mode][sid], runs["all"][sid]
            assert [ms.key(x) for x in a[0]] == [ms.key(x) for x in b[0]] and np.array_equal(a[1], b[1]), (mode, sid)
    dab = decoder(ctx, 1)  # DAB+ -1 alone: what it gave beside MP2 -1
    dab.set_auto_config(0, True)
    dab.set_dabplus(0, -1)
    dab.run([rec.iq])
    for sid in (5, 6, 7):
        a, b = dab.superframes(0, sid), dab_both[sid]
        assert [bytes(x) for x in a[0]] == [bytes(x) for x in b[0]] and np.array_equal(a[1], b[1]), sid


def test_level2_runs_the_pass_once_after_the_final_pass(ctx):
    """With self-configuration level 2 a run decodes the recording more than once (it makes more launches than the same run at
    level 1); the MP2 pass (three launches: scan, walk, compact) still runs once, after the final pass."""
    rec, _ = make_recording(40, seed=51, fmt=synth.FMT_U8, fig_mode=1)
    launches = {}
    for mode in ("level1", "level2", "level2_mp2"):
        dp = decoder(ctx, 1)
        dp.set_auto_config(0, True, tii_null_symbols=mode != "level1")
        dp.set_tii_processing(0, True)
        if mode == "level2_mp2":
            dp.set_mp2(0, -1)
        before = ctx.kernel_launches
        dp.run([rec.iq])
        launches[mode] = ctx.kernel_launches - before
    assert launches["level2"] > launches["level1"], launches
    assert launches["level2_mp2"] - launches["level2"] == 3, launches


def test_no_side_effects(ctx):
    rec, _ = make_recording(30, seed=61, fmt=synth.FMT_U8)
    out = []
    for on in (False, True):
        dp = decoder(ctx, 1)
        dp.set_audio_channel(0, SUBCH)
        for sid in (5, 6):  # DAB+ on two sub-channels in both runs; the same two also MP2-decoded in the second
            dp.set_dabplus(0, sid)
        if on:
            for sid in MP2:
                dp.set_mp2(0, sid)
        dp.run([rec.iq])
        res = dp.result(0)
        msc = {s.sub_ch_id: res.msc[s.sub_ch_id].copy() for s in SUBCH}
        dab = {sid: ([bytes(x) for x in dp.superframes(0, sid)[0]], dp.superframes(0, sid)[1]) for sid in (5, 6)}
        out.append((res.fib_bits, res.fic_valid, msc, [bytes(i) for i in res.info], res.counters, dp.fib_packed(0), dab))
    a, b = out
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[3] == b[3] and np.array_equal(a[4], b[4]) and np.array_equal(a[5], b[5])
    for sid in a[2]:
        assert np.array_equal(a[2][sid], b[2][sid])
    for sid in (5, 6):
        assert a[6][sid][0] == b[6][sid][0] and np.array_equal(a[6][sid][1], b[6][sid][1])


@pytest.mark.parametrize("bit_rate", [8, 32, 64, 128, 160, 384])
def test_tap_on_the_batched_path(ctx, bit_rate):
    rng = np.random.default_rng(bit_rate)
    streams = [ms.mp2_stream(bit_rate, 61, rng, mixed=True, byte_errors=0.002, lead=1)[0], ms.mp2_stream(bit_rate, 7, rng, junk=range(100))[0],
               ms.mp2_stream(bit_rate, 1, rng, sample_rate=24000 if bit_rate in ms.RATES_LSF else 48000)[0],
               # longer than the walk's 256 threads: chunks of several slots whose borders fall inside 24 kHz frames
               ms.mp2_stream(bit_rate, 1999, rng, mixed=True, byte_errors=0.001, slip=37, damage_header=(50, 51, 300))[0]]
    for s in streams:
        want_rec, want_pay = ms.oracle().run(s, bit_rate)
        got_rec, got_pay = api.Mp2Processor(bit_rate, ctx).add_frames(s)
        assert [ms.key(g) for g in got_rec] == [ms.key(w) for w in want_rec]
        assert np.array_equal(got_pay, want_pay)


def test_rejections(ctx):
    dp = decoder(ctx, 1)
    dp.set_audio_channel(0, SUBCH)
    for sid in (-1, 17, 7):  # -1 without self-configuration; an unknown sub-channel; 72 kbit/s, no layer II rate
        with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
            dp.set_mp2(0, sid)
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        api.Mp2Processor(72, ctx).add_frames(np.zeros((2, 24 * 72), np.uint8))
    rec, _ = make_recording(6, seed=81, fmt=synth.FMT_U8)
    st = decoder(ctx, 1)
    st.set_audio_channel(0, SUBCH)
    st.set_mp2(0, 3)
    st.set_streaming(True)
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_UNSUPPORTED):
        st.run([rec.iq])
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_UNSUPPORTED):
        st.set_mp2(0, 2)
    ok = decoder(ctx, 1)
    ok.set_audio_channel(0, SUBCH)
    ok.set_mp2(0, 3)
    ok.run([rec.iq])
    ok.mp2_frames(0, 3)
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        ok.mp2_frames(0, 2)  # decoded, but not MP2-decoded
    scan = decoder(ctx, 1, scan_mode=True)
    scan.set_audio_channel(0, SUBCH)
    scan.set_mp2(0, 3)
    scan.run([rec.iq])
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        scan.mp2_frames(0, 3)  # no MSC, so no frames


def test_file_harness_writes_the_frames(ctx, tmp_path):
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "dab_file_decode")
    subprocess.run(["g++", "-std=c++17", "-O2", os.path.join(root, "dabstar_b200", "host", "dab_file_decode.cpp"), "-I", os.path.join(root, "include"),
                    "-L", os.path.join(root, "dabstar_b200"), "-ldabstar_b200", "-Wl,-rpath," + os.path.join(root, "dabstar_b200"), "-o", exe], check=True)
    rec, _ = make_recording(30, seed=91, fmt=synth.FMT_U8, fig_mode=1)
    path = str(tmp_path / "rec.iq")
    rec.iq.tofile(path)
    r = subprocess.run([exe, "-f", "u8", "-a", "-m", "all", "-o", str(tmp_path / "o_"), path], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lines = {int(l.split("MP2 sub-channel ")[1].split(":")[0]): l for l in r.stdout.splitlines() if "MP2 sub-channel" in l}
    assert sorted(lines) == UEP, r.stdout
    dp = decoder(ctx, 1)
    dp.set_auto_config(0, True)
    dp.set_mp2(0, -1)
    dp.run([rec.iq])
    for sid in UEP:
        recs, pay = dp.mp2_frames(0, sid)
        assert f"{len(recs)} slots, {sum(x.status == OK for x in recs)} ok" in lines[sid]
        assert open(str(tmp_path / f"o_0.subch{sid}.mp2"), "rb").read() == pay.tobytes() and pay.size > 0
