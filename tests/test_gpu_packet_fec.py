"""-m gpu: packet-mode FEC inside the whole-path decoder (dabstar_decoder_set_packet_fec), and the stage taps dabstar_packet_fec and
dabstar_packet_groups_fec on the same device pass. FEC streams built by tests/pfec_support.py travel through the RF chain (synth
msc_payload) on the packet-mode sub-channels of test_gpu_packet_decoder's layout; every stream is compared, record for record and
byte for byte, with the taps, the host build of pfec.cuh and the plain-C restatement run on the decoder's own MSC bits."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import packet_support as ps
import pfec_support as fs
from dabstar_b200 import api, synth
from dabstar_b200._lib import DabstarError
from test_gpu_packet_decoder import LAYOUT, RATE, SUBCH

pytestmark = pytest.mark.gpu
E_INVALID, E_UNSUPPORTED = -1, -4
# one stream per packet-mode sub-channel: (sub_ch_id, scid, address, dscty, dg_flag)
PACKET = [(4, 0x101, 1, 7, 0), (5, 0x202, 17, 60, 0), (6, 0x301, 300, 44, 0), (7, 0x401, 2, 7, 0)]
STREAMS = [(s, a) for s, _, a, _, _ in PACKET]


def make_recording(n_frames, seed, fmt=synth.FMT_U8, snr_db=25.0, fig_mode=0, errors=0.0, fec_subs=(4, 5, 6, 7), fec_flags=None):
    """sub-channels in fec_subs carry FEC frames, the other packet-mode ones plain packet streams; errors: byte error rate injected
    into every packet stream before transmission. truths: per sub-channel [(group bytes, (first slot, last slot))] of the groups sent"""
    rng = np.random.default_rng(seed)
    pays, truths = [], {}
    for sid, *_, br in LAYOUT:
        addrs = [a for s, a in STREAMS if s == sid]
        if not addrs:
            pays.append(None)
            continue
        groups = {addrs[0]: ps.random_groups(rng, 4 * n_frames * br // 48 + 4, (4 * br, 12 * br))}
        if sid in fec_subs:
            _, raw, truth = fs.build_fec_stream(br, 4 * n_frames, groups, rng, lead_slots=int(rng.integers(0, 40)))
            sent = list(zip(truth["groups"][addrs[0]], truth["spans"][addrs[0]]))
        else:
            _, raw, t = ps.build_stream(br, 4 * n_frames, groups, rng)
            sent = [(g, (f0 * br // 8, (f1 + 1) * br // 8 - 1)) for f0, f1, g in t[addrs[0]]]
        raw = fs.byte_errors(raw, rng, rate=errors)
        pays.append(np.unpackbits(raw, axis=1))
        truths[sid] = sent
    rec = synth.generate(n_frames, seed=seed, snr_db=snr_db, subch=SUBCH, fmt=fmt, fig_mode=fig_mode, msc_payload=pays,
                         packet=PACKET if fig_mode else None, fec=fec_flags)
    return rec, truths


def groups_of(recs, pay):
    return [bytes(pay[r.offset:r.offset + r.length]) for r in recs]


def check_fec_stream(ctx, dp, r, sid, addr):
    """The decoder's groups, payload, counters and FEC records equal dabstar_packet_groups_fec's, the host build's and the
    restatement's on the decoder's own MSC bits."""
    bits = dp.result(r).msc[sid]
    br = RATE[sid]
    raw = np.packbits(bits, axis=1)
    got_rec, got_pay = dp.data_groups(r, sid, addr)
    tap = api.PacketProcessor(br, addr, ctx, fec=True)
    tap_rec, tap_pay = tap.add_frames(bits)
    h_rec, h_pay, h_st = fs.host_check().groups(bits, br, addr)
    o_rec, o_pay, _ = fs.oracle_groups(raw, br, addr)
    assert [ps.key(g) for g in got_rec] == [ps.key(t) for t in tap_rec] == [ps.key(h) for h in h_rec] == [ps.key(o) for o in o_rec], (r, sid)
    assert np.array_equal(got_pay, tap_pay) and np.array_equal(got_pay, h_pay) and np.array_equal(got_pay, o_pay), (r, sid)
    st = dp.packet_stats(r, sid, addr)
    assert ps.stats_key(st) == ps.stats_key(tap.stats) == ps.stats_key(h_st), (r, sid)
    frames = dp.fec_frames(r, sid)
    o_cor, _, o_frames = fs.oracle().run(raw, br)
    assert [fs.fec_key(f) for f in frames] == [fs.fec_key(f) for f in tap.fec_frames] == [fs.fec_key(f) for f in o_frames], (r, sid)
    return got_rec, got_pay, st, frames


@pytest.mark.parametrize("bit_rate", [8, 16, 24, 64, 96])
def test_tap_equals_restatement(ctx, bit_rate):
    """dabstar_packet_fec on 24 streams of each rate with random errors, bursts and junk (test_tap_long_stream spans more than one
    wave of CTAs in every FEC kernel)"""
    rng = np.random.default_rng(bit_rate)
    fec = api.PacketFec(bit_rate, ctx)
    n_frames = 60000 // bit_rate
    for k in range(24):
        _, raw, _ = fs.build_fec_stream(bit_rate, n_frames, {7: ps.random_groups(rng, 400, (0, 300))}, rng, lead_slots=int(rng.integers(0, 200)))
        bad = fs.byte_errors(raw, rng, rate=[0.0, 0.005, 0.02, 0.05][k % 4], bursts=k % 3 * 20)
        if k == 23:
            bad[: n_frames // 4] = rng.integers(0, 256, bad[: n_frames // 4].shape, np.uint8)
        cor, frames = fec.correct(np.unpackbits(bad, axis=1))
        o_cor, _, o_frames = fs.oracle().run(bad, bit_rate)
        assert np.array_equal(np.packbits(cor, axis=1), o_cor), k
        assert [fs.fec_key(f) for f in frames] == [fs.fec_key(f) for f in o_frames], k
        assert len(frames) > 0


def test_tap_long_stream(ctx):
    """One 96 kbit/s stream of 20 160 FEC frames (2.07 M slots): the per-slot kernels run 8 100 CTAs of 256 threads and
    k_pfec_correct 2 520 CTAs of 128 threads (8 frames each), more than one wave of the 148 SMs (at most 8 and 16 such CTAs per
    SM). Corrected bytes and records equal the restatement's."""
    rng = np.random.default_rng(96)
    _, base, _ = fs.build_fec_stream(96, 412, {7: ps.random_groups(rng, 300, (0, 600))}, rng)  # 48 whole FEC frames
    raw = fs.byte_errors(np.tile(base, (420, 1)), rng, rate=0.004, bursts=3000)
    cor, frames = api.PacketFec(96, ctx).correct(np.unpackbits(raw, axis=1))
    o_cor, _, o_frames = fs.oracle().run(raw, 96)
    assert len(frames) > 20000  # a burst over four or more FEC headers of a run hides it
    assert np.array_equal(np.packbits(cor, axis=1), o_cor)
    assert [fs.fec_key(f) for f in frames] == [fs.fec_key(f) for f in o_frames]
    assert sum(f.status == fs.CORRECTED for f in frames) > 10000


@pytest.mark.parametrize("fmt", [synth.FMT_U8, synth.FMT_I16])
def test_chain_explicit_selection(ctx, fmt):
    rec, truths = make_recording(40, seed=70, fmt=fmt, errors=0.01)
    dp = api.DabProcessor(1, input_format=fmt, ctx=ctx)
    dp.set_audio_channel(0, SUBCH)
    for sid, addr in STREAMS:
        dp.set_packet(0, sid, addr)
        dp.set_packet_fec(0, sid)
    dp.run([rec.iq])
    assert dp.packet_fec_ms() > 0
    for sid, addr in STREAMS:
        got_rec, got_pay, st, frames = check_fec_stream(ctx, dp, 0, sid, addr)
        got = groups_of(got_rec, got_pay)
        complete = [f for f in frames if f.status != fs.INCOMPLETE]
        assert complete and all(f.status in (fs.CLEAN, fs.CORRECTED) for f in complete), sid
        assert sum(f.status == fs.CORRECTED for f in frames) > 0
        # every group sent inside the complete frames is recovered
        sent = [g for g, (a, b) in truths[sid] if any(f.first_slot <= a and b < f.run_slot for f in complete)]
        assert sent and all(g in got for g in sent), sid
        plain_rec, plain_pay = api.PacketProcessor(RATE[sid], addr, ctx).add_frames(dp.result(0).msc[sid])
        plain = groups_of(plain_rec, plain_pay)
        if RATE[sid] >= 16:  # without FEC most are lost
            assert sum(g in plain for g in sent) < len(sent) // 2, sid


def test_low_snr_without_injected_errors(ctx):
    rec, _ = make_recording(30, seed=71, snr_db=6.2)
    dp = api.DabProcessor(1, ctx=ctx)
    dp.set_audio_channel(0, SUBCH)
    for sid, addr in STREAMS:
        dp.set_packet(0, sid, addr)
        dp.set_packet_fec(0, sid)
    dp.run([rec.iq])
    for sid, addr in STREAMS:
        got_rec, _, _, _ = check_fec_stream(ctx, dp, 0, sid, addr)
        plain_rec, _ = api.PacketProcessor(RATE[sid], addr, ctx).add_frames(dp.result(0).msc[sid])
        assert sum(r.status == ps.OK for r in got_rec) >= sum(r.status == ps.OK for r in plain_rec), sid


def test_self_configuration(ctx):
    rec, truths = make_recording(30, seed=72, fig_mode=1, errors=0.01, fec_subs=(5, 7), fec_flags=[5, 7])
    dp = api.DabProcessor(1, ctx=ctx)
    dp.set_auto_config(0, True)
    dp.set_packet(0, -1)
    dp.set_packet_fec(0, -1)
    dp.run([rec.iq])
    assert dp.fec_schemes(0) == [(5, 1), (7, 1)]
    for sid, addr in STREAMS:
        if sid in (5, 7):
            check_fec_stream(ctx, dp, 0, sid, addr)
        else:
            with pytest.raises(DabstarError):
                dp.fec_frames(0, sid)
            bits = dp.result(0).msc[sid]
            got = dp.data_groups(0, sid, addr)
            plain = api.PacketProcessor(RATE[sid], addr, ctx).add_frames(bits)
            assert [ps.key(x) for x in got[0]] == [ps.key(x) for x in plain[0]] and np.array_equal(got[1], plain[1])


def test_no_side_effects(ctx):
    rec, _ = make_recording(24, seed=73, fec_subs=(4, 5, 6))  # sub-channel 7 carries no FEC frames
    out = []
    for on in (False, True):
        dp = api.DabProcessor(1, ctx=ctx)
        dp.set_audio_channel(0, SUBCH)
        dp.set_dabplus(0, 2)
        dp.set_mp2(0, 1)
        for sid, addr in STREAMS:
            dp.set_packet(0, sid, addr)
            if on:
                dp.set_packet_fec(0, sid)
        dp.run([rec.iq])
        res = dp.result(0)
        out.append(([res.msc[s].copy() for s in sorted(res.msc)], dp.superframes(0, 2), dp.mp2_frames(0, 1),
                    {(s, a): (dp.data_groups(0, s, a), ps.stats_key(dp.packet_stats(0, s, a))) for s, a in STREAMS}))
        if on:
            assert [f.status for f in dp.fec_frames(0, 7)] == []
    (m0, d0, p0, g0), (m1, d1, p1, g1) = out
    assert all(np.array_equal(a, b) for a, b in zip(m0, m1))
    assert [bytes(x) for x in d0[0]] == [bytes(x) for x in d1[0]] and np.array_equal(d0[1], d1[1])
    assert [bytes(x) for x in p0[0]] == [bytes(x) for x in p1[0]] and np.array_equal(p0[1], p1[1])
    a, b = g0[(7, 2)], g1[(7, 2)]
    assert [ps.key(x) for x in a[0][0]] == [ps.key(x) for x in b[0][0]] and np.array_equal(a[0][1], b[0][1]) and a[1] == b[1]


def test_batch_and_segmentation(ctx):
    n_rec = 64
    uniq = [make_recording(24, seed=80 + k, errors=0.01) for k in range(3)]
    runs = []
    for seg in (False, True):
        dp = api.DabProcessor(n_rec, ctx=ctx)
        if seg:
            dp.set_segmentation(6, 18)
        for r in range(n_rec):
            dp.set_audio_channel(r, SUBCH)
            for sid, addr in STREAMS:
                dp.set_packet(r, sid, addr)
                dp.set_packet_fec(r, sid)
        dp.run([uniq[r % 3][0].iq for r in range(n_rec)])
        runs.append({(r, s): ([fs.fec_key(f) for f in dp.fec_frames(r, s)], dp.data_groups(r, s, a)) for r in range(n_rec) for s, a in STREAMS})
    for u in range(3):
        alone = api.DabProcessor(1, ctx=ctx)
        alone.set_audio_channel(0, SUBCH)
        for sid, addr in STREAMS:
            alone.set_packet(0, sid, addr)
            alone.set_packet_fec(0, sid)
        alone.run([uniq[u][0].iq])
        for sid, addr in STREAMS:
            f = [fs.fec_key(x) for x in alone.fec_frames(0, sid)]
            g = alone.data_groups(0, sid, addr)
            for run in runs:
                for r in range(u, n_rec, 3):
                    assert run[(r, sid)][0] == f
                    assert [ps.key(x) for x in run[(r, sid)][1][0]] == [ps.key(x) for x in g[0]] and np.array_equal(run[(r, sid)][1][1], g[1])


def test_level2_runs_the_pass_once_after_the_final_pass(ctx):
    """The FEC pass (four launches: fit codes, run starts, list, correct) runs once, after the final pass."""
    rec, _ = make_recording(30, seed=74, fig_mode=1, fec_flags=[4, 5, 6, 7])
    launches = {}
    for mode in ("packet", "packet_fec"):
        dp = api.DabProcessor(1, ctx=ctx)
        dp.set_auto_config(0, True, tii_null_symbols=True)
        dp.set_tii_processing(0, True)
        dp.set_packet(0, -1)
        if mode == "packet_fec":
            dp.set_packet_fec(0, -1)
        before = ctx.kernel_launches
        dp.run([rec.iq])
        launches[mode] = ctx.kernel_launches - before
    assert launches["packet_fec"] - launches["packet"] == 4, launches


def test_rejections(ctx):
    dp = api.DabProcessor(1, ctx=ctx)
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        dp.set_packet_fec(0, -1)  # needs self-configuration
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        dp.set_packet_fec(0, 64)
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        dp.set_packet_fec(0, 9)   # no such sub-channel
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        api.PacketFec(12, ctx).correct(np.zeros((2, 24 * 12), np.uint8))  # not a multiple of 8
    # every sub-channel a decoder accepts has a multiple of 8 kbit/s (EEP-A 8n, EEP-B 32n, the UEP table), so the decoder's own
    # check of an explicit FEC id's bit rate guards a layout that cannot be set
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        dp.set_audio_channel(0, [synth.SubChannel(8, 0, 9, 0, 0, 12)])
    dp.set_audio_channel(0, SUBCH)
    dp.set_packet_fec(0, 4)
    st = api.DabProcessor(1, ctx=ctx)
    st.set_audio_channel(0, SUBCH)
    st.set_streaming(True)
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_UNSUPPORTED):
        st.set_packet_fec(0, 4)
    rec, _ = make_recording(6, seed=75)
    scan = api.DabProcessor(1, scan_mode=True, ctx=ctx)
    scan.set_audio_channel(0, SUBCH)
    scan.set_packet(0, 4, 1)
    scan.set_packet_fec(0, 4)
    scan.run([rec.iq])
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        scan.fec_frames(0, 4)  # no MSC, so no FEC pass


def test_file_harness_prints_the_fec_counters(ctx, tmp_path):
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "dab_file_decode")
    subprocess.run(["g++", "-std=c++17", "-O2", os.path.join(root, "dabstar_b200", "host", "dab_file_decode.cpp"), "-I", os.path.join(root, "include"),
                    "-L", os.path.join(root, "dabstar_b200"), "-ldabstar_b200", "-Wl,-rpath," + os.path.join(root, "dabstar_b200"), "-o", exe], check=True)
    rec, _ = make_recording(30, seed=92, fig_mode=1, errors=0.01, fec_subs=(5, 7), fec_flags=[5, 7])
    path = str(tmp_path / "rec.iq")
    rec.iq.tofile(path)
    for fec in ("all", "5,7"):
        r = subprocess.run([exe, "-f", "u8", "-a", "-p", "all", "-F", fec, path], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        lines = [l for l in r.stdout.splitlines() if "FEC sub-channel" in l]
        assert len(lines) == 2, r.stdout
        dp = api.DabProcessor(1, ctx=ctx)
        dp.set_auto_config(0, True)
        dp.set_packet(0, -1)
        dp.set_packet_fec(0, -1)
        dp.run([rec.iq])
        for sid in (5, 7):
            fr = dp.fec_frames(0, sid)
            cnt = [sum(f.status == k for f in fr) for k in range(4)]
            want = (f"FEC sub-channel {sid}: {len(fr)} FEC frames, {cnt[0]} clean, {cnt[1]} corrected, {cnt[2]} partial, {cnt[3]} incomplete; "
                    f"{sum(f.rows_corrected for f in fr)} rows corrected ({sum(f.bytes_corrected for f in fr)} bytes), {sum(f.rows_failed for f in fr)} rows failed")
            assert any(l.endswith(want) for l in lines), (want, lines)
            assert cnt[1] > 0
