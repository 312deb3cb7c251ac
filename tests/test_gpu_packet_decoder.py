"""-m gpu: packet-mode data groups inside the whole-path decoder (dabstar_decoder_set_packet), and the stage tap dabstar_packet_groups
on the same batched device pass. Packet streams with several addresses per sub-channel and padding packets between them travel
through the RF chain (synth msc_payload) on EEP-A and EEP-B sub-channels; every stream is compared, record for record, byte for
byte and counter for counter, with the tap and the plain-C restatement run on the decoder's own MSC bits."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import packet_support as ps
from dabstar_b200 import api, synth
from dabstar_b200._lib import DabstarError

pytestmark = pytest.mark.gpu
E_INVALID, E_UNSUPPORTED = -1, -4

# (sub_ch_id, start_cu, size_cu, short_form, prot_level, bit_rate): an MP2 (UEP) and a DAB+ (EEP) sub-channel with random bits, and
# packet-mode sub-channels at 8 (1-A), 16 (3-A), 32 (2-B) and 64 kbit/s (1-B)
LAYOUT = [(1, 0, 96, 1, 3, 128), (2, 96, 48, 0, 2, 64), (4, 144, 12, 0, 0, 8), (5, 156, 12, 0, 2, 16), (6, 168, 21, 0, 5, 32), (7, 189, 54, 0, 4, 64)]
SUBCH = [synth.SubChannel(*x) for x in LAYOUT]
RATE = {x[0]: x[5] for x in LAYOUT}
# (sub_ch_id, scid, address, dscty, dg_flag)
PACKET = [(4, 0x101, 1, 7, 0), (5, 0x202, 17, 60, 0), (5, 0x203, 1023, 5, 1), (6, 0x301, 300, 44, 0), (7, 0x401, 2, 7, 0), (7, 0x402, 3, 7, 0),
          (7, 0x403, 700, 5, 1)]
STREAMS = [(s, a) for s, _, a, _, _ in PACKET]
DG = {(s, a): g for s, _, a, _, g in PACKET}


def make_recording(n_frames, seed, fmt, snr_db=25.0, fig_mode=0, drop=0.0, byte_errors=0.0):
    rng = np.random.default_rng(seed)
    pays, truths = [], {}
    for sid, *_, br in LAYOUT:
        addrs = [a for s, a in STREAMS if s == sid]
        if not addrs:
            pays.append(None)
            continue
        groups = {a: ps.random_groups(rng, 4 * n_frames * br // 64 + 4, (0, 3 * br)) for a in addrs}
        bits, _, truth = ps.build_stream(br, 4 * n_frames, groups, rng, padding=0.15, drop=drop)
        if byte_errors:
            hit = rng.random(bits.shape[0] * bits.shape[1] // 8) < byte_errors
            flat = bits.reshape(-1, 8)
            flat[hit] ^= rng.integers(0, 2, (int(hit.sum()), 8), np.uint8)
        pays.append(bits)
        truths.update({(sid, a): truth[a] for a in addrs})
    rec = synth.generate(n_frames, seed=seed, snr_db=snr_db, subch=SUBCH, fmt=fmt, fig_mode=fig_mode, msc_payload=pays,
                         packet=PACKET if fig_mode else None)
    return rec, truths


def decoder(ctx, n, fmt=synth.FMT_U8, **kw):
    return api.DabProcessor(n, input_format=fmt, ctx=ctx, **kw)


def check_stream(ctx, dp, r, sid, addr, dg_flag=0):
    """The decoder's records, payload and counters of one stream equal the tap's and the restatement's on the decoder's own bits."""
    bits = dp.result(r).msc[sid]
    got_rec, got_pay = dp.data_groups(r, sid, addr)
    want_rec, want_pay, want_st = ps.oracle().run(bits, RATE[sid], addr, dg_flag)
    tap_rec, tap_pay = api.PacketProcessor(RATE[sid], addr, ctx, dg_flag).add_frames(bits)
    assert [ps.key(g) for g in got_rec] == [ps.key(w) for w in want_rec] == [ps.key(t) for t in tap_rec], (r, sid, addr)
    assert np.array_equal(got_pay, want_pay) and np.array_equal(tap_pay, want_pay), (r, sid, addr)
    st = dp.packet_stats(r, sid, addr)
    assert ps.stats_key(st) == ps.stats_key(want_st), (r, sid, addr)
    return got_rec, got_pay, st


def selected(dp, r, sid, addr):
    try:
        dp.data_groups(r, sid, addr)
        return True
    except DabstarError:
        return False


def select_all(dp, r):
    for sid, addr in STREAMS:
        dp.set_packet(r, sid, addr)


@pytest.mark.parametrize("fmt", [synth.FMT_U8, synth.FMT_I16])
def test_chain_clean(ctx, fmt):
    recs = [make_recording(30, seed=20 + k, fmt=fmt) for k in range(2)]
    dp = decoder(ctx, 2, fmt)
    for r in range(2):
        dp.set_audio_channel(r, SUBCH)
        select_all(dp, r)
    dp.run([rec.iq for rec, _ in recs])
    assert dp.packet_ms() > 0
    for r, (rec, truths) in enumerate(recs):
        assert not selected(dp, r, 2, 1) and not selected(dp, r, 5, 1)
        for sid, addr in STREAMS:
            got_rec, got_pay, st = check_stream(ctx, dp, r, sid, addr)
            n = dp.result(r).msc[sid].shape[0]
            got = iter(bytes(got_pay[x.offset:x.offset + x.length]) for x in got_rec)
            sent = [g for f0, f1, g in truths[(sid, addr)] if f1 < n]
            assert len(sent) > 3 and all(g in got for g in sent), (r, sid, addr)  # in order
            assert st.crc_errors == 0 and st.padding > 0


@pytest.mark.parametrize("case", ["low_snr", "dropped_packets"])
def test_chain_damaged(ctx, case):
    if case == "low_snr":
        rec, _ = make_recording(30, seed=31, fmt=synth.FMT_U8, snr_db=6.2, byte_errors=0.002)
    else:
        rec, _ = make_recording(30, seed=32, fmt=synth.FMT_U8, drop=0.05)
    dp = decoder(ctx, 1)
    dp.set_audio_channel(0, SUBCH)
    select_all(dp, 0)
    dp.run([rec.iq])
    stats = [check_stream(ctx, dp, 0, sid, addr)[2] for sid, addr in STREAMS]
    assert sum(s.groups[0] for s in stats) > 0
    assert sum(s.abandoned + s.dropped for s in stats) > 0
    if case == "low_snr":
        assert sum(s.crc_errors for s in stats) > 0


def test_batch_beyond_one_wave_and_segmentation(ctx):
    """64 recordings x 7 streams: the scan (one thread per logical frame) and the compaction (one warp per group) span more than one
    wave of the 148 SMs. Every stream equals its recording decoded alone, with and without segmentation."""
    n_rec = 64
    uniq = [make_recording(24, seed=40 + k, fmt=synth.FMT_U8) for k in range(3)]
    iqs = [uniq[r % 3][0].iq for r in range(n_rec)]
    runs = []
    for seg in (False, True):
        dp = decoder(ctx, n_rec)
        if seg:
            dp.set_segmentation(6, 18)
        for r in range(n_rec):
            dp.set_audio_channel(r, SUBCH)
            select_all(dp, r)
        dp.run(iqs)
        runs.append({(r, s, a): dp.data_groups(r, s, a) for r in range(n_rec) for s, a in STREAMS})
    groups = sum(len(v[0]) for v in runs[0].values())
    assert groups > 148 * 4, groups
    for u in range(3):
        alone = decoder(ctx, 1)
        alone.set_audio_channel(0, SUBCH)
        select_all(alone, 0)
        alone.run([uniq[u][0].iq])
        for r in range(u, n_rec, 3):
            for s, a in STREAMS:
                a_rec, a_pay = alone.data_groups(0, s, a)
                for run in runs:
                    g_rec, g_pay = run[(r, s, a)]
                    assert [ps.key(x) for x in g_rec] == [ps.key(x) for x in a_rec] and np.array_equal(g_pay, a_pay), (r, s, a)


def test_self_configuration(ctx):
    rec, truths = make_recording(30, seed=51, fmt=synth.FMT_U8, fig_mode=1)
    runs = {}
    for mode in ("all", "explicit", "level2", "with_audio"):
        dp = decoder(ctx, 1)
        dp.set_auto_config(0, True, tii_null_symbols=mode == "level2")
        if mode == "level2":
            dp.set_tii_processing(0, True)
        if mode == "explicit":
            select_all(dp, 0)
        else:
            dp.set_packet(0, -1)
        if mode == "with_audio":
            dp.set_mp2(0, -1)
            dp.set_dabplus(0, -1)
        dp.run([rec.iq])
        got = sorted((s, a) for s in range(64) for a in (1, 2, 3, 17, 300, 700, 1023) if selected(dp, 0, s, a))
        assert got == sorted(STREAMS), mode
        assert [(c.sub_ch_id, c.scid, c.packet_address, c.dscty, c.dg_flag) for c in dp.packet_components(0)] == PACKET
        runs[mode] = {(s, a): check_stream(ctx, dp, 0, s, a, DG[(s, a)]) for s, a in STREAMS}
        for s, a in STREAMS:
            recs = runs[mode][(s, a)][0]
            assert len(recs) >= 3 and all((x.status == ps.RAW) == (DG[(s, a)] == 1) for x in recs)
        if mode == "with_audio":
            audio = (dp.mp2_frames(0, 1), dp.superframes(0, 2))
    for mode in ("explicit", "level2", "with_audio"):
        for k in STREAMS:
            a, b = runs[mode][k], runs["all"][k]
            assert [ps.key(x) for x in a[0]] == [ps.key(x) for x in b[0]] and np.array_equal(a[1], b[1]), (mode, k)
    alone = decoder(ctx, 1)
    alone.set_auto_config(0, True)
    alone.set_mp2(0, -1)
    alone.set_dabplus(0, -1)
    alone.run([rec.iq])
    m, d = alone.mp2_frames(0, 1), alone.superframes(0, 2)
    assert [bytes(x) for x in m[0]] == [bytes(x) for x in audio[0][0]] and np.array_equal(m[1], audio[0][1])
    assert [bytes(x) for x in d[0]] == [bytes(x) for x in audio[1][0]] and np.array_equal(d[1], audio[1][1])


def test_level2_runs_the_pass_once_after_the_final_pass(ctx):
    """At self-configuration level 2 the run decodes the recording more than once; the packet pass (three launches: scan, walk,
    compact) still runs once, after the final pass."""
    rec, _ = make_recording(30, seed=51, fmt=synth.FMT_U8, fig_mode=1)
    launches = {}
    for mode in ("level1", "level2", "level2_packet"):
        dp = decoder(ctx, 1)
        dp.set_auto_config(0, True, tii_null_symbols=mode != "level1")
        dp.set_tii_processing(0, True)
        if mode == "level2_packet":
            dp.set_packet(0, -1)
        before = ctx.kernel_launches
        dp.run([rec.iq])
        launches[mode] = ctx.kernel_launches - before
    assert launches["level2"] > launches["level1"], launches
    assert launches["level2_packet"] - launches["level2"] == 3, launches


def test_no_side_effects(ctx):
    rec, _ = make_recording(24, seed=61, fmt=synth.FMT_U8)
    out = []
    for on in (False, True):
        dp = decoder(ctx, 1)
        dp.set_audio_channel(0, SUBCH)
        dp.set_dabplus(0, 2)
        dp.set_mp2(0, 1)
        if on:
            select_all(dp, 0)
        dp.run([rec.iq])
        res = dp.result(0)
        msc = {s.sub_ch_id: res.msc[s.sub_ch_id].copy() for s in SUBCH}
        audio = ([bytes(x) for x in dp.superframes(0, 2)[0]], dp.superframes(0, 2)[1], [bytes(x) for x in dp.mp2_frames(0, 1)[0]], dp.mp2_frames(0, 1)[1])
        out.append((res.fib_bits, res.fic_valid, msc, [bytes(i) for i in res.info], res.counters, dp.fib_packed(0), audio))
    a, b = out
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[3] == b[3] and np.array_equal(a[4], b[4]) and np.array_equal(a[5], b[5])
    for sid in a[2]:
        assert np.array_equal(a[2][sid], b[2][sid])
    assert a[6][0] == b[6][0] and np.array_equal(a[6][1], b[6][1]) and a[6][2] == b[6][2] and np.array_equal(a[6][3], b[6][3])


@pytest.mark.parametrize("bit_rate", [8, 16, 32, 64, 136])
def test_tap(ctx, bit_rate):
    rng = np.random.default_rng(bit_rate)
    streams = []
    for n, sizes, drop in ((40, (0, 200), 0.0), (9, (0, 20), 0.1), (2000, (0, 3000), 0.01)):
        # the last is longer than the walk's 256 threads: chunks of many slots whose borders fall inside groups
        groups = {a: ps.random_groups(rng, max(2, n * bit_rate // 300), sizes) for a in (1, 5, 1023)}
        streams.append(ps.build_stream(bit_rate, n, groups, rng, drop=drop, command=0.01)[0])
    streams.append(rng.integers(0, 2, (300, 24 * bit_rate), np.uint8))
    host = ps.host_check()
    for s in streams:
        for a in (1, 5, 1023):
            for dg in (0, 1):
                want_rec, want_pay, _ = ps.oracle().run(s, bit_rate, a, dg)
                host_rec, host_pay, _ = host.run(s, bit_rate, a, dg)
                got_rec, got_pay = api.PacketProcessor(bit_rate, a, ctx, dg).add_frames(s)
                assert [ps.key(g) for g in got_rec] == [ps.key(w) for w in want_rec] == [ps.key(h) for h in host_rec]
                assert np.array_equal(got_pay, want_pay) and np.array_equal(host_pay, want_pay)


def test_rejections(ctx):
    dp = decoder(ctx, 1)
    dp.set_audio_channel(0, SUBCH)
    for sid, addr in ((-1, 0), (4, 0), (4, 1024), (17, 1)):  # -1 without self-configuration; addresses 0 and 1024; an unknown sub-channel
        with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
            dp.set_packet(0, sid, addr)
    for addr in (0, 1024):
        with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
            api.PacketProcessor(32, addr, ctx).add_frames(np.zeros((2, 24 * 32), np.uint8))
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        api.PacketProcessor(12, 1, ctx).add_frames(np.zeros((2, 24 * 12), np.uint8))
    rec, _ = make_recording(6, seed=81, fmt=synth.FMT_U8)
    st = decoder(ctx, 1)
    st.set_audio_channel(0, SUBCH)
    st.set_packet(0, 4, 1)
    st.set_streaming(True)
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_UNSUPPORTED):
        st.run([rec.iq])
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_UNSUPPORTED):
        st.set_packet(0, 5, 17)
    ok = decoder(ctx, 1)
    ok.set_audio_channel(0, SUBCH)
    ok.set_packet(0, 4, 1)
    ok.run([rec.iq])
    ok.data_groups(0, 4, 1)
    for sid, addr in ((4, 2), (5, 17)):  # not selected
        with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
            ok.data_groups(0, sid, addr)
        with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
            ok.packet_stats(0, sid, addr)
    scan = decoder(ctx, 1, scan_mode=True)
    scan.set_audio_channel(0, SUBCH)
    scan.set_packet(0, 4, 1)
    scan.run([rec.iq])
    with pytest.raises(DabstarError, match=r"\(%d\)" % E_INVALID):
        scan.data_groups(0, 4, 1)  # no MSC, so no groups


def test_file_harness_writes_the_groups(ctx, tmp_path):
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "dab_file_decode")
    subprocess.run(["g++", "-std=c++17", "-O2", os.path.join(root, "dabstar_b200", "host", "dab_file_decode.cpp"), "-I", os.path.join(root, "include"),
                    "-L", os.path.join(root, "dabstar_b200"), "-ldabstar_b200", "-Wl,-rpath," + os.path.join(root, "dabstar_b200"), "-o", exe], check=True)
    rec, _ = make_recording(24, seed=91, fmt=synth.FMT_U8, fig_mode=1)
    path = str(tmp_path / "rec.iq")
    rec.iq.tofile(path)
    r = subprocess.run([exe, "-f", "u8", "-a", "-p", "all", "-o", str(tmp_path / "o_"), path], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if "packet sub-channel" in l]
    assert len(lines) == len(STREAMS), r.stdout
    dp = decoder(ctx, 1)
    dp.set_auto_config(0, True)
    dp.set_packet(0, -1)
    dp.run([rec.iq])
    for sid, addr in STREAMS:
        recs, pay = dp.data_groups(0, sid, addr)
        assert any(f"sub-channel {sid} address {addr}: {len(recs)} groups" in l for l in lines)
        assert open(str(tmp_path / f"o_0.subch{sid}.addr{addr}.dg"), "rb").read() == pay.tobytes() and pay.size > 0
