"""CPU part of packet-mode FEC: the host build of dabstar_b200/csrc/pfec.cuh (what the device pass compiles), the plain-C restatement
tests/native/pfec_oracle.c and the Python RS(204,188) encoder and FEC frame builder, three statements written apart; FIG 0/14 in the
multiplex parser and the synthetic transmitter."""
import os
import shutil

import numpy as np
import pytest

import packet_support as ps
import pfec_support as fs
from dabstar_b200 import api, synth

NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


@pytest.fixture(scope="module")
def host():
    if not os.path.exists(NVCC):
        pytest.skip("nvcc not available")
    return fs.host_check()


@pytest.fixture(scope="module")
def orc():
    return fs.oracle()


def agree(host, orc, raw, bit_rate):
    a, b = host.run(raw, bit_rate), orc.run(raw, bit_rate)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert [fs.fec_key(x) for x in a[2]] == [fs.fec_key(x) for x in b[2]]
    return a


# ---- FIG 0/14
def fib(figs: list[bytes]) -> np.ndarray:
    body = b"".join(figs)
    body = body + b"\xff" + bytes(30 - len(body) - 1) if len(body) < 30 else body
    crc = ps.crc16(body)
    return np.unpackbits(np.frombuffer(body + crc.to_bytes(2, "big"), np.uint8))


def fig0(ext: int, data: bytes, cn: int = 0) -> bytes:
    return bytes([(0 << 5) | (1 + len(data)), (cn << 7) | ext]) + data


def test_fig0_14_schemes_and_edges():
    p = api.FibParser()
    e = lambda sid, sch: bytes([(sid << 2) | sch])
    p.process_FIB(fib([fig0(14, e(3, 0) + e(4, 1) + e(5, 2) + e(6, 3)), fig0(14, e(7, 1), cn=1)]))  # C/N 1 ignored
    p.process_FIB(fib([fig0(14, e(4, 0) + e(8, 1))]))  # SubChId 4 already known: first appearance kept
    assert p.fec_schemes() == [(3, 0), (4, 1), (5, 2), (6, 3), (8, 1)]
    assert p.sub_channels() == [] and p.components() == [] and p.packet_components() == [] and p.ensemble() is None


def test_fig0_14_entries_past_the_fig_end_are_not_read():
    p = api.FibParser()
    # FIG length 2: one entry; the byte after it belongs to no FIG 0/14 and a FIG without entries reads none
    p.process_FIB(fib([bytes([(0 << 5) | 2, 14, (9 << 2) | 1, (10 << 2) | 1])]))
    p.process_FIB(fib([bytes([(0 << 5) | 1, 14])]))
    assert p.fec_schemes() == [(9, 1)]


def test_fig0_14_changes_no_other_list():
    sub = [synth.SubChannel(1, 0, 12, 0, 0, 8), synth.SubChannel(2, 12, 12, 0, 0, 8)]
    rec = synth.generate(1, seed=3, subch=sub, fig_mode=1, packet=[(1, 0x101, 5, 7, 0)], lead_samples=100, tail_samples=100)
    p, q = api.FibParser(), api.FibParser()
    fibs = rec.fib_truth.reshape(-1, 256)
    p.process_FIB(fibs)
    q.process_FIB(fibs)
    q.process_FIB(fib([fig0(14, bytes([(1 << 2) | 1, (2 << 2) | 3]))]))
    q.process_FIB(fibs)
    assert q.fec_schemes() == [(1, 1), (2, 3)] and p.fec_schemes() == []
    assert q.sub_channels() == p.sub_channels() and q.components() == p.components() and q.packet_components() == p.packet_components()
    assert q.ensemble().restarts == p.ensemble().restarts


def test_transmitter_fig0_14_and_byte_identity():
    sub = [synth.SubChannel(1, 0, 12, 0, 0, 8), synth.SubChannel(2, 12, 12, 0, 0, 8)]
    packet = [(1, 0x101, 5, 7, 0), (2, 0x102, 6, 7, 0)]
    a = synth.generate(2, seed=3, subch=sub, fig_mode=1, packet=packet, lead_samples=100, tail_samples=100)
    b = synth.generate(2, seed=3, subch=sub, fig_mode=1, packet=packet, lead_samples=100, tail_samples=100, fec=None)
    assert np.array_equal(a.iq, b.iq) and np.array_equal(a.fib_truth, b.fib_truth)
    c = synth.generate(2, seed=3, subch=sub, fig_mode=1, packet=packet, lead_samples=100, tail_samples=100, fec=[2])
    p = api.FibParser()
    p.process_FIB(c.fib_truth.reshape(-1, 256))
    assert p.fec_schemes() == [(2, 1)]
    assert [x.sub_ch_id for x in p.packet_components()] == [1, 2]


# ---- RS(204,188)
def code_word(rng) -> bytes:
    info = bytes(rng.integers(0, 256, 188, np.uint8))
    return info + fs.rs_encode(info)


def test_encoder_words_have_zero_syndromes(host, orc):
    rng = np.random.default_rng(1)
    for _ in range(50):
        cw = code_word(rng)
        assert orc.decode(cw) == (0, cw) and host.decode(cw) == (0, cw)


@pytest.mark.parametrize("n_err", range(9))
def test_up_to_eight_errors_corrected(host, orc, n_err):
    rng = np.random.default_rng(100 + n_err)
    for t in range(40):
        cw = code_word(rng)
        # the first information byte, the last parity byte, eight errors at the start of the row, or random positions
        forced = [0] if t == 0 else [203] if t == 1 else list(range(8)) if t == 2 else []
        pos = (forced + [int(x) for x in rng.permutation(np.arange(8, 203))])[:n_err]
        bad = bytearray(cw)
        for p in pos:
            bad[p] ^= int(rng.integers(1, 256))
        assert orc.decode(bytes(bad)) == (n_err, cw)
        assert host.decode(bytes(bad)) == (n_err, cw)


@pytest.mark.parametrize("n_err", range(9, 17))
def test_beyond_eight_errors_same_outcome(host, orc, n_err):
    rng = np.random.default_rng(200 + n_err)
    for _ in range(40):
        bad = bytearray(code_word(rng))
        for p in rng.choice(204, n_err, replace=False):
            bad[p] ^= int(rng.integers(1, 256))
        assert orc.decode(bytes(bad)) == host.decode(bytes(bad))


# ---- locate
@pytest.mark.parametrize("bit_rate", [8, 16, 24, 64, 96])
def test_frames_at_every_slot_offset(host, orc, bit_rate):
    rng = np.random.default_rng(bit_rate)
    spf = bit_rate // 8
    for lead in range(0, spf + 1) if spf > 1 else range(2):
        n_frames = (103 * 3 + 94 + lead) // spf + 2
        groups = {9: ps.random_groups(rng, 30, (0, 150))}
        _, raw, truth = fs.build_fec_stream(bit_rate, n_frames, groups, rng, lead_slots=94 + lead)
        cor, mask, recs = agree(host, orc, raw, bit_rate)
        n = n_frames * spf
        assert [r.run_slot for r in recs] == [s for s in truth["runs"] if min(s + 9, n) - s >= 6]
        for r in recs:
            assert r.status == (fs.CLEAN if r.run_slot + 9 <= n else fs.INCOMPLETE)
            assert r.first_slot == r.run_slot - 94 and r.headers_matched == min(9, n - r.run_slot)
        assert np.array_equal(cor, raw)


@pytest.mark.parametrize("n_damaged", range(4))
def test_damaged_fec_headers(host, orc, n_damaged):
    rng = np.random.default_rng(40 + n_damaged)
    bit_rate, n_frames = 16, 600
    _, raw, truth = fs.build_fec_stream(bit_rate, n_frames, {3: ps.random_groups(rng, 100, (0, 200))}, rng, lead_slots=5)
    bad = raw.copy().reshape(-1, 24)
    found_expected = []
    for s in truth["runs"]:
        if s + 9 > n_frames * 2:
            continue
        while True:  # three damaged headers: not the first, the last and one beside them (pfec.cuh)
            hit = sorted(rng.choice(9, n_damaged, replace=False))
            if not (n_damaged == 3 and 0 in hit and 8 in hit and (1 in hit or 7 in hit)):
                break
        for k in hit:
            bad[s + k, 1] ^= 0x40  # the address is no longer 1022
        found_expected.append(s)
    bad = bad.reshape(raw.shape)
    cor, mask, recs = agree(host, orc, bad, bit_rate)
    assert [r.run_slot for r in recs if r.run_slot + 9 <= n_frames * 2] == found_expected
    assert all(r.headers_matched == 9 - n_damaged for r in recs if r.run_slot + 9 <= n_frames * 2)
    # the headers are not covered by the code: only they differ from what was sent
    assert np.array_equal(cor, bad)


def test_below_threshold_not_found(host, orc):
    rng = np.random.default_rng(7)
    _, raw, truth = fs.build_fec_stream(16, 400, {3: ps.random_groups(rng, 40, (0, 200))}, rng, lead_slots=0)
    bad = raw.copy().reshape(-1, 24)
    s = truth["runs"][1]
    for k in (1, 3, 5, 7):  # four damaged: 5 of 9 fit
        bad[s + k, 0] ^= 0xC0
    _, _, recs = agree(host, orc, bad.reshape(raw.shape), 16)
    runs = [r.run_slot for r in recs]
    assert s not in runs and truth["runs"][0] in runs and truth["runs"][2] in runs
    nxt = [r for r in recs if r.run_slot == truth["runs"][2]][0]
    assert nxt.status == fs.CLEAN  # the previous run it knows is two frames back


def test_cut_by_stream_start_and_end_and_close_runs(host, orc):
    rng = np.random.default_rng(8)
    bit_rate, n_frames = 32, 200
    _, raw, truth = fs.build_fec_stream(bit_rate, n_frames, {3: ps.random_groups(rng, 60, (0, 200))}, rng, lead_slots=0)
    # cut the stream 40 slots into it: the first frame has fewer than 94 slots before its run
    cut = raw.reshape(-1, 24)[40 - 40 % 4:].reshape(-1, 3 * bit_rate)
    _, _, recs = agree(host, orc, cut, bit_rate)
    assert recs[0].status == fs.INCOMPLETE and recs[0].first_slot < 0 and all(r.status == fs.CLEAN for r in recs[1:-1])
    # a copy of a run 50 slots after a real one: the second lies inside the next ADT, the real next one is overlapped by it
    bad = raw.copy().reshape(-1, 24)
    s = truth["runs"][2]
    bad[s + 50:s + 59] = bad[s:s + 9]
    _, _, recs = agree(host, orc, bad.reshape(raw.shape), bit_rate)
    by = {r.run_slot: r for r in recs}
    assert by[s].status in (fs.CLEAN, fs.CORRECTED, fs.PARTIAL) and by[s + 50].status == fs.INCOMPLETE and by[truth["runs"][3]].status == fs.INCOMPLETE


def test_junk_and_stray_headers(host, orc):
    rng = np.random.default_rng(9)
    junk = rng.integers(0, 256, (300, 48), np.uint8)
    junk.reshape(-1, 24)[::7, :2] = [0x03, 0xFE]  # stray address-1022 headers, flags 00
    agree(host, orc, junk, 16)
    bits, raw, _ = ps.build_stream(16, 300, {1022: ps.random_groups(rng, 40, (0, 100))}, rng)
    _, _, recs = agree(host, orc, raw, 16)
    assert recs == []  # ordinary packets with address 1022 never fit a 9-packet run's flags


# ---- end to end
@pytest.mark.parametrize("case", ["random", "bursts"])
def test_end_to_end_groups_recovered(host, orc, case):
    rng = np.random.default_rng(11 if case == "random" else 12)
    bit_rate, n_frames = 32, 600
    groups = {5: ps.random_groups(rng, 150, (0, 300)), 600: ps.random_groups(rng, 60, (0, 100))}
    _, raw, truth = fs.build_fec_stream(bit_rate, n_frames, groups, rng, lead_slots=0)
    if case == "random":
        bad = fs.byte_errors(raw, rng, rate=0.01)
    else:  # one burst of up to 96 bytes in every FEC frame
        bad = raw.copy().reshape(-1)
        for s in truth["runs"]:
            ln = int(rng.integers(1, 97))
            at = (s - 94) * 24 + int(rng.integers(0, 103 * 24 - ln))
            bad[at:at + ln] ^= rng.integers(1, 256, ln, np.uint8)
        bad = bad[:raw.size].reshape(raw.shape)
    cor, mask, recs = agree(host, orc, bad, bit_rate)
    complete = [r for r in recs if r.status != fs.INCOMPLETE]
    assert complete and all(r.status in (fs.CLEAN, fs.CORRECTED) for r in complete)
    bits = np.unpackbits(bad, axis=1)
    for a, gs in groups.items():
        sent = truth["groups"][a]
        got_rec, got_pay, st = host.groups(bits, bit_rate, a)
        o_rec, o_pay, _ = fs.oracle_groups(bad, bit_rate, a)
        assert [ps.key(x) for x in got_rec] == [ps.key(x) for x in o_rec] and np.array_equal(got_pay, o_pay)
        got = [bytes(got_pay[r.offset:r.offset + r.length]) for r in got_rec]
        # every group sent inside the complete frames (all but the one the stream's end cuts) is recovered
        inside = [g for g, (s0, s1) in zip(sent, truth["spans"][a]) if complete[0].first_slot <= s0 and s1 < complete[-1].run_slot]
        assert len(inside) >= len(sent) - 3 and all(g in got for g in inside), a
        p_rec, p_pay, _ = ps.oracle().run(bits, bit_rate, a)
        plain = [bytes(p_pay[r.offset:r.offset + r.length]) for r in p_rec]
        if case == "random" and a == 5:
            assert sum(g in plain for g in inside) < len(inside) // 2
