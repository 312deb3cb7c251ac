"""CPU part of the packet-mode pass: the host build of dabstar_b200/csrc/packet.cuh (what the device pass compiles), the plain-C
restatement tests/native/packet_oracle.c and the Python packet and data group builder, three statements written apart, against the
known answers of the standard and against each other; and FIG 0/3 in the multiplex parser and the synthetic transmitter."""
import os
import shutil

import numpy as np
import pytest

import packet_support as ps
from dabstar_b200 import api, synth
from packet_support import CRC_ERROR, MALFORMED, NO_CRC, OK, RAW

NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


@pytest.fixture(scope="module")
def host():
    if not os.path.exists(NVCC):
        pytest.skip("nvcc not available")
    return ps.host_check()


@pytest.fixture(scope="module")
def orc():
    return ps.oracle()


def agree(host, orc, bits, bit_rate, address, dg_flag=0):
    """host build == restatement: records, payload and counters; returns them"""
    a, b = host.run(bits, bit_rate, address, dg_flag), orc.run(bits, bit_rate, address, dg_flag)
    assert [ps.key(x) for x in a[0]] == [ps.key(x) for x in b[0]]
    assert np.array_equal(a[1], b[1])
    assert ps.stats_key(a[2]) == ps.stats_key(b[2])
    return a


def groups_of(recs, pay):
    return [bytes(pay[r.offset:r.offset + r.length]) for r in recs]


def test_crc_known_answer(host, orc):
    assert ps.crc16(b"123456789") == 0xD64E
    assert orc.crc(b"123456789") == 0xD64E
    assert host.crc(b"123456789") == 0xD64E


@pytest.mark.parametrize("bit_rate", [8, 16, 32, 64, 96])
def test_every_length_flag_and_address(host, orc, bit_rate):
    rng = np.random.default_rng(bit_rate)
    groups = {1: ps.random_groups(rng, 12, (0, 300)), 1023: ps.random_groups(rng, 12, (0, 300)), 77: ps.random_groups(rng, 6, (0, 40))}
    bits, _, truth = ps.build_stream(bit_rate, 240 if bit_rate < 32 else 120, groups, rng, padding=0.2, command=0.05)
    commands = 0
    for a in groups:
        recs, pay, st = agree(host, orc, bits, bit_rate, a)
        assert groups_of(recs, pay) == [g for _, _, g in truth[a]]
        assert [(r.first_frame, r.last_frame) for r in recs] == [(f0, f1) for f0, f1, _ in truth[a]]
        assert st.padding > 0 and st.other_address > 0 and st.crc_errors == st.cut == st.bad_length == 0
        commands += st.command
        assert st.abandoned == st.dropped == st.continuity_breaks == 0
        assert [r.status for r in recs] == [OK if g[0] & 0x40 else NO_CRC for _, _, g in truth[a]]
    assert commands > 0
    # every length and every first / last value occurred
    raw = np.packbits(bits, axis=1)
    seen = set()
    for f in range(raw.shape[0]):
        pos = 0
        while pos < raw.shape[1]:
            h = int(raw[f, pos])
            seen.add(("len", 24 * (1 + (h >> 6))))
            seen.add(("fl", (h >> 2) & 3))
            pos += 24 * (1 + (h >> 6))
    assert {("len", x) for x in (24, 48, 72, 96) if x <= 3 * bit_rate} <= seen
    assert {("fl", x) for x in range(4)} <= seen


def test_single_bit_flips_of_header_and_crc(host, orc):
    g = ps.data_group(b"flip", crc=True)
    for L in (24, 48, 72, 96):
        frame = ps.packet(L, 1, 3, 5, g) + b"".join(ps.packet(24, 0, 3, 0, b"") for _ in range((96 - L) // 24))
        base = np.unpackbits(np.frombuffer(frame, np.uint8)).reshape(1, -1)
        recs, _, _ = agree(host, orc, base, 32, 5)
        assert len(recs) == 1 and recs[0].status == OK
        for bit in list(range(24)) + list(range(8 * L - 16, 8 * L)):
            b = base.copy()
            b[0, bit] ^= 1
            recs, _, st = agree(host, orc, b, 32, 5)
            assert recs == [] and st.packets == 0 and st.crc_errors + st.cut >= 1, (L, bit)


def test_bad_length_and_cut_packets(host, orc):
    good = ps.packet(24, 0, 3, 9, ps.data_group(b"x"))
    bad = ps.packet(24, 1, 3, 9, b"", useful_len=20)           # 20 > 24 - 5
    frame = good + bad + ps.packet(24, 0, 3, 0, b"") + ps.packet(96, 2, 3, 9, b"abc")[:24]  # a 96-byte packet in the last 24 bytes
    bits = np.unpackbits(np.frombuffer(frame, np.uint8)).reshape(1, -1)
    recs, _, st = agree(host, orc, bits, 32, 9)
    assert len(recs) == 1 and st.bad_length == 1 and st.cut == 1 and st.padding == 1 and st.packets == 1


@pytest.mark.parametrize("bit_rate", [8, 24, 64])
def test_junk(host, orc, bit_rate):
    rng = np.random.default_rng(7 + bit_rate)
    bits = rng.integers(0, 2, (700, 24 * bit_rate), np.uint8)   # thousands of slots of junk
    for a in (1, 513, 1023):
        agree(host, orc, bits, bit_rate, a)
        agree(host, orc, bits, bit_rate, a, dg_flag=1)


def test_data_group_fields_and_sizes(host, orc):
    rng = np.random.default_rng(3)
    sizes = [1, 2, 3, 50, 91, 92, 500, 2048, 8192]
    gs = []
    for i, n in enumerate(sizes):
        kw = [{}, {"extension": 0xBEEF}, {"segment": (1, 0x1234)}, {"transport_id": 0x4242}, {"transport_id": 7, "end_user": b"\1\2\3"},
              {"end_user": b"\7"}, {"extension": 1, "segment": (0, 5), "transport_id": 9, "end_user": b"ab"}, {}, {"segment": (0, 32767)}][i]
        gs.append(ps.data_group(bytes(rng.integers(0, 256, n, np.uint8)), dg_type=i, crc=i % 3 != 1, cont=i, rep=15 - i, **kw))
    bits, _, truth = ps.build_stream(16, 400, {300: gs}, rng, padding=0.1)
    recs, pay, st = agree(host, orc, bits, 16, 300)
    assert groups_of(recs, pay) == gs and [r.n_packets > 1 for r in recs][-1]
    assert recs[-1].last_frame - recs[-1].first_frame > 20   # 8 KB at 16 kbit/s spans many logical frames
    for i, r in enumerate(recs):
        assert r.type == i and r.continuity == i and r.repetition == 15 - i and r.status == (NO_CRC if i % 3 == 1 else OK)
    assert (recs[1].extension, recs[2].segment_last, recs[2].segment_number, recs[3].transport_id, recs[3].length_indicator) == (0xBEEF, 1, 0x1234, 0x4242, 2)
    assert (recs[4].transport_id, recs[4].length_indicator, recs[5].transport_id, recs[5].length_indicator) == (7, 5, -1, 1)
    assert recs[0].extension == recs[0].segment_number == recs[0].transport_id == recs[0].length_indicator == -1
    # data field: what the builder put there
    assert bytes(pay[recs[6].offset + recs[6].data_start:][:recs[6].data_length]) == gs[6][2 + 2 + 2 + 1 + 4:-2]
    # DG flag 1: RAW records of the same bytes
    raw, rpay, _ = agree(host, orc, bits, 16, 300, dg_flag=1)
    assert [r.status for r in raw] == [RAW] * len(gs) and np.array_equal(rpay, pay)
    assert all(r.data_start == 0 and r.data_length == r.length and r.type == -1 for r in raw)


def test_malformed_and_crc_error_groups(host, orc):
    rng = np.random.default_rng(11)
    good = ps.data_group(b"hello world", crc=True, segment=(0, 1))
    broken = bytearray(good)
    broken[5] ^= 0x40
    short = [bytes([0xA0]), bytes([0xB0, 0x00, 0x0F]), bytes([0x50, 0x00, 0x11, 0x00])]  # 1 byte; ext without room; ua with tid, li 1
    bits, _, truth = ps.build_stream(32, 40, {12: [good, bytes(broken)] + short}, rng)
    recs, pay, st = agree(host, orc, bits, 32, 12)
    assert [r.status for r in recs] == [OK, CRC_ERROR, MALFORMED, MALFORMED, MALFORMED]
    assert st.groups == [1, 0, 1, 3, 0]


@pytest.mark.parametrize("seed", range(4))
def test_gaps_lost_packets_and_interleaving(host, orc, seed):
    rng = np.random.default_rng(50 + seed)
    addrs = [1, 2, 700, 1023]
    groups = {a: ps.random_groups(rng, 30, (0, 600)) for a in addrs}
    bits, _, truth = ps.build_stream(24, 300, groups, rng, padding=0.1, drop=0.03, command=0.02)
    for a in addrs:
        recs, pay, st = agree(host, orc, bits, 24, a)
        got = groups_of(recs, pay)
        sent = [g for _, _, g in truth[a]]
        assert all(g in got for g in sent)
        assert len(sent) < len(groups[a]) and st.continuity_breaks > 0 and st.abandoned + st.dropped > 0


# ---- FIG 0/3
def fib_bits(body: bytes) -> np.ndarray:
    b = body + b"\xff" + bytes(29 - len(body)) if len(body) < 30 else body
    b = b + ps.crc16(b).to_bytes(2, "big")
    return np.unpackbits(np.frombuffer(b, np.uint8))


def fig03(entries, length=None):
    body = b""
    for scid, dg, dscty, sub, addr, ca in entries:
        body += bytes([scid >> 4, ((scid & 15) << 4) | (ca is not None), (dg << 7) | dscty, (sub << 2) | (addr >> 8), addr & 255])
        if ca is not None:
            body += ca.to_bytes(2, "big")
    n = len(body) + 1 if length is None else length
    return bytes([n, 0x03]) + body


def test_fig03_entries_with_and_without_caorg():
    p = api.FibParser()
    e = [(0x123, 0, 7, 5, 1, None), (0xFFF, 1, 60, 63, 1023, 0xCAFE), (0x001, 0, 0, 0, 512, None)]
    p.process_FIB(fib_bits(fig03(e)))
    got = [(c.scid, c.dg_flag, c.dscty, c.sub_ch_id, c.packet_address, c.ca_org) for c in p.packet_components()]
    assert got == [(s, d, t, u, a, -1 if c is None else c) for s, d, t, u, a, c in e]
    p.process_FIB(fib_bits(fig03([(0x123, 1, 1, 1, 1, None)])))   # first appearance kept
    assert len(p.packet_components()) == 3 and p.packet_components()[0].sub_ch_id == 5
    assert p.sub_channels() == [] and p.components() == [] and p.ensemble() is None


def test_fig03_crossing_entry_is_abandoned():
    p = api.FibParser()
    full = fig03([(0x10, 0, 1, 2, 3, None), (0x20, 0, 1, 2, 4, 0x1111)])
    p.process_FIB(fib_bits(bytes([len(full) - 1 - 3 + 1 - 1]) + full[1:-3]))   # the second entry's CAOrg crosses the FIG end
    assert [c.scid for c in p.packet_components()] == [0x10]
    q = api.FibParser()
    q.process_FIB(fib_bits(bytes([1 + 5 + 3]) + full[1:10]))                  # second entry cut inside its 5 bytes
    assert [c.scid for c in q.packet_components()] == [0x10]


@pytest.mark.parametrize("seed", range(6))
def test_fig03_changes_no_other_list(seed):
    from test_fib_parser import _random_mci
    rng = np.random.default_rng(900 + seed)
    figs01, figs02 = _random_mci(rng, int(rng.integers(3, 12)))
    figs = [bytes([len(e) + 1, 0x01]) + e for e in figs01] + [bytes([len(e) + 1, 0x22 if pd else 0x02]) + e for pd, e in figs02]
    f03 = [fig03([(int(rng.integers(4096)), int(rng.integers(2)), int(rng.integers(64)), int(rng.integers(64)), int(rng.integers(1024)),
                   None if rng.integers(2) else int(rng.integers(65536))) for _ in range(int(rng.integers(1, 4)))]) for _ in range(8)]
    with_03 = figs + f03
    order = rng.permutation(len(with_03))
    lists = []
    for keep03 in (False, True):
        p = api.FibParser()
        cur = b""
        for k in order:
            if k >= len(figs) and not keep03:
                continue
            if len(cur) + len(with_03[k]) > 30:
                p.process_FIB(fib_bits(cur))
                cur = b""
            cur += with_03[k]
        p.process_FIB(fib_bits(cur))
        e = p.ensemble()
        lists.append((p.sub_channels(), p.components(), e.restarts if e else 0, len(p.packet_components())))
    assert lists[0][:3] == lists[1][:3] and lists[0][3] == 0 and lists[1][3] > 0


PACKET_LAYOUT = [synth.SubChannel(1, 0, 96, 1, 3, 128), synth.SubChannel(4, 96, 12, 0, 0, 8), synth.SubChannel(5, 108, 32, 0, 1, 32),
                 synth.SubChannel(9, 140, 48, 0, 0, 32)]
PACKET = [(4, 0x101, 1, 7, 0), (5, 0x202, 17, 60, 0), (5, 0x203, 1023, 5, 1), (9, 0xABC, 300, 44, 0)]


def test_synth_packet_option_parses_back():
    rec = synth.generate(2, seed=3, subch=PACKET_LAYOUT, fig_mode=1, packet=PACKET)
    p = api.FibParser()
    for f in range(2):
        p.process_FIB(rec.fib_truth[f].reshape(12, 256))
    assert [(c.sub_ch_id, c.scid, c.packet_address, c.dscty, c.dg_flag, c.ca_org) for c in p.packet_components()] == [
        (s, c, a, d, g, -1) for s, c, a, d, g in PACKET]
    comps = p.components()
    assert sorted(c.type for c in comps if c.tmid == 3) == sorted(c for _, c, _, _, _ in PACKET)
    assert [c.sub_ch_id for c in comps if c.tmid == 0] == [1]
    assert len(p.sub_channels()) == len(PACKET_LAYOUT)


def test_synth_without_the_option_is_unchanged():
    a = synth.generate(2, seed=3, subch=PACKET_LAYOUT, fig_mode=1)
    for extra in ({"packet": None}, {"packet": []}):
        b = synth.generate(2, seed=3, subch=PACKET_LAYOUT, fig_mode=1, **extra)
        assert np.array_equal(a.iq, b.iq) and np.array_equal(a.fib_truth, b.fib_truth)
    c = synth.generate(2, seed=3, subch=PACKET_LAYOUT, fig_mode=1, packet=PACKET)
    assert np.array_equal(a.msc_truth[0], c.msc_truth[0]) and not np.array_equal(a.fib_truth, c.fib_truth)
