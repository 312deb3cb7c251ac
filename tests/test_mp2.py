"""CPU part of the MPEG layer II (MP2) frame check: the host build of dabstar_b200/csrc/mp2.cuh (what the device pass compiles),
the plain-C oracle tests/native/mp2_oracle.c and the Python frame builder, three statements written apart, against the known
answers of the standards and against each other, slot for slot."""
import os
import shutil

import numpy as np
import pytest

import mp2_support as ms
from mp2_support import CRC_ERROR, CUT, MISMATCH, NO_HEADER, OK

NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


@pytest.fixture(scope="module")
def exe():
    if not os.path.exists(NVCC):
        pytest.skip("nvcc not available")
    return ms.host_driver()


@pytest.fixture(scope="module")
def orc():
    return ms.oracle()


def frame_bits(bits):
    return np.ascontiguousarray(bits, np.uint8).reshape(-1)


def test_known_answers(exe, orc):
    check = b"123456789"
    assert ms.crc16(ms.bytes_to_bits(check)) == 0xAEE7
    assert orc.crc16(check) == 0xAEE7
    assert int(ms.host_command(exe, f"crc {check.hex()}\n")[0]) == 0xAEE7
    # allocation bits per channel: Table B.2a (sblimit 27), B.2c (8), 13818-3 B.1 (30); and joint stereo with bound 4
    host = [int(x) for x in ms.host_command(exe, "alloc 0 1 27\nalloc 1 1 8\nalloc 2 1 30\nalloc 0 2 4\n")]
    assert host == [88, 26, 75, 104]
    assert [orc.alloc_bits(48, 128, 3, 0), orc.alloc_bits(48, 32, 3, 0), orc.alloc_bits(24, 64, 3, 0), orc.alloc_bits(48, 128, 1, 0)] == [88, 26, 75, 104]
    assert [ms.alloc_bits(48000, 128, 3, 0), ms.alloc_bits(48000, 32, 3, 0), ms.alloc_bits(24000, 64, 3, 0), ms.alloc_bits(48000, 128, 1, 0)] == [88, 26, 75, 104]


def builder_frames():
    rng = np.random.default_rng(11)
    out = []
    for sr, rates in ((48000, ms.RATES_MPEG1), (24000, ms.RATES_LSF)):
        for br in rates:
            for mode in range(4):
                for ext in range(4):
                    out.append((sr, br, mode, ext, ms.mp2_frame(br, rng, sr, mode, ext)))
    return out


def test_builder_frames_classify_ok(exe, orc):
    """Every rate of both tables at every mode / mode_extension: one OK record covering the whole frame, in the oracle and in the
    host build of mp2.cuh, with the frame's bytes as payload."""
    frames = builder_frames()
    host = ms.host_run(exe, [(f, br) for _, br, _, _, f in frames])
    for (sr, br, mode, ext, f), (h_rec, h_pay) in zip(frames, host):
        o_rec, o_pay = orc.run(f, br)
        want = np.packbits(frame_bits(f)).tobytes()
        assert [ms.key(r) for r in o_rec] == h_rec, (sr, br, mode, ext)
        assert len(o_rec) == 1 and o_rec[0].status == OK and o_rec[0].n_frames == (2 if sr == 24000 else 1), (sr, br, mode, ext)
        assert o_rec[0].crc_stored == o_rec[0].crc_computed == int(ms.bytes_to_bits(want[4:6]).dot(1 << np.arange(15, -1, -1)))
        assert o_pay.tobytes() == want and h_pay == want


@pytest.mark.parametrize("sr,br,mode,ext", [(48000, 128, 1, 0), (48000, 384, 0, 0), (48000, 32, 3, 0), (48000, 64, 2, 0), (24000, 64, 1, 2),
                                            (24000, 8, 3, 0), (24000, 160, 0, 0)])
def test_single_bit_flips(exe, orc, sr, br, mode, ext):
    """A flip in the syncword, layer or protection bit is NO_HEADER; in ID, bitrate_index or sampling_frequency a MISMATCH; in the
    CRC-covered header bits 22..31, the allocation or the SCFSI a CRC_ERROR; in crc_check itself a CRC_ERROR; after the SCFSI the
    frame stays OK."""
    rng = np.random.default_rng(br * 10 + mode)
    f, (a0, a1, s1) = ms.mp2_frame(br, rng, sr, mode, ext, layout=True)
    flat = frame_bits(f)
    positions = list(range(0, s1 + 40))
    streams, want = [], []
    for p in positions:
        g = flat.copy()
        g[p] ^= 1
        streams.append((g.reshape(f.shape), br))
        if p < 12 or p in (13, 14, 15):
            want.append(NO_HEADER)
        elif p == 12 or 16 <= p < 22:
            want.append(MISMATCH)
        elif p < s1:
            want.append(CRC_ERROR)
        else:
            want.append(OK)
    host = ms.host_run(exe, streams)
    for p, (g, _), w, (h_rec, _) in zip(positions, streams, want, host):
        o_rec, _ = orc.run(g, br)
        assert [ms.key(r) for r in o_rec] == h_rec, p
        assert o_rec[0].status == w, (p, o_rec[0].status, w)
    assert a0 == 48 and a1 - a0 == ms.alloc_bits(sr, br, mode, ext)


SCENARIOS = {
    "junk": dict(junk=range(0, 10 ** 6)),
    "byte_errors": dict(byte_errors=0.004),
    "lsf_odd_start": dict(sample_rate=24000, lead=1),
    "lsf_odd_start_3": dict(sample_rate=24000, lead=3),
    "slip": dict(slip=7),
    "lsf_slip": dict(sample_rate=24000, slip=5),
    "lsf_damaged_header": dict(sample_rate=24000, damage_header=(2, 9, 10)),
    "damaged_header": dict(damage_header=(1, 4)),
    "mixed": dict(mixed=True),
    "mixed_errors": dict(mixed=True, byte_errors=0.002, lead=2),
}


def scenario(name, br, n, seed):
    return ms.mp2_stream(br, n, np.random.default_rng(seed), **SCENARIOS[name])


@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_host_equals_oracle_slot_for_slot(exe, orc, name):
    """Thousands of slots per scenario at rates of both tables; odd stream lengths end 24 kHz streams inside a frame (CUT)."""
    streams = []
    for k, br in enumerate([32, 48, 56, 64, 80, 96, 112, 128, 160, 8, 16, 24, 40, 144, 192, 384]):
        if name.startswith("lsf") and br not in ms.RATES_LSF:
            continue
        for n in (1, 2, 23, 40 + k):
            streams.append((scenario(name, br, n, seed=1000 * k + n)[0], br))
    host = ms.host_run(exe, streams)
    slots = 0
    for (bits, br), (h_rec, h_pay) in zip(streams, host):
        o_rec, o_pay = orc.run(bits, br)
        assert [ms.key(r) for r in o_rec] == h_rec, (name, br, bits.shape[0])
        assert o_pay.tobytes() == h_pay
        assert sum(r.n_frames for r in o_rec) == bits.shape[0]
        slots += len(o_rec)
    assert slots > 400


def test_walk_semantics(orc, exe):
    """The records a clean stream gives: every frame found with its bytes; a damaged 24 kHz header loses exactly that slot and
    finds the next frame two logical frames on; a 24 kHz stream ending inside a frame ends with CUT."""
    rng = np.random.default_rng(5)
    bits, truth = ms.mp2_stream(64, 22, rng, sample_rate=24000, lead=1)
    rec, pay = orc.run(bits, 64)
    assert rec[0].status != OK and rec[0].first_frame == 0
    oks = [r for r in rec if r.status == OK]
    assert [r.first_frame for r in oks] == sorted(truth) == list(range(1, 20, 2))
    assert (rec[-1].first_frame, rec[-1].n_frames, rec[-1].status) == (21, 1, CUT)
    assert pay.tobytes() == b"".join(np.packbits(frame_bits(truth[f])).tobytes() for f in sorted(truth))
    bits, truth = ms.mp2_stream(64, 20, np.random.default_rng(6), sample_rate=24000, damage_header=(3,))
    rec, _ = orc.run(bits, 64)
    firsts = [(r.first_frame, r.n_frames, r.status) for r in rec]
    assert (6, 1, NO_HEADER) in firsts or (6, 1, MISMATCH) in firsts or (6, 1, CRC_ERROR) in firsts
    assert (7, 1, OK) not in firsts and (8, 2, OK) in firsts
    h_rec, _ = ms.host_run(exe, [(bits, 64)])[0]
    assert h_rec == [ms.key(r) for r in rec]
