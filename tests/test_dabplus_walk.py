"""CPU part of the DAB+ pass over many streams: the super-frame walk (dabstar_b200/csrc/dabplus.cuh) as the device pass drives
it, round after round, against a direct replay of Mp4Processor's synchronisation loop, that replay against the oracle's
processor, and the synthetic transmitter's caller payload (what carries real super-frames through the RF chain)."""
import hashlib
import os
import shutil
import subprocess

import numpy as np
import pytest

import helpers
from dabstar_b200 import synth
from test_dabplus import make_stream

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "dabstar_b200", "csrc")
NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def replay(n_frames, pre_ok, ok):
    """Mp4Processor::add_to_frame's synchronisation (mp4processor.cpp:95-180) over known per-window outcomes."""
    in_buf = sync = 0
    att = []
    for f in range(n_frames):
        in_buf += 1
        if in_buf < 5:
            continue
        w = f - 4
        if sync == 0:
            if pre_ok[w]:
                sync = 4
            else:
                in_buf = 4
                continue
        in_buf = 0
        att.append(w)
        if ok[w]:
            sync = 4
        else:
            sync -= 1
            if sync == 0:
                in_buf = 4
    return att


def scenario_stream(oracle, bit_rate, scenario, seed=0):
    """Logical frames of one DAB+ sub-channel: clean, byte errors, lost synchronisation (five super-frames of noise), junk
    (no super-frames), resync (a one-frame slip), too short (four frames)."""
    rng = np.random.default_rng(1000 + seed)

    def byte_errors(stream, rate):
        by = np.packbits(stream.reshape(-1))
        pos = rng.choice(by.size, max(1, int(by.size * rate)), replace=False)
        by[pos] ^= rng.integers(1, 256, pos.size, dtype=np.uint8)
        stream[:] = np.unpackbits(by).reshape(stream.shape)

    n_sf = 1 if scenario == "too_short" else 12
    stream, truth = make_stream(oracle, bit_rate, n_sf, seed=seed + bit_rate, lead=0 if scenario == "too_short" else 2)
    if scenario == "byte_errors":
        byte_errors(stream, 0.02)
    elif scenario == "lost_sync":
        stream[10:36] = rng.integers(0, 2, stream[10:36].shape, dtype=np.uint8)
    elif scenario == "junk":
        stream = rng.integers(0, 2, stream.shape, dtype=np.uint8)
    elif scenario == "resync":
        stream[12:22] = rng.integers(0, 2, stream[12:22].shape, dtype=np.uint8)
        stream = np.concatenate([stream[:40], rng.integers(0, 2, (1, 24 * bit_rate), dtype=np.uint8), stream[40:]])
    elif scenario == "too_short":
        stream = stream[:4]
    return stream, truth


SCENARIOS = ["clean", "byte_errors", "lost_sync", "junk", "resync", "too_short"]


@pytest.fixture(scope="module")
def walk_exe(tmp_path_factory):
    if not os.path.exists(NVCC):
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("native") / "dabplus_walk")
    subprocess.run([NVCC, "-O1", "-std=c++17", "-Wno-deprecated-gpu-targets", "-I", CSRC, "-o", exe, os.path.join(ROOT, "tests", "native", "dabplus_walk.cu")], check=True)
    return exe


def run_walk(exe, streams):
    text = []
    for n, pre, ok in streams:
        text.append(f"{n}\n{' '.join(map(str, pre))}\n{' '.join(map(str, ok))}\n")
    out = subprocess.run([exe], input="".join(text), capture_output=True, text=True, check=True).stdout.splitlines()
    assert len(out) == len(streams)
    res = []
    for line in out:
        v = [int(x) for x in line.split()]
        res.append((v[0], v[1], v[2:]))
    return res


def test_walk_rounds_converge_to_the_direct_replay(walk_exe):
    """Random Fire-code and repair outcomes: false Fire-code hits, runs of four (and more) failures, streams below five frames.
    Whatever the walk assumed about windows it had no outcome for, its converged attempts are the replay's."""
    rng = np.random.default_rng(7)
    streams = []
    for t in range(600):
        n = int(rng.integers(0, 8)) if t % 10 == 0 else int(rng.integers(5, 400))
        nw = max(0, n - 4)
        p_pre, p_ok = [(0.05, 0.98), (0.5, 0.5), (0.9, 0.1), (0.2, 0.95)][t % 4]
        pre = (rng.random(nw) < p_pre).astype(int)
        ok = (rng.random(nw) < p_ok).astype(int)
        if t % 3 == 0 and nw > 40:  # a run of four or more failures where the stream is in sync
            a = int(rng.integers(0, nw - 30))
            ok[a:a + int(rng.integers(16, 30))] = 0
        streams.append((n, pre, ok))
    res = run_walk(walk_exe, streams)
    extra_rounds = 0
    for (n, pre, ok), (rounds, decoded, att) in zip(streams, res):
        want = replay(n, pre, ok)
        assert att == want, (n, rounds)
        assert decoded >= len(want)
        assert rounds <= 2 + decoded  # every round but the last decodes at least one window
        if all(ok[w] for w in want):
            assert rounds <= 2  # nothing the first walk assumed was wrong: the second walk confirms it
        extra_rounds += rounds > 2
    assert extra_rounds > 50  # the loss-of-sync path was exercised


@pytest.mark.parametrize("bit_rate", [8, 32, 72, 128, 192])
@pytest.mark.parametrize("scenario", SCENARIOS)
def test_replay_matches_the_oracle_processor(oracle, bit_rate, scenario):
    """The loop the walk restates, fed with the Fire code of every window and the outcome of the attempted ones, attempts
    exactly the super-frames the oracle's Mp4Processor attempts."""
    stream, _ = scenario_stream(oracle, bit_rate, scenario)
    rec, _ = oracle.dabplus_run(stream, bit_rate)
    n = stream.shape[0]
    packed = np.packbits(stream, axis=1)
    pre = [oracle.firecode_check(packed[w:w + 5].reshape(-1)[:11]) for w in range(max(0, n - 4))]
    outcome = {r.first_frame: bool(r.ok) for r in rec}

    class Known(dict):
        def __missing__(self, w):
            raise AssertionError(f"the replay consulted window {w}, which the oracle did not attempt")
    assert replay(n, pre, Known(outcome)) == [r.first_frame for r in rec]
    if scenario == "too_short":
        assert len(rec) == 0
    if scenario == "clean":
        assert [r.first_frame for r in rec] == [2 + 5 * i for i in range(12)]


def test_synth_carries_the_caller_payload(oracle):
    sc = [synth.SubChannel(3, 100, 54, 0, 2, 72), synth.SubChannel(7, 400, 64, 1, 5, 128)]
    nf = 7
    rng = np.random.default_rng(3)
    sf = np.concatenate([helpers.dabplus_superframe(72, rng, oracle.rs_encode)[0] for _ in range(4 * nf // 5 + 1)])[:4 * nf]
    plain = synth.generate(nf, seed=3, snr_db=25.0, subch=sc, fmt=synth.FMT_U8)
    rec = synth.generate(nf, seed=3, snr_db=25.0, subch=sc, fmt=synth.FMT_U8, msc_payload=[sf, None])
    assert np.array_equal(rec.msc_truth[0], sf)
    assert np.array_equal(rec.msc_truth[1], plain.msc_truth[1])  # the other sub-channel draws what it drew without a payload
    assert np.array_equal(rec.fib_truth, plain.fib_truth)
    r = oracle.chain_run(oracle.to_cf32(rec.iq), synth.subch_table(sc), 2)
    assert np.array_equal(r.msc[3], sf[:4 * nf - 16]) and np.array_equal(r.msc[7], plain.msc_truth[1][:4 * nf - 16])
    with pytest.raises(ValueError):
        synth.generate(nf, subch=sc, msc_payload=[sf])


def test_synth_without_payload_reproduces_the_golden_input():
    g = np.load(os.path.join(ROOT, "tests", "golden", "chain.npz"))
    kw = dict(n_frames=20, seed=1, snr_db=20.0, cfo_hz=0.0, subch=[synth.SubChannel(3, 100, 54, 0, 2, 72)])  # test_oracle_golden "c1"
    a = synth.generate(fmt=synth.FMT_U8, **kw)
    b = synth.generate(fmt=synth.FMT_U8, msc_payload=[None], **kw)
    assert np.array_equal(a.iq, b.iq) and np.array_equal(a.msc_truth[0], b.msc_truth[0])
    if hashlib.sha256(b.iq.tobytes()).hexdigest() != str(g["c1_iq_sha256"]):
        pytest.skip("the synthetic transmitter does not reproduce the golden input on this libm")
