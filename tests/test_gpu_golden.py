"""-m gpu: the CUDA path against the golden vectors the UNMODIFIED reference produced (tests/golden/*.npz, tools/make_golden.py)
directly - one hop from the reference instead of two (CUDA -> C restatement -> reference) - and, where oracle/_ref travelled
to the box, against the reference's own objects (`refo`)."""
import hashlib
import os

import numpy as np
import pytest

import helpers
from dabstar_b200 import api, synth
from test_oracle_golden import CASES, ETI_CASE, load

pytestmark = pytest.mark.gpu


def test_viterbi_known_answers_cuda(ctx, viterbi_path):
    g = load("viterbi.npz")
    for key in g.files:
        if not key.startswith("soft_"):
            continue
        n_bits = int(key.split("_")[1])
        want = np.unpackbits(g["bits" + key[4:]], axis=1)[:, :n_bits]
        got = api.ViterbiSpiral(n_bits, ctx).deconvolve(g[key])
        assert np.array_equal(got.reshape(want.shape), want), key


def test_protection_and_backend_cuda(ctx, viterbi_path):
    g = load("msc.npz")
    for sf, lvl, br, cu in helpers.ALL_PROFILES:
        want = np.unpackbits(g[f"prot_out_{sf}_{lvl}_{br}"])[:24 * br]
        soft = g[f"prot_in_{sf}_{lvl}_{br}"]
        got = api.Protection(sf, br, lvl, ctx).deconvolve(soft.reshape(1, -1), cu)
        assert np.array_equal(got.reshape(-1), want), (sf, lvl, br)
    cifs = np.zeros((19, 55296), np.int16)
    cifs[:, 11 * 64:(11 + 54) * 64] = g["backend_frag_i8"]
    out = api.Backend(synth.SubChannel(1, 11, 54, 0, 2, 72), ctx).process(cifs)
    assert int(g["backend_first"]) == 16 and out.shape[0] == 3
    assert np.array_equal(out, np.unpackbits(g["backend_out"], axis=1)[:, :1728])


def test_sweep_soft_bits_of_the_reference_cuda(ctx, viterbi_path):
    """configs[3]'s input: the reference's own soft bits per protection level (tests/golden/sweep_softbits.npz: OfdmDecoder output
    of oracle/_ref at 12 dB, time de-interleaved; tools/make_sweep_softbits.py). Protection::deconvolve on the GPU gives the
    reference's Backend output once the energy dispersal is put back; a tiled batch of 2 400 frames takes the
    thread-per-code-word path with its device-written job list, the 16 frames alone the warp-per-code-word kernel."""
    import bench
    g = bench.load_sweep_softbits()
    assert [tuple(int(x) for x in row) for row in g["profiles"]] == [p[1:] for p in bench.SWEEP_PROFILES]
    for li, (name, sf, lvl, br, cu) in enumerate(bench.SWEEP_PROFILES):
        soft = g[f"soft_{li}"]
        want = np.unpackbits(g[f"bits_{li}"], axis=1)[:, :24 * br] ^ bench.prbs_bits(24 * br)[None, :]
        assert soft.shape == (16, cu * 64) and want.shape == (16, 24 * br)
        prot = api.Protection(sf, br, lvl, ctx)
        assert np.array_equal(prot.deconvolve(soft, cu).reshape(want.shape), want), name
        big = prot.deconvolve(np.tile(soft, (150, 1)), cu).reshape(150, 16, 24 * br)
        assert np.array_equal(big, np.broadcast_to(want, big.shape)), name


def test_tables_cuda(ctx):
    g = load("tables.npz")
    fi = api.FreqInterleaver(ctx)
    assert np.array_equal([fi.map_k_to_fft_bin(k) for k in range(1536)], g["freq_interleaver"])
    for key in g.files:
        if key.startswith("addr_"):
            sf, lvl, br = map(int, key.split("_")[1:])
            try:
                got = api.Protection(sf, br, lvl, ctx).addresses()
            except api.DabstarError:
                assert (sf, br) == (1, 320)  # UEP 320 kbit/s level 1 overflows the reference's i16 bookkeeping: fenced off (DESIGN.md)
                continue
            assert np.array_equal(got, g[key]), key


@pytest.mark.parametrize("name", list(CASES))
def test_chain_against_reference_run_cuda(ctx, name):
    g = load("chain.npz")
    kw = CASES[name]
    rec = synth.generate(fmt=synth.FMT_U8, **kw)
    if hashlib.sha256(rec.iq.tobytes()).hexdigest() != str(g[f"{name}_iq_sha256"]):
        pytest.skip("the synthetic transmitter does not reproduce the golden input on this libm")
    dp = api.DabProcessor(1, input_format=synth.FMT_U8, ctx=ctx)
    dp.set_audio_channel(0, kw["subch"])
    dp.run([rec.iq])
    r = dp.result(0)
    assert r.n_frames == int(g[f"{name}_n_frames"])
    assert np.array_equal([i.sym0_pos for i in r.info], g[f"{name}_sym0_pos"])
    assert np.array_equal([i.start_index for i in r.info], g[f"{name}_start_index"])
    fbb = np.array([[i.fbb_sym0, i.fbb_data, i.fbb_null, i.fsync, i.phase_cp, i.clock_err] for i in r.info], np.float32)
    assert np.allclose(fbb, g[f"{name}_fbb"], atol=5e-2)
    assert np.array_equal(np.round(fbb[:, :3]), np.round(g[f"{name}_fbb"][:, :3]))  # integer-Hz derotation identical
    assert np.array_equal([[i.fic_ratio_before, i.fic_ratio_after] for i in r.info], g[f"{name}_ratio"])
    assert np.array_equal(r.fic_valid, g[f"{name}_fic_valid"])
    ok = r.fic_valid.astype(bool).repeat(768, axis=1)
    assert np.array_equal(r.fib_bits[ok], np.unpackbits(g[f"{name}_fib"], axis=1)[ok])
    assert r.n_good_fibs == int(g[f"{name}_good_fibs"])
    for s in kw["subch"]:
        want = np.unpackbits(g[f"{name}_msc_{s.sub_ch_id}"], axis=1)[:, :24 * s.bit_rate]
        assert np.array_equal(r.msc[s.sub_ch_id], want), s
    # level 2: soft bits within +-1 LSB of the REFERENCE's for >= 99.99 %
    for f, key in ((0, "soft_f0"), (2, "soft_f2")):
        d = np.abs(dp.soft_bits(0, f)[:3].astype(np.int32) - g[f"{name}_{key}"].astype(np.int32))
        assert (d > 1).mean() <= 1e-4, (key, d.max())
    # level 1: FFT bins within 1e-4 relative of the reference's (frames derotated by 0 Hz only: the tap transforms raw samples)
    if round(r.info[1].fbb_sym0) == 0 and round(r.info[1].fbb_data) == 0 and kw["cfo_hz"] == 0.0:
        x = ((rec.iq.astype(np.float32) - np.float32(127.38)) / np.float32(128.0)).view(np.complex64).reshape(-1)
        s0 = int(r.info[1].sym0_pos)
        rows = np.stack([x[s0:s0 + 2048], x[s0 + 2048 + 504:s0 + 2048 + 2552], x[s0 + 2048 + 75 * 2552 + 504:s0 + 2048 + 75 * 2552 + 2552]])
        fft = ctx.fft2048(rows)
        ref = g[f"{name}_fft_f1"]
        # the reference's samples carry the oscillator's constant phasor (0 Hz, but a phase left over from the acquisition)
        rot = np.array([np.vdot(a, b) for a, b in zip(fft, ref)])
        fft = fft * (rot / np.abs(rot))[:, None]
        assert np.abs(fft - ref).max() / np.abs(ref).max() < 1e-4


def test_eti_stream_against_reference_run_cuda(ctx):
    g = load("eti.npz")
    rec = synth.generate(fmt=synth.FMT_U8, **ETI_CASE)
    if hashlib.sha256(rec.iq.tobytes()).hexdigest() != str(g["iq_sha256"]):
        pytest.skip("the synthetic transmitter does not reproduce the golden input on this libm")
    dp = api.DabProcessor(1, input_format=synth.FMT_U8, ctx=ctx)
    dp.set_audio_channel(0, ETI_CASE["subch"])
    dp.start_eti_generator(0)
    dp.run([rec.iq])
    assert dp.result(0).n_frames == int(g["n_frames"]) == 9
    assert np.array_equal(dp.eti(0), g["eti"])


def test_cp_correlation_stage_tap(ctx):
    """k_cp_corr against the expression of dab_processor.cpp:326-333 evaluated in double."""
    rng = np.random.default_rng(5)
    n, per = 5, 75 * 2552
    x = (rng.standard_normal((n, per)) + 1j * rng.standard_normal((n, per))).astype(np.complex64) * 0.2
    for f in range(n):  # a cyclic prefix with a frequency offset: x[i + 2048] = x[i] e^{j phi}
        v = x[f].reshape(75, 2552)
        v[:, 2048:] = v[:, :504] * np.exp(1j * (0.1 * f - 0.2))
    got = api.cp_correlate(x, ctx)
    v = x.reshape(n, 75, 2552).astype(np.complex128)
    want = (v[:, :, 2048:] * np.conj(v[:, :, :504])).sum(axis=(1, 2))
    assert np.allclose(got, want, rtol=2e-5, atol=1e-3)
    assert np.allclose(np.angle(got), 0.1 * np.arange(n) - 0.2, atol=1e-4)
    assert api.cp_correlate(np.zeros((0, per), np.complex64), ctx).shape == (0,)


def test_cp_correlation_by_bulk_copy_equals_direct_loads(ctx, monkeypatch):
    """8-bit input: k_cp_corr_bulk (TMA copies into a ring in shared memory) and k_cp_corr (direct loads) add the same products
    in the same order, so the whole decode (frame positions, every soft bit, FIBs) is identical; the recordings start at odd
    sample offsets so that the 16-byte aligned copies see every alignment, and one ends inside a frame."""
    recs = []
    for i in range(6):
        r = synth.generate(5, seed=300 + i, snr_db=11.0 + i, cfo_hz=-2300.0 + 900.0 * i, fmt=synth.FMT_U8)
        iq = r.iq[3 + i:]  # (n, 2) samples: a different 16-byte alignment of the frame start in every recording
        recs.append(np.ascontiguousarray(iq[:len(iq) - (50000 if i == 5 else 0)]))
    out = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("DABSTAR_CP_BULK", mode)
        dp = api.DabProcessor(len(recs), input_format=synth.FMT_U8, ctx=ctx)
        dp.run(recs)
        out[mode] = [(dp.n_frames(r), dp.frame_positions(r).copy(), dp.fib_packed(r).copy(),
                      np.stack([dp.soft_bits(r, f) for f in range(dp.n_frames(r))]) if dp.n_frames(r) else None) for r in range(len(recs))]
    assert sum(o[0] for o in out["1"]) >= 20
    for a, b in zip(out["0"], out["1"]):
        assert a[0] == b[0]
        assert np.array_equal(a[1], b[1])
        assert np.array_equal(a[2], b[2])
        assert (a[3] is None and b[3] is None) or np.array_equal(a[3], b[3])


# ---- the reference's own objects on the GPU box (oracle/_ref/libdabref.so ships with the snapshot when it was built)
def test_chain_against_the_reference_itself(ctx, refo):
    sc = [synth.SubChannel(3, 100, 54, 0, 2, 72)]
    rec = synth.generate(16, seed=61, snr_db=13.0, cfo_hz=-800.0, subch=sc, fmt=synth.FMT_U8)
    want = refo.chain_run(refo.to_cf32(rec.iq), synth.subch_table(sc), 1, tap_soft=True)
    dp = api.DabProcessor(1, input_format=synth.FMT_U8, ctx=ctx)
    dp.set_audio_channel(0, sc)
    dp.run([rec.iq])
    got = dp.result(0)
    assert got.n_frames == want.n_frames
    assert [(i.sym0_pos, i.start_index, round(i.fbb_data)) for i in got.info] == [(i.sym0_pos, i.start_index, round(i.fbb_data)) for i in want.info]
    assert np.array_equal(got.fic_valid, want.fic_valid)
    ok = want.fic_valid.astype(bool).repeat(768, axis=1)
    assert np.array_equal(got.fib_bits[ok], want.fib_bits[ok])
    assert np.array_equal(got.msc[3], want.msc[3])
    for f in (0, got.n_frames - 1):
        d = np.abs(dp.soft_bits(0, f).astype(np.int32) - want.soft_bits(f).astype(np.int32))
        assert (d > 1).mean() <= 1e-4, (f, d.max())


def test_viterbi_against_the_reference_itself(ctx, refo, viterbi_path):
    for n_bits in (768, 1728, 3072):
        _, soft = helpers.random_codewords(64, n_bits, 45.0, seed=n_bits)
        want = np.stack([refo.viterbi(s, n_bits) for s in soft])
        got = api.ViterbiSpiral(n_bits, ctx).deconvolve(soft)
        assert np.array_equal(got.reshape(want.shape), want), n_bits
