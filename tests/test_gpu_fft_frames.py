"""The chain's frame FFT (`k_fft_frames`, and `k_fft_null` for the TII input) against a float64 model of the FrameDesc contract.

The kernel converts u8 / i16 / cf32 samples, strips the cyclic prefix, applies the integer-Hz oscillator, transforms and
scatters the carriers into the demapper's pair layout, all in one launch. The demapper downstream is differential, so an error
that is the same in consecutive symbols (a one-sample shift of every data row, an oscillator one sample off, a stale phasor)
cancels there; these tests look at the spectra themselves.

The model (float64): samples are `oracle.to_cf32` of the recording, zero outside it; sample i of a symbol read from phase ph is
multiplied by exp(j 2 pi ((ph - f (i + 1)) mod FS) / FS) with the modulo in exact integers (sample_reader.cpp:276-281); row 0
reads at sym0 with ph = ph_eval - f_sym0 (sym0 - eval), data row r at sym0 + T_U + T_G + (r - 1) T_S, the null row at
sym0 + T_U + 75 T_S + T_G; the transform is numpy's FFT; carrier k sits at bin map_k_to_fft_bin(k) (negative bins + 2048).
The unmarked tests anchor the model to the oracle chain's own FFT rows; the gpu tests hold the kernel to it.
"""
import numpy as np
import pytest

from dabstar_b200 import api, synth

FS, T_U, T_G, T_S = 2048000, 2048, 504, 2552
ROWS = 77
FMTS = {"u8": api.FMT_U8, "i16": api.FMT_I16, "cf32": api.FMT_CF32}
BAR = 1e-5  # max |got - model| <= BAR * max |model| per row: the bar test_cuda_fft_against_numpy holds k_fft_batch to


def frame(rec, sym0, eval_=None, f=(0, 0, 0), ph=(0, 0, 0), n_syms=75):
    return dict(sym0=int(sym0), eval=int(sym0 if eval_ is None else eval_), rec=int(rec), f_sym0=int(f[0]), ph_eval=int(ph[0]),
                f_data=int(f[1]), ph_data=int(ph[1]), f_null=int(f[2]), ph_null=int(ph[2]), n_syms=int(n_syms))


def row_params(d):
    """(start, f, phase before `start`) of rows 0..76 of descriptor d, from the FrameDesc contract (common.cuh)."""
    out = [(d["sym0"], d["f_sym0"], (d["ph_eval"] - d["f_sym0"] * (d["sym0"] - d["eval"])) % FS)]
    for r in range(1, 76):
        lead = T_G + (r - 1) * T_S  # samples read since the start of symbol 1's cyclic prefix
        out.append((d["sym0"] + T_U + lead, d["f_data"], (d["ph_data"] - d["f_data"] * lead) % FS))
    out.append((d["sym0"] + T_U + 75 * T_S + T_G, d["f_null"], (d["ph_null"] - d["f_null"] * T_G) % FS))
    return out


def segments(x, params):
    """The 2048 samples of each (start, f, ph) as read, zero outside x, before derotation: complex128[len(params), 2048]."""
    idx = np.array([p[0] for p in params], np.int64)[:, None] + np.arange(T_U)
    inside = (idx >= 0) & (idx < x.size)
    v = np.zeros(idx.shape, np.complex128)
    v[inside] = x[idx[inside]]
    return v


def model_rows(x, d, rows=range(ROWS)):
    """Natural-order float64 spectra of the listed rows of descriptor d over converted samples x."""
    return model_spectra(x, [row_params(d)[r] for r in rows])


def model_spectra(x, params):
    """Natural-order float64 spectra of the symbols (start, f, ph)."""
    i1 = np.arange(1, T_U + 1, dtype=np.int64)
    k = np.stack([(ph - f * i1) % FS for _, f, ph in params])  # exact integers
    return np.fft.fft(segments(x, params) * np.exp(2j * np.pi * k / FS), axis=1)


def carrier_bins(oracle):
    b = oracle.freq_interleaver().astype(np.int64)
    return np.where(b < 0, b + 2048, b)


def rel_err(got, want):
    return np.abs(got - want).max(axis=-1) / np.abs(want).max(axis=-1)


# ------------------------------------------------------------------------------------------------ CPU anchors
def test_model_reproduces_oracle_chain_rows_without_offset(oracle):
    rec = synth.generate(5, seed=2, snr_db=20.0, fmt=synth.FMT_U8)
    x = oracle.to_cf32(rec.iq).astype(np.complex128)
    r = oracle.chain_run(oracle.to_cf32(rec.iq), scan_mode=1, tap_fft=True)
    assert r.n_frames == 5
    for i, fi in enumerate(r.info):
        assert (round(fi.fbb_sym0), round(fi.fbb_data), round(fi.fbb_null)) == (0, 0, 0)  # the oscillator never moves
        got = r.fft(i).astype(np.complex128)
        want = model_rows(x, frame(0, fi.sym0_pos))
        e = rel_err(got, want)
        assert e.max() <= 1e-6, (i, int(e.argmax()), e.max())


def test_model_reproduces_oracle_chain_rows_with_offset(oracle):
    """2400 Hz: one common phase per row (the chain's oscillator phase is not reported) and its row-to-row step."""
    rec = synth.generate(6, seed=3, snr_db=20.0, cfo_hz=2400.0, fmt=synth.FMT_I16)
    x = oracle.to_cf32(rec.iq).astype(np.complex128)
    r = oracle.chain_run(oracle.to_cf32(rec.iq), scan_mode=1, tap_fft=True)
    used = 0
    for i, fi in enumerate(r.info):
        fbb = (fi.fbb_sym0, fi.fbb_data, fi.fbb_null)
        if any(abs(v - round(v)) > 0.25 for v in fbb):
            continue
        f = tuple(int(round(v)) for v in fbb)
        assert f[1] != 0
        used += 1
        got = r.fft(i).astype(np.complex128)
        want = model_spectra(x, [(start, fr, 0) for start, fr, _ in row_params(frame(0, fi.sym0_pos, f=f))])  # each row from phase 0
        c = np.einsum("rk,rk->r", got, want.conj())
        c /= np.abs(c)
        e = rel_err(got, c[:, None] * want)
        assert e.max() <= 1e-6, (i, int(e.argmax()), e.max())
        step = np.angle(c[2:76] * c[1:75].conj())
        expect = np.angle(np.exp(-2j * np.pi * f[1] * T_S / FS))
        assert np.abs(np.angle(np.exp(1j * (step - expect)))).max() <= 1e-6, (i, step[:3], expect)
        # the opposite sign of the oscillator is far off: the anchor can tell them apart
        flipped = model_spectra(x, [(row_params(frame(0, fi.sym0_pos))[1][0], -f[1], 0)])
        c1 = np.vdot(flipped[0], got[1])
        assert rel_err(got[1], c1 / abs(c1) * flipped[0]) > 1e-2
    assert used >= 2


# ------------------------------------------------------------------------------------------------ GPU: the descriptor sets
LENGTHS = (260_003, 231_518, 199_999)  # end to end: recordings 1 and 2 start 3 and 1 samples (mod 8) past an aligned address
FULL = T_U + 75 * T_S + T_G + T_U      # sym0 .. end of the null row's FFT window


def make_recordings(fmt, rng):
    recs = []
    for n in LENGTHS:
        if fmt == api.FMT_U8:
            a = rng.integers(0, 256, (n, 2), dtype=np.uint8)
            a[:4] = [[0, 255], [255, 0], [0, 0], [255, 255]]
            a[n // 2:n // 2 + 2] = [[0, 255], [255, 0]]
        elif fmt == api.FMT_I16:
            a = rng.integers(-32768, 32768, (n, 2), dtype=np.int64).astype(np.int16)
            a[:4] = [[-32768, 32767], [32767, -32768], [-32767, -32768], [32767, 32767]]
            a[n // 2:n // 2 + 2] = [[-32768, -32768], [32767, -32767]]
        else:
            a = (rng.normal(0.0, 0.5, n) + 1j * rng.normal(0.0, 0.5, n)).astype(np.complex64)
            a[:4] = [1.0 - 1.0j, -1.0 + 0.0j, 3.5 + 2.0j, -0.0 - 3.0j]
        recs.append(a)
    return recs


def make_frames(rng):
    """About 150 descriptors over the three recordings: the hand-made edge cases below, then random frames. Descriptors overlap
    in sample range; X is the large buffer."""
    n = LENGTHS
    fr = []
    # every sym0 mod 8 (every 16-byte offset class in every format), f = 0 and ph = 0 (bit identity with dabstar_fft2048)
    for rec in range(3):
        fr += [frame(rec, 1000 * (rec + 1) + k) for k in range(8)]
    # the bounds-checked path at the start of a recording, with an oscillator
    fr += [frame(k % 3, k, f=(2400, -2400, 1), ph=(FS - 1, 12345, 7)) for k in range(8)]
    # the async / bounds-checked border at the end: start + T_U + 8 == n (async) and == n + 1 (checked), for row 0, a data row, the null row
    for rec, extra in ((0, 0), (1, 1), (2, 0), (2, 1)):
        end = n[rec] + extra
        fr.append(frame(rec, end - 8 - T_U, f=(-34000, 0, 0), ph=(5, 0, 0), n_syms=0))
        fr.append(frame(rec, end - 8 - 2 * T_U - T_G - 39 * T_S, f=(0, 2400, 0), ph=(0, FS - 2, 0), n_syms=40))
        fr.append(frame(rec, end - 8 - T_U - (T_U + 75 * T_S + T_G), f=(1, -1, 34000), ph=(3, 4, FS - 1)))
    # rows cut by the end and rows entirely past it (exact zeros), f = 0 and f != 0
    fr.append(frame(0, n[0] - 100_000 + 3, f=(0, 2400, -2400), ph=(0, 99, 1_000_000)))
    fr.append(frame(1, n[1] - 150_001, f=(0, 0, 0), ph=(0, 0, 0)))
    fr.append(frame(2, n[2] + 5, f=(34000, -34000, 2), ph=(1, 2, 3)))
    fr.append(frame(2, n[2] - 2048 - 3, f=(0, 0, 0), ph=(0, 777, 0)))
    # f = 0 with a different phase in consecutive frames (and inside a frame: row 0, the data rows and the null row differ)
    for k in range(6):
        fr.append(frame(k % 3, 20_000 + 1111 * k, f=(0, 0, 0), ph=(311 * k + 1, 500_000 + 77_777 * k, FS - 1 - k)))
    # n_syms 0, 1, 37, 74, 75 at one frequency in consecutive frames, then the same frequency alternating with 0
    for k, ns in enumerate((0, 1, 37, 74, 75)):
        fr.append(frame(k % 3, 30_000 + 517 * k, f=(2400, 2400, 2400), ph=(1000 * k, 2000 * k, 3000 * k), n_syms=ns))
    for k in range(8):
        fv = -2400 if k % 2 == 0 else 0
        fr.append(frame(k % 3, 40_000 + 333 * k, f=(fv, fv, fv), ph=(0, 0, 0) if fv == 0 and k % 4 == 1 else (17 * k, 1 + k, 2 * k)))
    # every frequency of the list, f_sym0 != f_data != f_null, phases near FS - 1, eval far before and after sym0
    for k, fv in enumerate((1, -1, 2400, -2400, 34000, -34000)):
        fr.append(frame(k % 3, 50_000 + 7 * k, eval_=50_000 + 7 * k - 300_001 + 2 * k, f=(fv, -fv // 2 or 3, 2 * fv), ph=(FS - 1, FS - 2, FS - 1 - k)))
        fr.append(frame(k % 3, 51_000 + 5 * k, eval_=51_000 + 5 * k + 412_345, f=(-fv, fv, 0), ph=(FS - 3, k, FS - 1)))
    # the rest at random: any frequency of the list or an arbitrary one, random phases, mostly whole frames
    freqs = (0, 1, -1, 2, 2400, -2400, 34000, -34000, 117, -5003)
    while len(fr) < 150:
        rec = int(rng.integers(0, 3))
        sym0 = int(rng.integers(0, n[rec] - FULL + 30_000))
        f = tuple(int(v) for v in rng.choice(freqs, 3))
        ph = tuple(int(v) for v in rng.integers(0, FS, 3))
        ns = int(rng.choice([75, 75, 75, 0, 1, 37, 74, int(rng.integers(0, 76))]))
        fr.append(frame(rec, sym0, eval_=sym0 + int(rng.integers(-400_000, 400_000)), f=f, ph=ph, n_syms=ns))
    return fr


def written_rows(d):
    return list(range(d["n_syms"] + 1)) + ([ROWS - 1] if d["n_syms"] == 75 else [])


_CACHE = {}


def run_set(ctx, oracle, name):
    """Recordings, descriptors, X at the launcher's shape (with the null FFT) and at one CTA per SM, and the model."""
    if name in _CACHE:
        return _CACHE[name]
    fmt = FMTS[name]
    rng = np.random.default_rng(100 + fmt)
    recs = make_recordings(fmt, rng)
    frames = make_frames(rng)
    n_x = len(frames) + 17
    slots = rng.permutation(n_x)[:len(frames)]  # a permutation of descriptor order with unused slots between
    for d, s in zip(frames, slots):
        d["xslot"] = int(s)
    X0, null = api.fft_frames(recs, fmt, frames, n_x, 0, with_null=True, ctx=ctx)
    X1, _ = api.fft_frames(recs, fmt, frames, n_x, 1, ctx=ctx)
    xs = [oracle.to_cf32(r).astype(np.complex128) for r in recs]
    model = [model_rows(xs[d["rec"]], d) for d in frames]
    out = dict(fmt=fmt, recs=recs, xs=xs, frames=frames, n_x=n_x, X0=X0, X1=X1, null=null, model=model)
    _CACHE[name] = out
    return out


def test_descriptor_sets_cover_the_edges():
    """The hand-made part of the set reaches every case it is meant to (host arithmetic only)."""
    fr = make_frames(np.random.default_rng(0))
    async_offsets, ends, first = set(), set(), set()
    for d in fr:
        n = LENGTHS[d["rec"]]
        for r in written_rows(d):
            s = row_params(d)[r][0]
            if 8 <= s and s + T_U + 8 <= n:
                async_offsets.add((s + sum(LENGTHS[:d["rec"]])) % 8)  # sample offset from the buffer's aligned base
            first.add(s) if s < 8 else None
            ends.add(s + T_U + 8 - n)
    assert async_offsets == set(range(8)) and {d["sym0"] % 8 for d in fr} == set(range(8))
    assert set(range(8)) <= first
    assert {0, 1} <= ends and any(-T_U - 8 < e < 8 for e in ends - {0, 1})  # async border, checked border, a cut row
    assert max(ends) >= T_U + 8  # a row entirely past the end
    assert {0, 1, 37, 74, 75} <= {d["n_syms"] for d in fr}
    fs = {v for d in fr for v in (d["f_sym0"], d["f_data"], d["f_null"])}
    assert {0, 1, -1, 2400, -2400, 34000, -34000} <= fs
    assert any(d["f_sym0"] != d["f_data"] != d["f_null"] != d["f_sym0"] for d in fr)
    assert any(d["eval"] - d["sym0"] < -300_000 for d in fr) and any(d["eval"] - d["sym0"] > 400_000 for d in fr)
    assert any(FS - 3 <= d["ph_eval"] for d in fr) and 140 <= len(fr) <= 160


# ------------------------------------------------------------------------------------------------ GPU: assertions
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FMTS))
def test_rows_match_float64_model(ctx, oracle, name, record_property):
    s = run_set(ctx, oracle, name)
    bins = carrier_bins(oracle)
    worst, zeros = 0.0, 0
    for d, m in zip(s["frames"], s["model"]):
        for r in written_rows(d):
            got = s["X0"][d["xslot"], r].astype(np.complex128)
            want = m[r, bins]
            scale = np.abs(want).max()
            if scale == 0.0:  # every sample outside the recording
                assert np.all(got == 0), (d, r)
                zeros += 1
                continue
            e = np.abs(got - want).max() / scale
            assert e <= BAR, (d, r, e)
            worst = max(worst, e)
    assert zeros > 0
    record_property(f"fft_frames_max_rel_err_{name}", float(worst))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FMTS))
def test_unwritten_rows_keep_the_fill(ctx, oracle, name):
    s = run_set(ctx, oracle, name)
    bits = s["X0"].view(np.uint32).reshape(s["n_x"], ROWS, -1)
    written = np.zeros((s["n_x"], ROWS), bool)
    for d in s["frames"]:
        written[d["xslot"], written_rows(d)] = True
    assert (~written).sum() > 17 * ROWS  # unused slots plus short frames
    assert np.all(bits[~written] == 0xFFFFFFFF)
    assert not np.any(np.all(bits[written] == 0xFFFFFFFF, axis=1))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FMTS))
def test_rows_without_oscillator_equal_fft2048_bit_for_bit(ctx, oracle, name):
    """f = 0, ph = 0: no derotation, so the row is dabstar_fft2048 of the converted samples, selected at the carriers' bins."""
    s = run_set(ctx, oracle, name)
    bins = carrier_bins(oracle)
    segs, got = [], []
    for d in s["frames"]:
        params = row_params(d)
        plain = [r for r in written_rows(d) if params[r][1] == 0 and params[r][2] == 0]
        if plain:
            segs.append(segments(oracle.to_cf32(s["recs"][d["rec"]]), [params[r] for r in plain]).astype(np.complex64))
            got.append(s["X0"][d["xslot"], plain])
    segs, got = np.concatenate(segs), np.concatenate(got)
    assert segs.shape[0] > 24 * 76
    want = np.ascontiguousarray(ctx.fft2048(segs, -1)[:, bins])
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), int((got.view(np.uint32) != want.view(np.uint32)).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FMTS))
def test_launch_shapes_are_bit_identical(ctx, oracle, name):
    """One CTA per SM (148 CTAs walking ~80 items across frame borders) and one-frame calls (one item per CTA) give the same bits."""
    s = run_set(ctx, oracle, name)
    assert np.array_equal(s["X0"].view(np.uint32), s["X1"].view(np.uint32))
    for i in (8 * 3 + 1, 60, len(s["frames"]) - 1, 37):
        d = dict(s["frames"][i], xslot=0)
        X, _ = api.fft_frames(s["recs"], s["fmt"], [d], 1, 0, ctx=ctx)
        rows = written_rows(d)
        assert np.array_equal(X[0, rows].view(np.uint32), s["X0"][s["frames"][i]["xslot"], rows].view(np.uint32)), i


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FMTS))
def test_null_fft_matches_model_and_row_76(ctx, oracle, name):
    s = run_set(ctx, oracle, name)
    bins = carrier_bins(oracle)
    full = 0
    for f, (d, m) in enumerate(zip(s["frames"], s["model"])):
        got, want = s["null"][f].astype(np.complex128), m[ROWS - 1]
        scale = np.abs(want).max()
        if scale == 0.0:
            assert np.all(got == 0), d
        else:
            assert np.abs(got - want).max() <= BAR * scale, (d, np.abs(got - want).max() / scale)
        if d["n_syms"] == 75:
            full += 1
            a, b = np.ascontiguousarray(s["null"][f, bins]).view(np.uint32), s["X0"][d["xslot"], ROWS - 1].view(np.uint32)
            diff = np.flatnonzero(a != b)
            assert diff.size == 0, (d, [(hex(a[i]), hex(b[i])) for i in diff[:4]], diff.size)
    assert full > 50


@pytest.mark.gpu
def test_rejects_invalid_arguments_before_launching(ctx):
    rec = [np.zeros((T_U * 3, 2), np.uint8)]
    good = frame(0, 10)
    good["xslot"] = 1
    X, _ = api.fft_frames(rec, api.FMT_U8, [good], 2, 0, ctx=ctx)  # the valid call goes through
    assert np.all(X[0].view(np.uint32) == 0xFFFFFFFF) and not np.all(X[1, 0].view(np.uint32) == 0xFFFFFFFF)
    bad = [dict(good, xslot=2), dict(good, xslot=-1), dict(good, rec=1), dict(good, rec=-1), dict(good, n_syms=76), dict(good, n_syms=-1),
           dict(good, f_data=FS), dict(good, f_null=-FS)]
    before = ctx.kernel_launches
    for d in bad:
        with pytest.raises(api.DabstarError):
            api.fft_frames(rec, api.FMT_U8, [d], 2, 0, ctx=ctx)
    with pytest.raises(api.DabstarError):
        api.fft_frames(rec, 3, [good], 2, 0, ctx=ctx)
    with pytest.raises(api.DabstarError):
        api.fft_frames(rec, -1, [good], 2, 0, ctx=ctx)
    with pytest.raises(api.DabstarError):
        api.fft_frames(rec, api.FMT_U8, [good], 2, -1, ctx=ctx)
    # negative counts straight through the C ABI (the wrapper cannot express them)
    buf = np.ascontiguousarray(rec[0])
    fr = (api._lib.FftFrameC * 1)(api._lib.FftFrameC(**good))
    out = np.empty(2 * ROWS * 1536 * 2, np.float32)
    lib, p = ctx.lib, api._ptr
    for n_rec, n_fr, n_x, recn in ((-1, 1, 2, T_U * 3), (1, -1, 2, T_U * 3), (1, 1, -1, T_U * 3), (1, 1, 2, -5)):
        cnt = np.array([recn], np.int64)
        assert lib.dabstar_fft_frames(ctx.h, p(buf), api.FMT_U8, p(cnt), n_rec, fr, n_fr, n_x, 0, p(out), None, api.MEM_HOST) == -1
    assert ctx.kernel_launches == before
