#!/usr/bin/env python
"""Writes tests/golden/sweep_softbits.npz: time-de-interleaved soft bits of MSC logical frames for the 13 protection levels of
BASELINE.json configs[3] (EEP 1-A..4-A 72 kbit/s, 1-B..4-B 64 kbit/s, UEP 1..5 128 kbit/s), produced by the REFERENCE itself
(oracle/_ref/libdabref.so: the reference's own DabProcessor / OfdmDecoder run on a synthetic recording at 12 dB SNR), together
with the bits the reference's Protection::deconvolve + energy dispersal (Backend) gives for them. bench.py tiles these frames
for its Viterbi-only sweep ("on reference-generated soft bits"); tests/test_gpu_golden.py checks the CUDA path against the bits.

Run in the build container (needs /root/reference for oracle/_ref):  python tools/make_sweep_softbits.py
De-interleaving follows backend.cpp:131-138: tempX[i] = CIF[c - 16 + map[i & 15]][i]."""
import lzma
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from dabstar_b200 import synth  # noqa: E402
from oracle_api import Oracle   # noqa: E402

# name, short_form, prot_level, bit_rate, size_cu  (= bench.py SWEEP_PROFILES)
PROFILES = [("EEP 1-A 72k", 0, 0, 72, 108), ("EEP 2-A 72k", 0, 1, 72, 72), ("EEP 3-A 72k", 0, 2, 72, 54), ("EEP 4-A 72k", 0, 3, 72, 36),
            ("EEP 1-B 64k", 0, 4, 64, 54), ("EEP 2-B 64k", 0, 5, 64, 42), ("EEP 3-B 64k", 0, 6, 64, 36), ("EEP 4-B 64k", 0, 7, 64, 30),
            ("UEP 1 128k", 1, 1, 128, 140), ("UEP 2 128k", 1, 2, 128, 116), ("UEP 3 128k", 1, 3, 128, 96), ("UEP 4 128k", 1, 4, 128, 84),
            ("UEP 5 128k", 1, 5, 128, 64)]
MAP = np.array([0, 8, 4, 12, 2, 10, 6, 14, 1, 9, 5, 13, 3, 11, 7, 15])
N_FRAMES = 8   # 32 CIFs -> 16 complete logical frames per sub-channel
SNR_DB = 12.0


def main():
    o = Oracle("dabref")
    out = {}
    for group, seed in ((PROFILES[:10], 71), (PROFILES[10:], 72)):
        subch, cu = [], 0
        for i, (_, sf, lvl, br, size) in enumerate(group):
            subch.append(synth.SubChannel(i + 1, cu, size, sf, lvl, br))
            cu += size
        assert cu <= 864
        rec = synth.generate(N_FRAMES, seed=seed, snr_db=SNR_DB, subch=subch, fmt=synth.FMT_U8)
        res = o.chain_run(o.to_cf32(rec.iq), synth.subch_table(subch), len(subch), tap_soft=True)
        assert res.n_frames == N_FRAMES
        cifs = np.stack([res.soft_bits(f).reshape(-1)[9216:].reshape(4, 55296) for f in range(N_FRAMES)]).reshape(4 * N_FRAMES, 55296)
        for j, ((name, sf, lvl, br, size), s) in enumerate(zip(group, subch)):
            seg = cifs[:, s.start_cu * 64:(s.start_cu + s.size_cu) * 64]
            idx = np.arange(seg.shape[1])
            frames = np.stack([seg[c - 16 + MAP[idx & 15], idx] for c in range(16, 4 * N_FRAMES)])
            bits = res.msc[s.sub_ch_id]       # Backend output: rows from the 17th CIF on, energy dispersal removed
            assert bits.shape[0] == frames.shape[0], (bits.shape, frames.shape)
            assert np.array_equal(bits, rec.msc_truth[j][:bits.shape[0]]), name   # 12 dB: the reference decodes without errors
            # xz stream of little-endian int16: keeps the file under 1 MB (bench.load_sweep_softbits decodes it)
            out[f"soft_{len(out) // 2}"] = np.frombuffer(lzma.compress(frames.astype("<i2").tobytes(), preset=9 | lzma.PRESET_EXTREME), np.uint8)
            out[f"bits_{len(out) // 2}"] = np.packbits(bits, axis=1)
            print(name, frames.shape, int(np.abs(frames).max()))
    out["names"] = np.array([p[0] for p in PROFILES])
    out["profiles"] = np.array([p[1:] for p in PROFILES], np.int32)
    path = os.path.join(ROOT, "tests", "golden", "sweep_softbits.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
