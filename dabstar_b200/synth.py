"""ctypes front end of the bundled synthetic Mode-I transmitter (dabstar_b200/synth/dab_synth.c)."""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field

import numpy as np

from . import build

T_FRAME = 196608
FMT_CF32, FMT_U8, FMT_I16 = 0, 1, 2


@dataclass
class SubChannel:
    """One MSC sub-channel, the fields of the reference's SDescriptorType (dab_constants.h:119-135)."""
    sub_ch_id: int
    start_cu: int
    size_cu: int
    short_form: int      # 1 = UEP (prot_level 1..5), 0 = EEP (prot_level 0..3 = 1-A..4-A, 4..7 = 1-B..4-B)
    prot_level: int
    bit_rate: int
    start_frame: int = 0  # frame in which the receiver's Backend is created

    def as_row(self) -> list[int]:
        return [self.sub_ch_id, self.start_cu, self.size_cu, self.short_form, self.prot_level, self.bit_rate, self.start_frame]


def subch_table(subch: list[SubChannel]) -> np.ndarray:
    t = np.zeros((max(len(subch), 1), 7), np.int32)
    for i, s in enumerate(subch):
        t[i] = s.as_row()
    return t


class _Cfg(ctypes.Structure):
    _fields_ = [("n_frames", ctypes.c_int32), ("format", ctypes.c_int32), ("seed", ctypes.c_uint64),
                ("snr_db", ctypes.c_float), ("cfo_hz", ctypes.c_float), ("rms", ctypes.c_float),
                ("lead_samples", ctypes.c_int32), ("tail_samples", ctypes.c_int32), ("n_subch", ctypes.c_int32),
                ("subch", ctypes.c_void_p), ("fig_mode", ctypes.c_int32), ("eid", ctypes.c_int32), ("tii_main", ctypes.c_int32), ("tii_sub", ctypes.c_int32),
                ("msc_payload", ctypes.c_void_p), ("n_packet", ctypes.c_int32), ("packet", ctypes.c_void_p),
                ("n_fec", ctypes.c_int32), ("fec", ctypes.c_void_p)]


@dataclass
class Recording:
    iq: np.ndarray                 # cf32: complex64[n]; u8: uint8[n,2]; i16: int16[n,2]
    fmt: int
    fib_truth: np.ndarray          # uint8[n_frames, 3072], one bit per byte
    msc_truth: list[np.ndarray] = field(default_factory=list)  # per sub-channel uint8[n_cifs, 24*bitRate]
    subch: list[SubChannel] = field(default_factory=list)


_lib = None


def _load():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build.build_synth())
        _lib.dabsynth_num_samples.restype = ctypes.c_int64
        _lib.dabsynth_num_samples.argtypes = [ctypes.c_void_p]
        _lib.dabsynth_generate.restype = ctypes.c_int
        _lib.dabsynth_generate.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    return _lib


def generate(n_frames: int, seed: int = 1, snr_db: float = 20.0, cfo_hz: float = 0.0, subch: list[SubChannel] | None = None,
             fmt: int = FMT_U8, rms: float = 0.25, lead_samples: int = 60000, tail_samples: int = 4096, out: np.ndarray | None = None,
             fig_mode: int = 0, eid: int = 0x1234, tii: tuple[int, int] | None = None, msc_payload: list | None = None,
             packet: list | None = None, fec: list | None = None) -> Recording:
    """Synthesise `n_frames` Mode-I transmission frames. `lead_samples` of noise-like filler precede the first
    null symbol (the reference spends 40 960 samples on its level estimate before it searches the null).
    fig_mode 1: the FIC carries the ensemble's multiplex configuration (FIG 0/0 with a running CIF counter, FIG 0/1, FIG 0/2)
    instead of random FIB payloads. tii = (main id, sub id): with fig_mode 1 the null symbol after every frame whose CIF counter has
    (count & 7) >= 4 carries that transmitter identification.
    msc_payload: per sub-channel None (random bits) or the logical frames it carries, uint8[4 * n_frames, 24 * bit_rate] bits
    (e.g. DAB+ super-frames from tests/helpers.dabplus_superframe); the other sub-channels draw what they draw without it.
    packet: with fig_mode 1, [(sub_ch_id, scid, address, dscty, dg_flag), ...]: each listed sub-channel carries no programme service;
    each entry becomes a data service with one packet-mode (TMId 3) component in FIG 0/2 and a FIG 0/3 entry. Without it every
    output is what it is without the argument.
    fec: with fig_mode 1, [sub_ch_id, ...]: each is sent as a FIG 0/14 entry with FEC scheme 1 (packet-mode FEC); the payload itself
    is whatever msc_payload carries. Without it every output is what it is without the argument."""
    lib = _load()
    subch = subch or []
    tab = subch_table(subch)
    keep, pay = [], None
    if msc_payload is not None:
        if len(msc_payload) != len(subch):
            raise ValueError("msc_payload: one entry per sub-channel")
        for p, s in zip(msc_payload, subch):
            keep.append(None if p is None else np.ascontiguousarray(p, np.uint8).reshape(4 * n_frames, 24 * s.bit_rate))
        pay = (ctypes.c_void_p * max(len(subch), 1))(*[None if k is None else k.ctypes.data for k in keep])
    ptab = np.ascontiguousarray(np.array(packet or [], np.int32).reshape(-1, 5))
    ftab = np.ascontiguousarray(np.array(fec or [], np.int32).reshape(-1))
    cfg = _Cfg(n_frames, fmt, seed, snr_db, cfo_hz, rms, lead_samples, tail_samples, len(subch), tab.ctypes.data, fig_mode, eid, tii[0] if tii else -1, tii[1] if tii else -1,
               ctypes.cast(pay, ctypes.c_void_p) if pay is not None else None, len(ptab), ptab.ctypes.data if len(ptab) else None,
               len(ftab), ftab.ctypes.data if len(ftab) else None)
    n = lib.dabsynth_num_samples(ctypes.byref(cfg))
    if out is None:
        out = np.empty(n, np.complex64) if fmt == FMT_CF32 else np.empty((n, 2), np.uint8 if fmt == FMT_U8 else np.int16)
    fib = np.zeros((n_frames, 3072), np.uint8)
    msc = [np.zeros((4 * n_frames, 24 * s.bit_rate), np.uint8) for s in subch]
    ptrs = (ctypes.c_void_p * max(len(subch), 1))(*[m.ctypes.data for m in msc])
    rc = lib.dabsynth_generate(ctypes.byref(cfg), out.ctypes.data, fib.ctypes.data, ptrs)
    if rc != 0:
        raise ValueError(f"dabsynth_generate failed ({rc}): bad sub-channel table?")
    return Recording(out, fmt, fib, msc, list(subch))
