"""Packet-mode FEC test support: an RS(204,188) encoder of its own and an FEC frame builder (ETSI EN 300 401 clause 5.3.5) on top of
the packet builder of packet_support, the plain-C restatement tests/native/pfec_oracle.c and the host build of pfec.cuh
(tests/native/pfec_check.cu), both compiled into a temporary directory that is removed at exit."""
from __future__ import annotations

import ctypes
import functools
import os
import shutil
import subprocess

import numpy as np

import packet_support as ps

FEC_FIELDS = ("first_slot", "run_slot", "first_frame", "last_frame", "status", "rows_corrected", "rows_failed", "bytes_corrected", "headers_matched",
              "reserved")
CLEAN, CORRECTED, PARTIAL, INCOMPLETE = 0, 1, 2, 3

# ---- GF(2^8), x^8 + x^4 + x^3 + x^2 + 1
_EXP = [0] * 512
_LOG = [0] * 256
_x = 1
for _i in range(255):
    _EXP[_i] = _EXP[_i + 255] = _x
    _LOG[_x] = _i
    _x <<= 1
    if _x & 0x100:
        _x ^= 0x11D


def _mul(a: int, b: int) -> int:
    return _EXP[_LOG[a] + _LOG[b]] if a and b else 0


def _generator() -> list[int]:
    """prod_{i=0..15} (x + alpha^i), highest degree first"""
    g = [1]
    for i in range(16):
        r = _EXP[i]
        out = g + [0]
        for k in range(len(g)):
            out[k + 1] ^= _mul(g[k], r)
        g = out
    return g


_GEN = _generator()


def rs_encode(info: bytes) -> bytes:
    """the 16 parity bytes of 188 information bytes: info(x) x^16 mod g(x)"""
    assert len(info) == 188
    rem = [0] * 16
    for b in info:
        f = b ^ rem[0]
        rem = rem[1:] + [0]
        if f:
            for k in range(16):
                rem[k] ^= _mul(f, _GEN[k + 1])
    return bytes(rem)


def fec_packets(adt: bytes, ci0: int) -> bytes:
    """the 9 FEC packets of a 2256-byte ADT: 2-byte headers (length 00, CI counting from ci0, first / last flags of one run, address
    1022), then the 192 RS bytes (row j mod 12, parity byte j / 12) and 6 padding bytes"""
    par = [rs_encode(adt[r::12]) for r in range(12)]
    rs = bytes(par[j % 12][j // 12] for j in range(192)) + bytes(6)
    out = b""
    for q in range(9):
        fl = 2 if q == 0 else (1 if q == 8 else 0)
        ci = (ci0 + q) & 3
        out += bytes([(ci << 4) | (fl << 2) | (1022 >> 8), 1022 & 0xFF]) + rs[22 * q:22 * q + 22]
    return out


def build_fec_stream(bit_rate: int, n_frames: int, groups: dict, rng, lead_slots: int = 0, padding: float = 0.15, lengths=(24, 48, 72, 96)):
    """Logical frames of a packet-mode sub-channel with packet-mode FEC: after lead_slots slots of padding packets, FEC frames back to
    back until the stream ends (the last one may be cut). Each ADT holds whole packets carrying groups {address: [group bytes, ...]}
    (and padding), none crossing the ADT end or a logical-frame end. Returns (bits uint8[n_frames, 24 * bit_rate], bytes, truth)
    where truth = {"groups": {address: [group bytes sent complete]}, "spans": {address: [(slot of its first packet, slot of its last)]},
    "runs": [run slot of every FEC frame that starts in the stream]}."""
    spf = bit_rate // 8
    n = n_frames * spf
    buf = bytearray(n * 24 + 103 * 24 * 2)
    queue = {a: list(gs) for a, gs in groups.items()}
    cur = {a: None for a in groups}
    ci = {a: int(rng.integers(4)) for a in groups}
    sent = {a: [] for a in groups}
    span = {a: [] for a in groups}
    runs = []
    fec_ci = int(rng.integers(4))

    def put_packets(s0, s1, fill_only=False):
        s = s0
        while s < s1:
            room = min(s1 - s, spf - s % spf)
            L = int(rng.choice([x for x in lengths if x // 24 <= room]))
            live = [a for a in groups if cur[a] is not None or queue[a]]
            if fill_only or not live or rng.random() < padding:
                p = ps.packet(L, 0, 3, 0, b"")
            else:
                a = live[int(rng.integers(len(live)))]
                if cur[a] is None:
                    cur[a] = [queue[a].pop(0), 0, s]
                g, o, g0 = cur[a]
                take = min(L - 5, len(g) - o)
                fl = (2 if o == 0 else 0) | (1 if o + take == len(g) else 0)
                p = ps.packet(L, ci[a], fl, a, g[o:o + take])
                ci[a] = (ci[a] + 1) & 3
                cur[a][1] = o + take
                if o + take == len(g):
                    if s + L // 24 <= n:
                        sent[a].append(bytes(g))
                        span[a].append((g0, s))
                    cur[a] = None
            buf[s * 24:s * 24 + L] = p
            s += L // 24

    put_packets(0, lead_slots, fill_only=True)
    s = lead_slots
    while s < n:
        put_packets(s, s + 94)
        adt = bytes(buf[s * 24:(s + 94) * 24])
        buf[(s + 94) * 24:(s + 103) * 24] = fec_packets(adt, fec_ci)
        fec_ci = (fec_ci + 9) & 3
        if s + 94 < n:
            runs.append(s + 94)
        s += 103
    raw = np.frombuffer(bytes(buf[:n * 24]), np.uint8).reshape(n_frames, 3 * bit_rate).copy()
    return np.unpackbits(raw, axis=1), raw, {"groups": sent, "spans": span, "runs": runs}


def byte_errors(raw: np.ndarray, rng, rate: float = 0.0, bursts: int = 0, burst_len: int = 96) -> np.ndarray:
    """a copy of the packed bytes with random byte errors at `rate` and `bursts` bursts of up to burst_len bytes"""
    out = raw.copy().reshape(-1)
    hit = np.flatnonzero(rng.random(out.size) < rate)
    out[hit] ^= rng.integers(1, 256, hit.size, np.uint8)
    for _ in range(bursts):
        at, ln = int(rng.integers(out.size)), int(rng.integers(1, burst_len + 1))
        seg = out[at:at + ln]
        seg ^= rng.integers(1, 256, seg.size, np.uint8)
    return out.reshape(raw.shape)


def fec_key(r) -> tuple:
    return tuple(int(getattr(r, f)) for f in FEC_FIELDS)


class _FecRec:
    def __init__(self, row):
        for f, v in zip(FEC_FIELDS, row):
            setattr(self, f, int(v))


class _Runner:
    def __init__(self, so: str, prefix: str):
        self.lib = ctypes.CDLL(so)
        self.dec = getattr(self.lib, prefix + "decode")
        self.dec.restype = ctypes.c_int
        self.run_fn = getattr(self.lib, prefix + "run")
        self.run_fn.restype = ctypes.c_int

    def decode(self, cw: bytes):
        """(corrected bytes or -1, code word after the call)"""
        b = np.frombuffer(bytes(cw), np.uint8).copy()
        m = self.dec(b.ctypes.data_as(ctypes.c_void_p))
        return m, bytes(b)

    def run(self, raw: np.ndarray, bit_rate: int):
        """(corrected packed bytes, FEC mask per slot, records)"""
        b = np.ascontiguousarray(raw, np.uint8).reshape(-1, 3 * bit_rate)
        n = b.shape[0]
        cor = np.zeros_like(b)
        mask = np.zeros(n * (bit_rate // 8), np.uint8)
        cap = n * (bit_rate // 8) // 2 + 1
        rec = np.zeros((cap, 10), np.int32)
        m = self.run_fn(b.ctypes.data_as(ctypes.c_void_p), bit_rate, n, cor.ctypes.data_as(ctypes.c_void_p), mask.ctypes.data_as(ctypes.c_void_p),
                        rec.ctypes.data_as(ctypes.c_void_p), cap)
        return cor, mask, [_FecRec(r) for r in rec[:m]]


@functools.lru_cache(maxsize=None)
def oracle() -> _Runner:
    """tests/native/pfec_oracle.c, built with gcc."""
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        raise RuntimeError("no C compiler for the FEC oracle")
    so = os.path.join(ps._build_dir(), "libpfec_oracle.so")
    subprocess.run([cc, "-O2", "-std=c99", "-shared", "-fPIC", "-o", so, os.path.join(ps.NATIVE, "pfec_oracle.c")], check=True)
    return _Runner(so, "dabo_pfec_")


class _Check(_Runner):
    def __init__(self, so: str):
        super().__init__(so, "pfck_")
        self.groups_fn = self.lib.pfck_groups
        self.groups_fn.restype = ctypes.c_int

    def groups(self, frame_bits: np.ndarray, bit_rate: int, address: int, dg_flag: int = 0):
        """(records, payload uint8[bytes], stats) of the packet walk on the corrected bytes with the FEC packets skipped"""
        b = np.ascontiguousarray(frame_bits, np.uint8).reshape(-1, 24 * bit_rate)
        n = b.shape[0]
        cap = max(n * (bit_rate // 8), 1)
        rec = np.zeros((cap, len(ps.FIELDS)), np.int64)
        pay = np.zeros(max(n * 3 * bit_rate, 1), np.uint8)
        st = np.zeros(15, np.int64)
        m = self.groups_fn(b.ctypes.data_as(ctypes.c_void_p), bit_rate, n, address, dg_flag, rec.ctypes.data_as(ctypes.c_void_p), cap,
                           pay.ctypes.data_as(ctypes.c_void_p), st.ctypes.data_as(ctypes.c_void_p))
        recs = [ps._Rec(r) for r in rec[:m]]
        return recs, pay[:sum(r.length for r in recs)], ps._Stats(st)


@functools.lru_cache(maxsize=None)
def host_check() -> _Check:
    """tests/native/pfec_check.cu (the host build of pfec.cuh with packet.cuh), built with nvcc."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    so = os.path.join(ps._build_dir(), "libpfec_check.so")
    subprocess.run([nvcc, "-O1", "-std=c++17", "-Wno-deprecated-gpu-targets", "-diag-suppress", "20013,20015", "-Xcompiler", "-fPIC", "-shared", "-I", ps.CSRC,
                    "-o", so, os.path.join(ps.NATIVE, "pfec_check.cu")], check=True)
    return _Check(so)


def oracle_groups(raw: np.ndarray, bit_rate: int, address: int, dg_flag: int = 0):
    """The restatement's groups: its corrected bytes with every slot of a located FEC-packet run replaced by a padding packet, walked by
    the packet restatement (packet_oracle.c); records and payload equal those of the walk that skips the FEC packets."""
    cor, mask, _ = oracle().run(raw, bit_rate)
    flat = cor.reshape(-1, 24).copy()
    flat[mask.astype(bool)] = np.frombuffer(ps.packet(24, 0, 3, 0, b""), np.uint8)
    bits = np.unpackbits(flat.reshape(raw.shape), axis=1)
    return ps.oracle().run(bits, bit_rate, address, dg_flag)
