"""Packet-mode test support: a packet and MSC data group builder with its own CRC (ETSI EN 300 401 clauses 5.3.2, 5.3.3), the
plain-C restatement tests/native/packet_oracle.c and the host build of packet.cuh (tests/native/packet_check.cu), both compiled
into a temporary directory that is removed at exit."""
from __future__ import annotations

import atexit
import ctypes
import functools
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
NATIVE = os.path.join(HERE, "native")
CSRC = os.path.join(os.path.dirname(HERE), "dabstar_b200", "csrc")
OK, NO_CRC, CRC_ERROR, MALFORMED, RAW = 0, 1, 2, 3, 4
FIELDS = ("first_frame", "last_frame", "n_packets", "status", "extension_flag", "crc_flag", "segment_flag", "user_access_flag", "type", "continuity",
          "repetition", "extension", "segment_last", "segment_number", "transport_id", "length_indicator", "crc_stored", "crc_computed", "length",
          "data_start", "data_length", "reserved", "offset")
STATS = ("packets", "crc_errors", "bad_length", "cut", "padding", "command", "other_address", "continuity_breaks", "abandoned", "dropped")


# ---- CRC: the generator polynomial applied bit by bit to build a byte table
def _table():
    t = []
    for v in range(256):
        r = v << 8
        for _ in range(8):
            r = ((r << 1) ^ 0x1021) if r & 0x8000 else (r << 1)
        t.append(r & 0xFFFF)
    return t


_T = _table()


def crc16(data: bytes) -> int:
    """x^16 + x^12 + x^5 + 1, preset 0xFFFF, complemented (CRC-16/GENIBUS)."""
    r = 0xFFFF
    for b in data:
        r = ((r << 8) & 0xFFFF) ^ _T[(r >> 8) ^ b]
    return r ^ 0xFFFF


def data_group(data: bytes, dg_type: int = 4, crc: bool = True, cont: int = 0, rep: int = 0, extension: int | None = None,
               segment: tuple[int, int] | None = None, transport_id: int | None = None, end_user: bytes | None = None) -> bytes:
    """An MSC data group (clause 5.3.3): header, session header (segment field, user access field), data field, CRC."""
    ua = transport_id is not None or end_user is not None
    h = bytes([(extension is not None) << 7 | crc << 6 | (segment is not None) << 5 | ua << 4 | (dg_type & 15), (cont & 15) << 4 | (rep & 15)])
    if extension is not None:
        h += extension.to_bytes(2, "big")
    if segment is not None:
        h += ((segment[0] & 1) << 15 | (segment[1] & 0x7FFF)).to_bytes(2, "big")
    if ua:
        eu = end_user or b""
        li = (2 if transport_id is not None else 0) + len(eu)
        h += bytes([(transport_id is not None) << 4 | li]) + (transport_id.to_bytes(2, "big") if transport_id is not None else b"") + eu
    g = h + bytes(data)
    return g + crc16(g).to_bytes(2, "big") if crc else g


def packet(length: int, ci: int, fl: int, address: int, useful: bytes, command: int = 0, useful_len: int | None = None) -> bytes:
    """One packet (clause 5.3.2): 24-bit header, data field padded with zeros, CRC."""
    ul = len(useful) if useful_len is None else useful_len
    hdr = ((length // 24 - 1) << 22 | (ci & 3) << 20 | (fl & 3) << 18 | (address & 1023) << 8 | (command & 1) << 7 | (ul & 127)).to_bytes(3, "big")
    body = hdr + bytes(useful) + bytes(length - 5 - len(useful))
    return body + crc16(body).to_bytes(2, "big")


def build_stream(bit_rate: int, n_frames: int, groups: dict, rng, padding: float = 0.15, command: float = 0.0, drop: float = 0.0,
                 lengths=(24, 48, 72, 96), junk_frames=()):
    """Logical frames of a packet-mode sub-channel carrying groups {address: [group bytes, ...]} interleaved packet by packet, with
    padding packets between them. drop: probability that a data packet is replaced by a padding packet of its length (its
    group is then not complete). Returns (bits uint8[n_frames, 24 * bit_rate], bytes uint8[n_frames, 3 * bit_rate], truth
    {address: [(first_frame, last_frame, group bytes)]}) where truth lists the groups sent complete."""
    fb = 3 * bit_rate
    out = np.zeros((n_frames, fb), np.uint8)
    queue = {a: list(gs) for a, gs in groups.items()}
    cur = {a: None for a in groups}  # (group, offset, first_frame, intact)
    ci = {a: int(rng.integers(4)) for a in groups}
    truth = {a: [] for a in groups}
    for f in range(n_frames):
        pos = 0
        while pos < fb:
            room = fb - pos
            ok_len = [x for x in lengths if x <= room]
            L = int(rng.choice(ok_len))
            live = [a for a in groups if cur[a] is not None or queue[a]]
            if not live or rng.random() < padding:
                p = packet(L, 0, 3, 0, b"")
            elif command and rng.random() < command:
                a = live[int(rng.integers(len(live)))]
                p = packet(L, int(rng.integers(4)), 3, a, bytes(rng.integers(0, 256, min(L - 5, 7), np.uint8)), command=1)
            else:
                a = live[int(rng.integers(len(live)))]
                if cur[a] is None:
                    cur[a] = [queue[a].pop(0), 0, f, True]
                g, o, f0, intact = cur[a]
                take = min(L - 5, len(g) - o)
                fl = (2 if o == 0 else 0) | (1 if o + take == len(g) else 0)
                p = packet(L, ci[a], fl, a, g[o:o + take])
                ci[a] = (ci[a] + 1) & 3
                if drop and rng.random() < drop:
                    p = packet(L, 0, 3, 0, b"")
                    cur[a][3] = False
                cur[a][1] = o + take
                if o + take == len(g):
                    if cur[a][3]:
                        truth[a].append((f0, f, bytes(g)))
                    cur[a] = None
            out[f, pos:pos + L] = np.frombuffer(p, np.uint8)
            pos += L
    for f in junk_frames:
        out[f] = rng.integers(0, 256, fb, np.uint8)
    bits = np.unpackbits(out, axis=1)
    return bits, out, truth


def random_groups(rng, n: int, sizes=(0, 400), crc_share: float = 0.8) -> list[bytes]:
    gs = []
    for _ in range(n):
        size = int(rng.integers(sizes[0], sizes[1] + 1))
        kw = {}
        if rng.random() < 0.3:
            kw["extension"] = int(rng.integers(65536))
        if rng.random() < 0.5:
            kw["segment"] = (int(rng.integers(2)), int(rng.integers(32768)))
        if rng.random() < 0.4:
            kw["transport_id"] = int(rng.integers(65536))
            kw["end_user"] = bytes(rng.integers(0, 256, int(rng.integers(0, 4)), np.uint8))
        elif rng.random() < 0.2:
            kw["end_user"] = bytes(rng.integers(0, 256, int(rng.integers(0, 8)), np.uint8))
        gs.append(data_group(bytes(rng.integers(0, 256, size, np.uint8)), dg_type=int(rng.integers(16)), crc=rng.random() < crc_share,
                             cont=int(rng.integers(16)), rep=int(rng.integers(16)), **kw))
    return gs


def key(r) -> tuple:
    return tuple(int(getattr(r, f)) for f in FIELDS)


def stats_key(s) -> tuple:
    return tuple(int(getattr(s, f)) for f in STATS) + tuple(int(x) for x in s.groups)


@functools.lru_cache(maxsize=None)
def _build_dir() -> str:
    d = tempfile.mkdtemp(prefix="dabstar_packet_")
    atexit.register(shutil.rmtree, d, True)
    return d


class _Rec:
    def __init__(self, row):
        for f, v in zip(FIELDS, row):
            setattr(self, f, int(v))


class _Stats:
    def __init__(self, row):
        for f, v in zip(STATS, row[:10]):
            setattr(self, f, int(v))
        self.groups = [int(x) for x in row[10:15]]


class _Runner:
    def __init__(self, so: str, prefix: str):
        self.lib = ctypes.CDLL(so)
        self.crc_fn = getattr(self.lib, prefix + "crc")
        self.crc_fn.restype = ctypes.c_uint
        self.run_fn = getattr(self.lib, prefix + "run")
        self.run_fn.restype = ctypes.c_int

    def crc(self, data: bytes) -> int:
        b = np.frombuffer(bytes(data) or b"\0", np.uint8)
        return int(self.crc_fn(b.ctypes.data_as(ctypes.c_void_p), len(data)))

    def run(self, frame_bits: np.ndarray, bit_rate: int, address: int, dg_flag: int = 0):
        """(records, payload uint8[bytes], stats)"""
        b = np.ascontiguousarray(frame_bits, np.uint8).reshape(-1, 24 * bit_rate)
        n = b.shape[0]
        cap = max(n * (bit_rate // 8), 1)
        rec = np.zeros((cap, len(FIELDS)), np.int64)
        pay = np.zeros(max(n * 3 * bit_rate, 1), np.uint8)
        st = np.zeros(15, np.int64)
        m = self.run_fn(b.ctypes.data_as(ctypes.c_void_p), bit_rate, n, address, dg_flag, rec.ctypes.data_as(ctypes.c_void_p), cap,
                        pay.ctypes.data_as(ctypes.c_void_p), st.ctypes.data_as(ctypes.c_void_p))
        recs = [_Rec(r) for r in rec[:m]]
        return recs, pay[:sum(r.length for r in recs)], _Stats(st)


@functools.lru_cache(maxsize=None)
def oracle() -> _Runner:
    """tests/native/packet_oracle.c, built with gcc."""
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        raise RuntimeError("no C compiler for the packet oracle")
    so = os.path.join(_build_dir(), "libpacket_oracle.so")
    subprocess.run([cc, "-O2", "-std=c99", "-shared", "-fPIC", "-o", so, os.path.join(NATIVE, "packet_oracle.c")], check=True)
    return _Runner(so, "dabo_pkt_")


@functools.lru_cache(maxsize=None)
def host_check() -> _Runner:
    """tests/native/packet_check.cu (the host build of packet.cuh), built with nvcc."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    so = os.path.join(_build_dir(), "libpacket_check.so")
    subprocess.run([nvcc, "-O1", "-std=c++17", "-Wno-deprecated-gpu-targets", "-Xcompiler", "-fPIC", "-shared", "-I", CSRC, "-o", so,
                    os.path.join(NATIVE, "packet_check.cu")], check=True)
    return _Runner(so, "pchk_")
