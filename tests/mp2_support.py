"""MPEG layer II audio frames for the MP2 tests: a frame builder with its own CRC (a third statement of the check, beside
dabstar_b200/csrc/mp2.cuh and tests/native/mp2_oracle.c), the plain-C oracle and the host build of mp2.cuh, each compiled into a
temporary directory, and the stream scenarios both the CPU and the GPU tests use."""
from __future__ import annotations

import atexit
import ctypes
import functools
import os
import shutil
import subprocess
import tempfile

import numpy as np

from dabstar_b200._lib import Mp2FrameC

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NATIVE = os.path.join(ROOT, "tests", "native")
CSRC = os.path.join(ROOT, "dabstar_b200", "csrc")

RATES_MPEG1 = [32, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320, 384]
RATES_LSF = [8, 16, 24, 32, 40, 48, 56, 64, 80, 96, 112, 128, 144, 160]
OK, NO_HEADER, MISMATCH, CRC_ERROR, CUT = 0, 1, 2, 3, 4


def crc16(bits) -> int:
    """CRC-16 x^16 + x^15 + x^2 + 1, preset 0xFFFF, over bits (MSB first), no final inversion (ISO/IEC 11172-3 2.4.3.1)."""
    crc = 0xFFFF
    for b in bits:
        top = (crc >> 15) & 1
        crc = (crc << 1) & 0xFFFF
        if top ^ int(b):
            crc ^= 0x8005
    return crc


def bytes_to_bits(data: bytes) -> np.ndarray:
    return np.unpackbits(np.frombuffer(bytes(data), np.uint8))


def nbal_table(sample_rate: int, bit_rate: int, mode: int) -> list[int]:
    nch = 1 if mode == 3 else 2
    if sample_rate == 24000:  # ISO/IEC 13818-3 Table B.1
        return [4] * 4 + [3] * 7 + [2] * 19
    if bit_rate // nch >= 56:  # ISO/IEC 11172-3 Table B.2a
        return [4] * 11 + [3] * 12 + [2] * 4
    return [4] * 2 + [3] * 6   # Table B.2c


def alloc_bits(sample_rate: int, bit_rate: int, mode: int, mode_ext: int) -> int:
    nbal = nbal_table(sample_rate, bit_rate, mode)
    nch = 1 if mode == 3 else 2
    bound = min(4 * (mode_ext + 1), len(nbal)) if mode == 1 else len(nbal)
    return sum(n * (nch if sb < bound else 1) for sb, n in enumerate(nbal))


def mp2_frame(bit_rate: int, rng: np.random.Generator, sample_rate: int = 48000, mode: int = 0, mode_ext: int = 0, layout: bool = False):
    """One DAB audio frame, uint8[n_logical, 24 * bit_rate] bits (n_logical 1 at 48 kHz, 2 at 24 kHz): a valid layer II header with
    CRC, random allocations (a share of them zero) and SCFSI, random bits after. layout=True also returns the bit positions
    (allocation start, SCFSI start, SCFSI end)."""
    lsf = sample_rate == 24000
    rates = RATES_LSF if lsf else RATES_MPEG1
    n_bits = (48 if lsf else 24) * bit_rate
    bits = rng.integers(0, 2, n_bits, dtype=np.uint8)

    def put(pos, value, n):
        for i in range(n):
            bits[pos + i] = (value >> (n - 1 - i)) & 1

    put(0, 0xFFF, 12)
    put(12, 0 if lsf else 1, 1)
    put(13, 2, 2)                  # layer II
    put(15, 0, 1)                  # protection_bit 0: CRC present
    put(16, rates.index(bit_rate) + 1, 4)
    put(20, 1, 2)                  # 48 kHz (ID 1) / 24 kHz (ID 0)
    put(24, mode, 2)
    put(26, mode_ext, 2)
    nbal = nbal_table(sample_rate, bit_rate, mode)
    nch = 1 if mode == 3 else 2
    bound = min(4 * (mode_ext + 1), len(nbal)) if mode == 1 else len(nbal)
    pos = 48
    alloc = []
    for sb, nb in enumerate(nbal):
        vals = [int(rng.integers(0, 1 << nb)) if rng.random() < 0.7 else 0 for _ in range(nch if sb < bound else 1)]
        for v in vals:  # one per channel below the bound, one shared from there on
            put(pos, v, nb)
            pos += nb
        alloc.append(vals if sb < bound else vals * nch)
    a_end = pos
    pos += 2 * sum(1 for vals in alloc for v in vals if v)  # SCFSI: random bits already there
    crc = crc16(np.concatenate([bits[16:32], bits[48:pos]]))
    put(32, crc, 16)
    out = bits.reshape(-1, 24 * bit_rate)
    return (out, (48, a_end, pos)) if layout else out


def mp2_stream(bit_rate: int, n: int, rng: np.random.Generator, sample_rate=48000, lead: int = 0, junk=(), slip=None, byte_errors: float = 0.0,
               damage_header=(), mixed: bool = False, mode: int | None = None):
    """n logical frames of one sub-channel: random bits for `lead` frames, then back-to-back audio frames (modes drawn at random;
    mixed: 48 and 24 kHz frames alternate in runs), junk: frame slots left random, slip: one random logical frame inserted before
    slot `slip`, damage_header: slots whose header gets one bit flipped; byte_errors: that share of all bytes corrupted; mode: one
    mode for every frame (mode_extension cycling through 0..3) instead of random ones. Returns
    (bits uint8[n, 24 * bit_rate], {first logical frame: frame bits} of the frames sent intact)."""
    out = rng.integers(0, 2, (n, 24 * bit_rate), dtype=np.uint8)
    truth = {}
    f, k = lead, 0
    while f < n:
        if slip is not None and k == slip:
            f += 1
            slip = None
            continue
        sr = sample_rate if not mixed else (48000 if (k // 3) % 2 == 0 else 24000)
        if sr == 24000 and bit_rate not in RATES_LSF or sr == 48000 and bit_rate not in RATES_MPEG1:
            sr = 24000 if sr == 48000 else 48000
        m = int(rng.integers(0, 4)) if mode is None else mode
        fr = mp2_frame(bit_rate, rng, sr, m, int(rng.integers(0, 4)) if mode is None else k % 4)
        span = min(fr.shape[0], n - f)
        if k not in junk:
            out[f:f + span] = fr[:span]
            if k in damage_header:
                out[f, int(rng.integers(12, 32))] ^= 1
            elif span == fr.shape[0]:
                truth[f] = fr
        f += fr.shape[0]
        k += 1
    if byte_errors:
        by = np.packbits(out.reshape(-1))
        pos = rng.choice(by.size, max(1, int(by.size * byte_errors)), replace=False)
        by[pos] ^= rng.integers(1, 256, pos.size, dtype=np.uint8)
        out = np.unpackbits(by).reshape(out.shape)
        truth = {f: t for f, t in truth.items() if np.array_equal(out[f:f + t.shape[0]], t)}
    return out, truth


def key(r):
    return (r.first_frame, r.n_frames, r.status, r.header, r.crc_stored, r.crc_computed)


@functools.lru_cache(maxsize=None)
def _build_dir() -> str:
    d = tempfile.mkdtemp(prefix="dabstar_mp2_")
    atexit.register(shutil.rmtree, d, True)
    return d


class Mp2Oracle:
    """tests/native/mp2_oracle.c, built with gcc into a temporary directory."""

    def __init__(self):
        cc = shutil.which("gcc") or shutil.which("cc")
        if cc is None:
            raise RuntimeError("no C compiler for the MP2 oracle")
        so = os.path.join(_build_dir(), "libmp2_oracle.so")
        if not os.path.exists(so):
            subprocess.run([cc, "-std=c99", "-O2", "-shared", "-fPIC", "-o", so, os.path.join(NATIVE, "mp2_oracle.c")], check=True)
        self.lib = ctypes.CDLL(so)
        self.lib.dabo_mp2_crc16.restype = ctypes.c_uint
        self.lib.dabo_mp2_alloc_bits.restype = ctypes.c_int
        self.lib.dabo_mp2_run.restype = ctypes.c_int

    def crc16(self, data: bytes) -> int:
        b = np.frombuffer(bytes(data), np.uint8).copy()
        return int(self.lib.dabo_mp2_crc16(b.ctypes.data_as(ctypes.c_void_p), b.size))

    def alloc_bits(self, khz: int, bit_rate: int, mode: int, mode_ext: int) -> int:
        return int(self.lib.dabo_mp2_alloc_bits(khz, bit_rate, mode, mode_ext))

    def run(self, frame_bits: np.ndarray, bit_rate: int):
        """dabo_mp2_run: (records, payload uint8[bytes])."""
        b = np.ascontiguousarray(frame_bits, np.uint8).reshape(-1, 24 * bit_rate)
        n = b.shape[0]
        rec = (Mp2FrameC * max(n, 1))()
        pay = np.zeros(max(n, 1) * 3 * bit_rate, np.uint8)
        m = self.lib.dabo_mp2_run(b.ctypes.data_as(ctypes.c_void_p), bit_rate, n, rec, n, pay.ctypes.data_as(ctypes.c_void_p))
        recs = list(rec[:m])
        return recs, pay[:sum(3 * bit_rate * r.n_frames for r in recs if r.status == OK)]


@functools.lru_cache(maxsize=None)
def oracle() -> Mp2Oracle:
    return Mp2Oracle()


@functools.lru_cache(maxsize=None)
def host_driver() -> str:
    """tests/native/mp2_check.cu (the host build of mp2.cuh), built with nvcc into a temporary directory."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    exe = os.path.join(_build_dir(), "mp2_check")
    subprocess.run([nvcc, "-O1", "-std=c++17", "-Wno-deprecated-gpu-targets", "-I", CSRC, "-o", exe, os.path.join(NATIVE, "mp2_check.cu")], check=True)
    return exe


def host_run(exe: str, streams):
    """streams: [(frame_bits, bit_rate)] -> [(records as key tuples, payload bytes)] from the host build of mp2.cuh."""
    lines = []
    for bits, br in streams:
        packed = np.packbits(np.ascontiguousarray(bits, np.uint8).reshape(-1))
        lines.append(f"run {br} {bits.shape[0]} {packed.tobytes().hex()}\n")
    out = subprocess.run([exe], input="".join(lines), capture_output=True, text=True, check=True).stdout.splitlines()
    res, i = [], 0
    for _ in streams:
        n = int(out[i])
        recs = [tuple(int(x) for x in out[i + 1 + k].split()) for k in range(n)]
        pay = b"" if out[i + 1 + n] == "-" else bytes.fromhex(out[i + 1 + n])
        res.append((recs, pay))
        i += n + 2
    return res


def host_command(exe: str, text: str) -> list[str]:
    return subprocess.run([exe], input=text, capture_output=True, text=True, check=True).stdout.split()
