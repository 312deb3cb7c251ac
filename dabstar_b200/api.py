"""Host-side mirror of the reference's receive-chain classes over the C ABI (include/dabstar_b200.h).

The class and method names follow the reference (OfdmDecoder, PhaseReference, FreqInterleaver, FicDecoder alias
FicHandler, Backend, Protection, ViterbiSpiral, DabProcessor) so the parity tests read like calls into it; the
arguments are batches because the device boundary is batch granular (SURVEY.md section 7). numpy arrays are host
memory, torch CUDA tensors are passed by device pointer. Nothing here computes on the CPU.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import DabstarError, DecoderCfg, FrameInfo, SubCh, c_p
from .synth import SubChannel

MEM_HOST, MEM_DEVICE = 0, 1
FMT_CF32, FMT_U8, FMT_I16 = 0, 1, 2
T_FRAME = 196608
FRAME_SOFT = 75 * 3072


def _np(a, dtype) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=dtype)


def _ptr(a: np.ndarray) -> c_p:
    return a.ctypes.data_as(c_p)


CONTAINERS = {"int8": 0, "uint8": 1, "int16": 2, "int24": 3, "int32": 4, "float32": 5, "uint8_pcm": 6, "int32_pcm": 7}
FILE_KINDS = ("raw", "xml", "wav")
READER_XML, READER_WAV = 0, 1
IQ_ORDERS = {"IQ": 0, "QI": 1, "I_Only": 2, "Q_Only": 3}


@dataclass
class SampleFormat:
    """Sample description of an XML/UFF, raw or WAV recording (xml-descriptor fields Container / bitsperChannel / Ordering / iqOrder)."""
    container: str = "uint8"
    bits_per_channel: int = 0   # 0: the container's width
    byte_order: str = "LSB"
    iq_order: str = "IQ"

    def c_struct(self) -> _lib.SampleFormatC:
        return _lib.SampleFormatC(CONTAINERS.get(self.container, -1), int(self.bits_per_channel), 1 if self.byte_order == "MSB" else 0, IQ_ORDERS.get(self.iq_order, -1))

    def native(self) -> int | None:
        """The decoder input format that reads this layout directly (converted inside the FFT kernel), if any."""
        if self.iq_order != "IQ":
            return None
        if self.container == "uint8":
            return FMT_U8
        if self.container == "int16" and self.byte_order == "LSB" and self.bits_per_channel in (0, 16):
            return FMT_I16
        if self.container == "float32" and self.byte_order == "LSB":
            return FMT_CF32
        return None


class Mp4Processor:
    """backend/audio/mp4processor.h for a run of logical frames: super-frame sync, RS(120,110), Fire code, AU borders and CRCs on the GPU."""

    def __init__(self, bit_rate: int, ctx: "Context | None" = None):
        self.ctx = ctx or default_context()
        self.bit_rate = int(bit_rate)

    def add_frames(self, frame_bits: np.ndarray):
        """frame_bits: uint8[n_frames, 24*bit_rate] (FrameProcessor::add_to_frame payloads). Returns (records, payload[n, 110*bit_rate/8])."""
        b = _np(frame_bits, np.uint8).reshape(-1, 24 * self.bit_rate)
        n = b.shape[0]
        cap = max(n, 1)
        rec = (_lib.SuperFrameC * cap)()
        pay = np.zeros((cap, 110 * (self.bit_rate // 8)), np.uint8)
        m = self.ctx.check(self.ctx.lib.dabstar_dabplus_decode(self.ctx.h, _ptr(b), self.bit_rate, n, rec, cap, _ptr(pay), MEM_HOST), "dabstar_dabplus_decode")
        return list(rec[:m]), pay[:m]

    @staticmethod
    def access_units(rec, payload_row: np.ndarray) -> list[bytes]:
        """The CRC-good access units of an accepted super-frame, as handed to the AAC decoder (mp4processor.cpp:333-372)."""
        if not rec.ok:
            return []
        return [payload_row[rec.au_start[u]:rec.au_start[u + 1] - 2].tobytes() for u in range(rec.num_aus) if rec.au_state[u] == 1]


@dataclass
class ServiceComponent:
    sid: int
    comp_index: int
    tmid: int
    type: int
    sub_ch_id: int
    primary: int
    ca_flag: int


class FibParser:
    """FibDecoder::process_FIB for FIG 0/0, 0/1, 0/2 (fib_decoder.cpp:59-106, fib_decoder_fig0.cpp:89-290): host code, no device."""

    def __init__(self):
        self.lib = _lib.load()
        self.h = c_p()
        if self.lib.dabstar_fib_parser_create(ctypes.byref(self.h)) != 0:
            raise DabstarError("dabstar_fib_parser_create failed")

    def __del__(self):
        try:
            if self.h:
                self.lib.dabstar_fib_parser_destroy(self.h)
                self.h = c_p()
        except Exception:
            pass

    def process_FIB(self, fib_bits: np.ndarray):
        """fib_bits: uint8[n, 256] (or [256]), one bit per byte; the caller has checked the CRCs."""
        b = _np(fib_bits, np.uint8).reshape(-1, 256)
        if self.lib.dabstar_fib_parser_push(self.h, _ptr(b), b.shape[0]) != 0:
            raise DabstarError("dabstar_fib_parser_push failed")

    def ensemble(self) -> _lib.EnsembleInfoC | None:
        e = _lib.EnsembleInfoC()
        seen = self.lib.dabstar_fib_parser_ensemble(self.h, ctypes.byref(e))
        return e if seen == 1 else None

    def get_cif_count(self) -> tuple[int, int]:
        e = _lib.EnsembleInfoC()
        seen = self.lib.dabstar_fib_parser_ensemble(self.h, ctypes.byref(e))
        return (e.cif_count_hi, e.cif_count_lo) if seen == 1 else (-1, -1)

    def sub_channels(self) -> list[SubChannel]:
        n = self.lib.dabstar_fib_parser_subchannels(self.h, None, 0)
        arr = (SubCh * max(n, 1))()
        self.lib.dabstar_fib_parser_subchannels(self.h, arr, n)
        return [SubChannel(a.sub_ch_id, a.start_cu, a.size_cu, a.short_form, a.prot_level, a.bit_rate, a.start_frame) for a in arr[:n]]

    def components(self) -> list[ServiceComponent]:
        n = self.lib.dabstar_fib_parser_components(self.h, None, 0)
        arr = (_lib.ServiceCompC * max(n, 1))()
        self.lib.dabstar_fib_parser_components(self.h, arr, n)
        return [ServiceComponent(a.sid, a.comp_index, a.tmid, a.type, a.sub_ch_id, a.primary, a.ca_flag) for a in arr[:n]]


class Context:
    """One CUDA device + stream (dabstar_create). `stream` may be a torch.cuda.Stream or None for a private stream."""

    def __init__(self, device: int = 0, stream=None):
        self.lib = _lib.load()
        self.h = c_p()
        sp = c_p(stream.cuda_stream) if stream is not None else None
        rc = self.lib.dabstar_create(ctypes.byref(self.h), int(device), sp)
        if rc != 0:
            raise DabstarError(f"dabstar_create failed ({rc}): no usable CUDA device {device}; there is no CPU fallback")
        self.device = device

    def close(self):
        if self.h:
            self.lib.dabstar_destroy(self.h)
            self.h = c_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc: int, what: str) -> int:
        if rc < 0:
            raise DabstarError(f"{what} failed ({rc}): {self.lib.dabstar_last_error(self.h).decode()}")
        return rc

    @property
    def kernel_launches(self) -> int:
        return int(self.lib.dabstar_kernel_launches(self.h))

    # ---- ingest (row I1)
    def ingest_convert(self, raw: np.ndarray, fmt: "SampleFormat", n_samples: int | None = None) -> np.ndarray:
        """File samples -> complex64 as the reference's file readers convert them (xml_reader.cpp:254-800,
        raw_reader.cpp:66-70, wav_reader.cpp:164). raw: the bytes of the file's data section."""
        raw = np.ascontiguousarray(raw).view(np.uint8).reshape(-1)
        c = fmt.c_struct()
        elem = int(self.lib.dabstar_sample_format_bytes(ctypes.byref(c)))
        if elem == 0:
            raise DabstarError(f"unknown sample format {fmt}")
        n = raw.size // elem if n_samples is None else int(n_samples)
        out = np.empty(n, np.complex64)
        self.check(self.lib.dabstar_ingest_convert(self.h, _ptr(raw), ctypes.byref(c), ctypes.c_int64(n), _ptr(out), MEM_HOST), "dabstar_ingest_convert")
        return out

    def dc_iq_correct(self, x: np.ndarray, do_iq: bool = False, state: "_lib.DcIqStateC | None" = None) -> np.ndarray:
        """SampleReader::set_dc_and_iq_correction(True, do_iq) over a whole recording (sample_reader.cpp:216-243). state: filter
        values carried from an earlier call (updated in place); None = a fresh reader."""
        x = _np(x, np.complex64).reshape(-1)
        out = np.empty_like(x)
        self.check(self.lib.dabstar_dc_iq_correct(self.h, _ptr(x), ctypes.c_int64(x.size), 1 if do_iq else 0, ctypes.byref(state) if state is not None else None,
                                                  _ptr(out), MEM_HOST), "dabstar_dc_iq_correct")
        return out

    def resample_linear(self, x: np.ndarray, sample_rate: int, reader: int = READER_XML) -> np.ndarray:
        """The file readers' conversion to 2.048 MS/s (linear interpolation per 1 ms block; xml_reader.cpp:212-231,
        wav_reader.cpp:196-211). x: complex64 at sample_rate."""
        x = _np(x, np.complex64).reshape(-1)
        n = int(self.lib.dabstar_resample_count(ctypes.c_int64(x.size), int(sample_rate), int(reader)))
        if n < 0:
            raise DabstarError(f"resample: unsupported rate {sample_rate} / reader {reader}")
        out = np.empty(n, np.complex64)
        got = int(self.lib.dabstar_resample_linear(self.h, _ptr(x), ctypes.c_int64(x.size), int(sample_rate), int(reader), _ptr(out), ctypes.c_int64(n), MEM_HOST))
        self.check(min(got, 0), "dabstar_resample_linear")
        return out[:got]

    def read_file(self, data: np.ndarray | bytes | str) -> tuple[np.ndarray, "FileInfo"]:
        """A recording file (path, bytes or uint8 array: raw u8 IQ, XML/UFF, RIFF/WAVE) -> complex64 at 2.048 MS/s, the
        sample stream the reference's file reader would hand to DabProcessor, plus what the header said."""
        if isinstance(data, str):
            data = np.fromfile(data, np.uint8)
        raw = np.frombuffer(data, np.uint8) if isinstance(data, (bytes, bytearray)) else np.ascontiguousarray(data).view(np.uint8).reshape(-1)
        info = file_probe(raw)
        elem = int(self.lib.dabstar_sample_format_bytes(ctypes.byref(info.fmt.c_struct())))
        body = raw[info.data_offset:info.data_offset + info.n_samples * elem]
        x = self.ingest_convert(body, info.fmt, info.n_samples)
        if info.sample_rate != 2048000:
            x = self.resample_linear(x, info.sample_rate, info.reader)
        return x, info

    # ---- stage taps
    def fft2048(self, x: np.ndarray, sign: int = -1) -> np.ndarray:
        """fftwf_execute on the reference's 2048-point plans (dab_processor.cpp:63): x complex64[n, 2048]."""
        x = _np(x, np.complex64).reshape(-1, 2048)
        y = np.empty_like(x)
        self.check(self.lib.dabstar_fft2048(self.h, _ptr(x), _ptr(y), x.shape[0], sign, MEM_HOST), "dabstar_fft2048")
        return y


@dataclass
class FileInfo:
    kind: str            # "raw" | "xml" | "wav"
    reader: int          # READER_XML / READER_WAV
    sample_rate: int
    n_channels: int
    fmt: SampleFormat
    data_offset: int
    n_samples: int
    frequency_hz: int


def file_probe(head: np.ndarray | bytes, file_bytes: int | None = None) -> FileInfo:
    """XmlDescriptor / WavFileHandler / RawReader header inspection (host code, no GPU): see dabstar_file_probe."""
    lib = _lib.load()
    raw = np.frombuffer(head, np.uint8) if isinstance(head, (bytes, bytearray)) else np.ascontiguousarray(head).view(np.uint8).reshape(-1)
    fi = _lib.FileInfoC()
    n = int(raw.size)
    rc = lib.dabstar_file_probe(_ptr(raw), ctypes.c_int64(n), ctypes.c_int64(n if file_bytes is None else file_bytes), ctypes.byref(fi))
    if rc < 0:
        raise DabstarError("dabstar_file_probe: not a playable recording (unsupported header)")
    inv_c = {v: k for k, v in CONTAINERS.items()}
    inv_o = {v: k for k, v in IQ_ORDERS.items()}
    fmt = SampleFormat(inv_c[fi.fmt.container], fi.fmt.bits_per_channel, "MSB" if fi.fmt.msb_first else "LSB", inv_o[fi.fmt.iq_order])
    return FileInfo(FILE_KINDS[fi.kind], fi.reader, fi.sample_rate, fi.n_channels, fmt, int(fi.data_offset), int(fi.n_samples), fi.frequency_hz)


_default_ctx: Context | None = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


class FreqInterleaver:
    """ofdm/freq_interleaver.h:50"""

    def __init__(self, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self.table = np.zeros(1536, np.int16)
        self.ctx.check(self.ctx.lib.dabstar_freq_interleaver(self.ctx.h, _ptr(self.table)), "dabstar_freq_interleaver")

    def map_k_to_fft_bin(self, k: int) -> int:
        return int(self.table[k])


class PhaseReference:
    """ofdm/phasereference.h:53-58"""
    IDX_NOT_FOUND = 100000

    def __init__(self, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self.strongest = 0
        self.mRefTable = np.zeros(2048, np.complex64)
        self.ctx.check(self.ctx.lib.dabstar_phase_table(self.ctx.h, _ptr(self.mRefTable)), "dabstar_phase_table")

    def set_sync_on_strongest_peak(self, sync: bool):
        self.strongest = int(bool(sync))

    def correlate_with_phase_ref_and_find_max_peak(self, samples: np.ndarray, threshold: float) -> np.ndarray:
        x = _np(samples, np.complex64).reshape(-1, 2048)
        out = np.zeros(x.shape[0], np.int32)
        self.ctx.check(self.ctx.lib.dabstar_prs_correlate(self.ctx.h, _ptr(x), x.shape[0], ctypes.c_float(threshold), self.strongest, _ptr(out), MEM_HOST),
                       "dabstar_prs_correlate")
        return out

    def estimate_carrier_offset_from_sync_symbol_0(self, fft: np.ndarray) -> np.ndarray:
        x = _np(fft, np.complex64).reshape(-1, 2048)
        out = np.zeros(x.shape[0], np.int32)
        self.ctx.check(self.ctx.lib.dabstar_estimate_carrier_offset(self.ctx.h, _ptr(x), x.shape[0], _ptr(out), MEM_HOST), "dabstar_estimate_carrier_offset")
        return out


def cp_correlate(frames: np.ndarray, ctx: Context | None = None) -> np.ndarray:
    """Cyclic-prefix correlation of DabProcessor::_process_ofdm_symbols_1_to_L (dab_processor.cpp:317-333): frames = complex64[n, 75 * 2552]
    (symbols 1..75 with prefixes) -> complex64[n]."""
    ctx = ctx or default_context()
    x = _np(frames, np.complex64).reshape(-1, 75 * 2552)
    out = np.zeros(x.shape[0], np.complex64)
    ctx.check(ctx.lib.dabstar_cp_correlate(ctx.h, _ptr(x), x.shape[0], _ptr(out), MEM_HOST), "dabstar_cp_correlate")
    return out


def fft_frames(recordings: list[np.ndarray], fmt: int, frames: list[dict], n_xslots: int, max_ctas_per_sm: int = 0, with_null: bool = False,
               ctx: Context | None = None):
    """The decoder's frame FFT (k_fft_frames; with_null: k_fft_null too) over caller-made frame descriptors (see dabstar_fft_frames).
    recordings: arrays of one format (cf32: complex64[n]; u8: uint8[n, 2]; i16: int16[n, 2]), laid end to end in one buffer.
    frames: dicts with the fields of dabstar_fft_frame (missing ones are 0). Returns (X complex64[n_xslots, 77, 1536] in nominal
    carrier order, unwritten rows holding the 0xFF fill bit for bit; null complex64[n_frames, 2048] or None)."""
    ctx = ctx or default_context()
    dt = {FMT_CF32: np.complex64, FMT_U8: np.uint8, FMT_I16: np.int16}.get(fmt, np.uint8)
    recs = [_np(r, dt).reshape(-1) for r in recordings]
    n_rec = np.array([r.size if fmt == FMT_CF32 else r.size // 2 for r in recs], np.int64)
    buf = np.concatenate(recs) if recs else np.zeros(1, dt)
    fr = (_lib.FftFrameC * max(len(frames), 1))(*[_lib.FftFrameC(**f) for f in frames])
    raw = np.empty((n_xslots, 77, 768, 4), np.float32)
    null = np.empty((len(frames), 2048), np.complex64) if with_null else None
    ctx.check(ctx.lib.dabstar_fft_frames(ctx.h, _ptr(buf), int(fmt), _ptr(n_rec), len(recs), fr, len(frames), int(n_xslots), int(max_ctas_per_sm),
                                         _ptr(raw), _ptr(null) if with_null else None, MEM_HOST), "dabstar_fft_frames")
    x = np.empty((n_xslots, 77, 768, 2, 2), np.float32)  # [pair][carrier 2p / 2p + 1][re / im]
    x[..., 0] = raw[..., 0:2]
    x[..., 1] = raw[..., 2:4]
    return x.view(np.complex64).reshape(n_xslots, 77, 1536), null


class ViterbiSpiral:
    """support/viterbi_spiral/viterbi_spiral.h:20 — deconvolve() over a batch of equally long code words."""

    def __init__(self, frame_bits: int, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self.frame_bits = int(frame_bits)

    def deconvolve(self, soft: np.ndarray) -> np.ndarray:
        n_in = 4 * (self.frame_bits + 6)
        soft = _np(soft, np.int16).reshape(-1, n_in)
        n = soft.shape[0]
        bits = np.zeros((n, self.frame_bits), np.uint8)
        soft_off = (np.arange(n, dtype=np.int64) * n_in)
        bits_off = (np.arange(n, dtype=np.int64) * self.frame_bits)
        fb = np.full(n, self.frame_bits, np.int32)
        self.ctx.check(self.ctx.lib.dabstar_viterbi(self.ctx.h, _ptr(soft), _ptr(soft_off), _ptr(fb), n, _ptr(bits), _ptr(bits_off), MEM_HOST), "dabstar_viterbi")
        return bits


def viterbi_ragged(ctx: Context, soft_list: list[np.ndarray], frame_bits: list[int]) -> list[np.ndarray]:
    """dabstar_viterbi on code words of different lengths in one launch."""
    soft = np.concatenate([_np(s, np.int16).ravel() for s in soft_list]) if soft_list else np.zeros(0, np.int16)
    fb = np.asarray(frame_bits, np.int32)
    soft_off = np.concatenate([[0], np.cumsum(4 * (fb.astype(np.int64) + 6))[:-1]]).astype(np.int64) if len(fb) else np.zeros(0, np.int64)
    bits_off = np.concatenate([[0], np.cumsum(fb.astype(np.int64))[:-1]]).astype(np.int64) if len(fb) else np.zeros(0, np.int64)
    bits = np.zeros(int(fb.sum()), np.uint8)
    ctx.check(ctx.lib.dabstar_viterbi(ctx.h, _ptr(soft), _ptr(soft_off), _ptr(fb), len(fb), _ptr(bits), _ptr(bits_off), MEM_HOST), "dabstar_viterbi")
    return [bits[o:o + n] for o, n in zip(bits_off, fb)]


class Protection:
    """protection/protection.h:44 (EepProtection / UepProtection): depuncture + Viterbi."""

    def __init__(self, short_form: int, bit_rate: int, prot_level: int, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self.short_form, self.bit_rate, self.prot_level = int(short_form), int(bit_rate), int(prot_level)

    def addresses(self) -> np.ndarray:
        cap = 4 * 24 * self.bit_rate + 24
        a = np.zeros(cap, np.int32)
        n = self.ctx.check(self.ctx.lib.dabstar_protection_addresses(self.ctx.h, self.short_form, self.bit_rate, self.prot_level, _ptr(a), cap),
                           "dabstar_protection_addresses")
        return a[:n].copy()

    def deconvolve(self, soft: np.ndarray, size_cu: int) -> np.ndarray:
        soft = _np(soft, np.int16).reshape(-1, size_cu * 64)
        out = np.zeros((soft.shape[0], 24 * self.bit_rate), np.uint8)
        self.ctx.check(self.ctx.lib.dabstar_protection_deconvolve(self.ctx.h, self.short_form, self.bit_rate, self.prot_level, size_cu, _ptr(soft),
                                                                  soft.shape[0], _ptr(out), MEM_HOST), "dabstar_protection_deconvolve")
        return out


class TiiDetector:
    """ofdm/tii_detector.h:30-45 for n recordings at once (one detector each)."""

    def __init__(self, n_detectors: int = 1, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self.n = int(n_detectors)
        self.h = c_p()
        self.ctx.check(self.ctx.lib.dabstar_tii_create(self.ctx.h, self.n, ctypes.byref(self.h)), "dabstar_tii_create")

    def __del__(self):
        try:
            if self.h:
                self.ctx.lib.dabstar_tii_destroy(self.h)
        except Exception:
            pass

    def reset(self):
        self.ctx.check(self.ctx.lib.dabstar_tii_reset(self.h), "dabstar_tii_reset")

    def set_detect_collisions(self, on: bool, sub_id: int = 0):
        self.ctx.check(self.ctx.lib.dabstar_tii_set_collisions(self.h, int(on), int(sub_id)), "dabstar_tii_set_collisions")

    def add_to_tii_buffer(self, fft: np.ndarray):
        """fft: complex64[n_detectors, n_symbols, 2048] (or [n_symbols, 2048] for a single detector): null-symbol spectra, fft order."""
        fft = _np(fft, np.complex64).reshape(self.n, -1, 2048)
        self.ctx.check(self.ctx.lib.dabstar_tii_add(self.h, _ptr(fft), fft.shape[1], MEM_HOST), "dabstar_tii_add")

    def process_tii_data(self, threshold_db: int, cap: int = 128) -> list[list[tuple]]:
        """Per detector: [(main_id, sub_id, strength, phase_deg, non_etsi), ...], strongest first."""
        out = (_lib.TiiResultC * (self.n * cap))()
        cnt = np.zeros(self.n, np.int32)
        self.ctx.check(self.ctx.lib.dabstar_tii_process(self.h, int(threshold_db), out, cap, _ptr(cnt)), "dabstar_tii_process")
        return [[(r.main_id, r.sub_id, r.strength, r.phase_deg, r.non_etsi) for r in out[d * cap:d * cap + min(int(cnt[d]), cap)]] for d in range(self.n)]

    def decoded(self, detector: int = 0) -> np.ndarray:
        out = np.zeros(768, np.complex64)
        self.ctx.check(self.ctx.lib.dabstar_tii_decoded(self.h, detector, _ptr(out)), "dabstar_tii_decoded")
        return out


class FicDecoder:
    """decoder/fic_decoder.h:49-58 (the member DabProcessor calls mFicHandler)."""

    def __init__(self, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self.ratio = 0

    def process_frames(self, soft: np.ndarray):
        """soft: int16[n, >=9216] (symbols 1..3 first). Returns fib_bits[n,3072], crc_ok[n,12], ber[n,4,2], ratio_percent[n]."""
        soft = _np(soft, np.int16)
        soft = soft.reshape(soft.shape[0], -1)
        n, stride = soft.shape
        bits = np.zeros((n, 3072), np.uint8)
        crc = np.zeros((n, 12), np.uint8)
        ber = np.zeros((n, 4, 2), np.int32)
        self.ctx.check(self.ctx.lib.dabstar_fic_decode(self.ctx.h, _ptr(soft), ctypes.c_int64(stride), n, _ptr(bits), _ptr(crc), _ptr(ber), MEM_HOST), "dabstar_fic_decode")
        ratio = np.zeros(n, np.int32)
        for i in range(n):  # saturating success counter (fic_decoder.cpp:247-259)
            for ok in crc[i]:
                self.ratio = min(10, self.ratio + 1) if ok else max(0, self.ratio - 1)
            ratio[i] = self.ratio * 10
        return bits, crc, ber, ratio

    def get_fic_decode_ratio_percent(self) -> int:
        return self.ratio * 10


FicHandler = FicDecoder


class Backend:
    """backend/backend.h:60 for one sub-channel over consecutive CIFs."""

    def __init__(self, desc: SubChannel, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self.desc = desc

    def process(self, cifs: np.ndarray) -> np.ndarray:
        cifs = _np(cifs, np.int16).reshape(-1, 55296)
        n_out = max(0, cifs.shape[0] - 16)
        out = np.zeros((n_out, 24 * self.desc.bit_rate), np.uint8)
        sc = SubCh(*self.desc.as_row())
        self.ctx.check(self.ctx.lib.dabstar_backend_process(self.ctx.h, ctypes.byref(sc), _ptr(cifs), cifs.shape[0], _ptr(out), MEM_HOST), "dabstar_backend_process")
        return out


class OfdmDecoder:
    """ofdm/ofdm_decoder.h:63-73 over whole frames."""

    def __init__(self, soft_bit_type: int = 0, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self.soft_bit_type = soft_bit_type
        self.st = c_p()
        self.ctx.check(self.ctx.lib.dabstar_ofdm_state_create(self.ctx.h, ctypes.byref(self.st)), "dabstar_ofdm_state_create")

    def __del__(self):
        try:
            if self.st:
                self.ctx.lib.dabstar_ofdm_state_destroy(self.ctx.h, self.st)
        except Exception:
            pass

    def reset(self):
        self.ctx.check(self.ctx.lib.dabstar_ofdm_state_reset(self.ctx.h, self.st), "dabstar_ofdm_state_reset")

    def set_soft_bit_gen_type(self, t: int):
        self.soft_bit_type = int(t)

    def state(self, which: int) -> np.ndarray:
        out = np.zeros(2 if which == 5 else 1536, np.float32)
        self.ctx.check(self.ctx.lib.dabstar_ofdm_state_get(self.ctx.h, self.st, which, _ptr(out)), "dabstar_ofdm_state_get")
        return out

    QUALITY = ("mer_db", "snr_db", "mean_value", "mean_power_overall", "noise_power", "sigma_freq_corr")

    def quality(self) -> dict:
        """SLcdData figures (ofdm_decoder.h:53-61) from the current state."""
        out = np.zeros(6, np.float32)
        self.ctx.check(self.ctx.lib.dabstar_ofdm_state_quality(self.ctx.h, self.st, _ptr(out)), "dabstar_ofdm_state_quality")
        return dict(zip(self.QUALITY, (float(v) for v in out)))

    def decode_frames(self, fft: np.ndarray, clock_err: np.ndarray | None = None, null_is_tii: np.ndarray | None = None,
                      quality: bool = False) -> np.ndarray | tuple[np.ndarray, np.ndarray]:
        """fft: complex64[n, 77, 2048] (symbol 0, symbols 1..75, null). Returns int16[n, 75, 3072]; with quality, also
        float32[n, 6] in QUALITY order: row f is quality() after frame f's null symbol (sigma_freq_corr 0)."""
        fft = _np(fft, np.complex64).reshape(-1, 77, 2048)
        n = fft.shape[0]
        ce = _np(clock_err if clock_err is not None else np.zeros(n), np.float32)
        tii = _np(null_is_tii if null_is_tii is not None else np.zeros(n), np.uint8)
        soft = np.zeros((n, 75, 3072), np.int16)
        if not quality:
            self.ctx.check(self.ctx.lib.dabstar_ofdm_decode_frames(self.ctx.h, self.st, _ptr(fft), n, _ptr(ce), _ptr(tii), self.soft_bit_type, _ptr(soft), MEM_HOST),
                           "dabstar_ofdm_decode_frames")
            return soft
        q = np.zeros((n, 6), np.float32)
        self.ctx.check(self.ctx.lib.dabstar_ofdm_decode_frames_quality(self.ctx.h, self.st, _ptr(fft), n, _ptr(ce), _ptr(tii), self.soft_bit_type, _ptr(soft),
                                                                       MEM_HOST, _ptr(q)), "dabstar_ofdm_decode_frames_quality")
        return soft, q


@dataclass
class RecordingResult:
    n_frames: int
    info: list
    fib_bits: np.ndarray    # uint8[n_frames, 3072]
    fic_valid: np.ndarray   # uint8[n_frames, 4]
    msc: dict               # sub_ch_id -> uint8[n_logical_frames, 24*bitRate]
    counters: np.ndarray    # int64[8]

    @property
    def n_good_fibs(self) -> int:
        return int(self.counters[0])


class DabProcessor:
    """main/dab_processor.h:71 for a batch of recordings (one reference DabProcessor per recording, in lock step)."""

    def __init__(self, n_recordings: int = 1, input_format: int = FMT_U8, soft_bit_type: int = 0, sync_threshold: float = 3.0,
                 strongest_peak: bool = False, scan_mode: bool = False, max_window: int = 0, upload_chunk_frames: int = 0,
                 ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self.n = int(n_recordings)
        self.cfg = DecoderCfg(input_format, soft_bit_type, sync_threshold, int(strongest_peak), int(scan_mode), 1, max_window, upload_chunk_frames)
        self.h = c_p()
        self.ctx.check(self.ctx.lib.dabstar_decoder_create(self.ctx.h, ctypes.byref(self.cfg), self.n, ctypes.byref(self.h)), "dabstar_decoder_create")
        self.subch: list[list[SubChannel]] = [[] for _ in range(self.n)]
        self.auto: dict[int, bool] = {}

    def __del__(self):
        try:
            if self.h:
                self.ctx.lib.dabstar_decoder_destroy(self.h)
        except Exception:
            pass

    def set_audio_channel(self, recording: int, subch: list[SubChannel]):
        """DabProcessor::set_audio_channel for every entry (start_frame = frame in which the Backend is created)."""
        arr = (SubCh * max(len(subch), 1))(*[SubCh(*s.as_row()) for s in subch])
        self.ctx.check(self.ctx.lib.dabstar_decoder_set_subchannels(self.h, recording, arr, len(subch)), "dabstar_decoder_set_subchannels")
        self.subch[recording] = list(subch)

    def set_auto_config(self, recording: int, enable: bool = True, tii_null_symbols: bool = False):
        """Take the recording's sub-channels and CIF counter from its own FIC (FIG 0/0, 0/1) instead of set_audio_channel.
        tii_null_symbols: also what DabProcessor does with a real FIB decoder behind get_cif_count(): null symbols whose CIF counter
        has (count & 7) >= 4 are TII symbols and leave the null power alone (costs a second pass over the recording)."""
        self.ctx.check(self.ctx.lib.dabstar_decoder_set_auto_config(self.h, recording, (2 if tii_null_symbols else 1) if enable else 0), "dabstar_decoder_set_auto_config")
        self.auto[recording] = bool(enable)

    def sub_channels(self, recording: int) -> list[SubChannel]:
        n = self.ctx.check(self.ctx.lib.dabstar_decoder_subchannels(self.h, recording, None, 0), "dabstar_decoder_subchannels")
        arr = (SubCh * max(n, 1))()
        self.ctx.lib.dabstar_decoder_subchannels(self.h, recording, arr, n)
        return [SubChannel(a.sub_ch_id, a.start_cu, a.size_cu, a.short_form, a.prot_level, a.bit_rate, a.start_frame) for a in arr[:n]]

    def ensemble(self, recording: int) -> _lib.EnsembleInfoC:
        e = _lib.EnsembleInfoC()
        self.ctx.check(self.ctx.lib.dabstar_decoder_ensemble(self.h, recording, ctypes.byref(e)), "dabstar_decoder_ensemble")
        return e

    def start_eti_generator(self, recording: int, cif_count_hi: int = 0, cif_count_lo: int = 0):
        """DabProcessor::start_eti_generator (dab_processor.cpp:529-546): the next run also produces the ETI(NI) stream of
        this recording with every sub-channel set through set_audio_channel; see eti()."""
        self.ctx.check(self.ctx.lib.dabstar_decoder_enable_eti(self.h, recording, 1, cif_count_hi, cif_count_lo), "dabstar_decoder_enable_eti")

    def stop_eti_generator(self, recording: int):
        self.ctx.check(self.ctx.lib.dabstar_decoder_enable_eti(self.h, recording, 0, 0, 0), "dabstar_decoder_enable_eti")

    def eti(self, recording: int) -> np.ndarray:
        """ETI(NI) frames of the last run, uint8[n_frames, 6144] (what EtiGenerator writes to its file)."""
        n = int(self.ctx.check(self.ctx.lib.dabstar_decoder_eti_size(self.h, recording), "dabstar_decoder_eti_size"))
        buf = np.zeros(n, np.uint8)
        if n:
            self.ctx.lib.dabstar_decoder_eti_copy(self.h, recording, _ptr(buf), ctypes.c_int64(n))
        return buf.reshape(-1, 6144)

    # ---- long recordings: segments inside a run, chunks of a stream across runs (include/dabstar_b200.h, "long recordings")
    def set_segmentation(self, segment_frames: int, warmup_frames: int = 18):
        """A verified window of >= 2 x segment_frames frames of one recording is demapped as parallel segments, each warm-started
        warmup_frames early (OfdmDecoder's per-carrier IIRs, ofdm_decoder.cpp:182-251, are the only state approximated)."""
        self.ctx.check(self.ctx.lib.dabstar_decoder_set_segmentation(self.h, int(segment_frames), int(warmup_frames)), "dabstar_decoder_set_segmentation")

    def set_streaming(self, enable: bool = True):
        """Runs decode chunks of a longer stream: an incomplete trailing frame is left for the next chunk (see consumed())."""
        self.ctx.check(self.ctx.lib.dabstar_decoder_set_streaming(self.h, int(enable)), "dabstar_decoder_set_streaming")

    def consumed(self, recording: int) -> int:
        """Stream index of the first sample the decoder has not consumed."""
        return int(self.ctx.check(self.ctx.lib.dabstar_decoder_consumed(self.h, recording), "dabstar_decoder_consumed"))

    def warmup_frames(self, recording: int) -> int:
        return int(self.ctx.check(self.ctx.lib.dabstar_decoder_warmup_frames(self.h, recording), "dabstar_decoder_warmup_frames"))

    def export_state(self, recording: int) -> np.ndarray:
        """Everything the stream's next chunk depends on (DabProcessor's loops, OfdmDecoder state, 16 CIFs of soft bits) as bytes."""
        n = int(self.ctx.check(self.ctx.lib.dabstar_decoder_state_size(self.h, recording), "dabstar_decoder_state_size"))
        blob = np.zeros(n, np.uint8)
        self.ctx.check(self.ctx.lib.dabstar_decoder_export_state(self.h, recording, _ptr(blob), ctypes.c_int64(n)), "dabstar_decoder_export_state")
        return blob

    def import_state(self, recording: int, blob: np.ndarray, lead_samples: int = 0):
        """The recording's next run continues the stream `blob` was exported from; its input must start lead_samples before
        the exported consumed() position."""
        blob = np.ascontiguousarray(blob, np.uint8)
        self.ctx.check(self.ctx.lib.dabstar_decoder_import_state(self.h, recording, _ptr(blob), ctypes.c_int64(blob.size), ctypes.c_int64(lead_samples)),
                       "dabstar_decoder_import_state")

    def run_ptrs(self, ptrs: list[int], n_samples: list[int], mem: int) -> float:
        """Decode complete recordings given raw pointers. Returns the device time in ms (CUDA events)."""
        p = (c_p * self.n)(*[c_p(x) for x in ptrs])
        ns = (ctypes.c_int64 * self.n)(*n_samples)
        self.ctx.check(self.ctx.lib.dabstar_decoder_run(self.h, p, ns, mem), "dabstar_decoder_run")
        return float(self.ctx.lib.dabstar_decoder_last_ms(self.h))

    def prepared(self, ptrs: list[int], n_samples: list[int], mem: int):
        """run_ptrs with the argument arrays built once: returns a callable that decodes the same buffers again (a caller that
        decodes in a loop, e.g. bench.py, keeps the ctypes marshalling out of its timed region)."""
        p = (c_p * self.n)(*[c_p(x) for x in ptrs])
        ns = (ctypes.c_int64 * self.n)(*n_samples)
        run, check, h = self.ctx.lib.dabstar_decoder_run, self.ctx.check, self.h

        def call():
            check(run(h, p, ns, mem), "dabstar_decoder_run")
        return call

    def run(self, recordings: list[np.ndarray]) -> float:
        """recordings: host arrays (uint8[n,2] / int16[n,2] / complex64[n]) in the configured input format."""
        dt = {FMT_U8: np.uint8, FMT_I16: np.int16, FMT_CF32: np.complex64}[self.cfg.input_format]
        arrs = [_np(r, dt) for r in recordings]
        self._keep = arrs
        n = [a.shape[0] for a in arrs]
        return self.run_ptrs([a.ctypes.data for a in arrs], n, MEM_HOST)

    def run_files(self, raws: list[np.ndarray], fmt: SampleFormat) -> float:
        """Recordings in any file sample format: layouts the FFT kernel does not read natively are first converted to
        complex float on the device (dabstar_ingest_convert); the decoder must have been created with FMT_CF32 then."""
        nat = fmt.native()
        if nat is not None and nat == self.cfg.input_format:
            dt = {FMT_U8: np.uint8, FMT_I16: np.int16, FMT_CF32: np.complex64}[nat]
            flat = [np.ascontiguousarray(r).view(np.uint8).reshape(-1).view(dt) for r in raws]
            return self.run([f if nat == FMT_CF32 else f.reshape(-1, 2) for f in flat])
        if self.cfg.input_format != FMT_CF32:
            raise DabstarError("run_files with a converted sample format needs a decoder created with input_format=FMT_CF32")
        return self.run([self.ctx.ingest_convert(r, fmt) for r in raws])

    def result(self, recording: int) -> RecordingResult:
        lib = self.ctx.lib
        nf = self.ctx.check(lib.dabstar_decoder_n_frames(self.h, recording), "dabstar_decoder_n_frames")
        info = (FrameInfo * max(nf, 1))()
        lib.dabstar_decoder_frame_info(self.h, recording, info, nf)
        bits = np.zeros((nf, 3072), np.uint8)
        valid = np.zeros((nf, 4), np.uint8)
        lib.dabstar_decoder_fib_bits(self.h, recording, _ptr(bits), _ptr(valid))
        msc = {}
        for s in (self.sub_channels(recording) if self.auto.get(recording) else self.subch[recording]):
            n = int(lib.dabstar_decoder_msc_size(self.h, recording, s.sub_ch_id))
            buf = np.zeros(n, np.uint8)
            if n:
                lib.dabstar_decoder_msc_copy(self.h, recording, s.sub_ch_id, _ptr(buf), ctypes.c_int64(n))
            msc[s.sub_ch_id] = buf.reshape(-1, 24 * s.bit_rate)
        cnt = np.zeros(8, np.int64)
        lib.dabstar_decoder_counters(self.h, recording, _ptr(cnt))
        return RecordingResult(nf, list(info)[:nf], bits, valid, msc, cnt)

    def n_frames(self, recording: int) -> int:
        return int(self.ctx.check(self.ctx.lib.dabstar_decoder_n_frames(self.h, recording), "dabstar_decoder_n_frames"))

    def counters(self, recording: int) -> np.ndarray:
        """dabstar_decoder_counters: [good FIBs, time syncs, time-sync failures, samples consumed, windows run, windows cut, frames
        decoded, frames through the heavy pass] of the last run(), without copying the decoded bits."""
        cnt = np.zeros(8, np.int64)
        self.ctx.check(self.ctx.lib.dabstar_decoder_counters(self.h, recording, _ptr(cnt)), "dabstar_decoder_counters")
        return cnt

    def frame_positions(self, recording: int) -> np.ndarray:
        """Stream index of symbol 0 of every decoded frame."""
        nf = self.n_frames(recording)
        info = (FrameInfo * max(nf, 1))()
        self.ctx.lib.dabstar_decoder_frame_info(self.h, recording, info, nf)
        return np.array([info[i].sym0_pos for i in range(nf)], np.int64)

    def set_tii_processing(self, recording: int, on: bool = True, frames_to_count: int = 5, threshold_db: int = 8, collisions: bool = False, sub_id: int = 0):
        """DabProcessor::set_tii_processing / set_tii_threshold / set_tii_collisions / set_tii_sub_id (+ ProcessParams::tiiFramesToCount);
        needs set_auto_config (the CIF counter decides which null symbols carry TII)."""
        self.ctx.check(self.ctx.lib.dabstar_decoder_enable_tii(self.h, recording, int(on), int(frames_to_count), int(threshold_db), int(collisions), int(sub_id)),
                       "dabstar_decoder_enable_tii")

    def tii_events(self, recording: int, cap: int = 128) -> list[tuple[int, list[tuple]]]:
        """[(frame, [(main_id, sub_id, strength, phase_deg, non_etsi), ...]), ...]: what signal_show_tii would have carried, per search."""
        n = self.ctx.check(self.ctx.lib.dabstar_decoder_tii_events(self.h, recording), "dabstar_decoder_tii_events")
        out = []
        for e in range(n):
            buf = (_lib.TiiResultC * cap)()
            fr = ctypes.c_int32(0)
            k = self.ctx.check(self.ctx.lib.dabstar_decoder_tii_results(self.h, recording, e, buf, cap, ctypes.byref(fr)), "dabstar_decoder_tii_results")
            out.append((fr.value, [(r.main_id, r.sub_id, r.strength, r.phase_deg, r.non_etsi) for r in buf[:min(k, cap)]]))
        return out

    def fib_packed(self, recording: int) -> np.ndarray:
        """The recording's FIBs packed 8 bits per byte (uint8[n_frames, 12, 32]), as they come back from the device."""
        nf = self.ctx.check(self.ctx.lib.dabstar_decoder_n_frames(self.h, recording), "dabstar_decoder_n_frames")
        out = np.zeros((nf, 12, 32), np.uint8)
        self.ctx.check(self.ctx.lib.dabstar_decoder_fib_packed(self.h, recording, _ptr(out)), "dabstar_decoder_fib_packed")
        return out

    def quality(self, recording: int) -> dict:
        """SLcdData figures (MER, SNR, ...) of a recording's OFDM decoder at the end of the last run()."""
        out = np.zeros(6, np.float32)
        self.ctx.check(self.ctx.lib.dabstar_decoder_quality(self.h, recording, _ptr(out)), "dabstar_decoder_quality")
        return dict(zip(OfdmDecoder.QUALITY, (float(v) for v in out)))

    def set_frame_quality(self, on: bool = True):
        """Capture quality() for every frame of the next runs (see frame_quality); off by default."""
        self.ctx.check(self.ctx.lib.dabstar_decoder_set_frame_quality(self.h, int(on)), "dabstar_decoder_set_frame_quality")

    def frame_quality(self, recording: int) -> np.ndarray:
        """float32[n_frames, 6] in OfdmDecoder.QUALITY order: row f is quality() as it would have been had the recording ended
        after frame f (the last run must have had set_frame_quality on)."""
        nf = self.n_frames(recording)
        out = np.zeros((nf, 6), np.float32)
        self.ctx.check(self.ctx.lib.dabstar_decoder_frame_quality(self.h, recording, _ptr(out), nf), "dabstar_decoder_frame_quality")
        return out

    STAGES = ("time_sync", "prs_corr", "cp_corr", "coarse_afc", "ingest_fft", "demap", "fic_viterbi", "msc_viterbi")

    def stage_ms(self) -> dict:
        """Device milliseconds and launch counts per kernel family of the last run()."""
        ms = (ctypes.c_double * 8)()
        ln = (ctypes.c_int64 * 8)()
        self.ctx.check(self.ctx.lib.dabstar_decoder_stage_ms(self.h, ms, ln), "dabstar_decoder_stage_ms")
        return {n: (ms[i], int(ln[i])) for i, n in enumerate(self.STAGES)}

    def msc_kernel_ms(self) -> tuple[float, float]:
        """(gather, trellis) device milliseconds of the MSC pass of the last run()."""
        a, b = ctypes.c_double(0), ctypes.c_double(0)
        self.ctx.check(self.ctx.lib.dabstar_decoder_msc_kernel_ms(self.h, ctypes.byref(a), ctypes.byref(b)), "dabstar_decoder_msc_kernel_ms")
        return a.value, b.value

    def heavy_ms(self, with_fic: bool = True) -> float:
        """Device milliseconds of the FFT + demap (+ FIC) passes of the last run(), one span per window."""
        return float(self.ctx.lib.dabstar_decoder_heavy_ms(self.h, int(with_fic)))

    def soft_bits(self, recording: int, frame: int) -> np.ndarray:
        out = np.zeros((75, 3072), np.int16)
        self.ctx.check(self.ctx.lib.dabstar_decoder_soft_bits(self.h, recording, frame, _ptr(out)), "dabstar_decoder_soft_bits")
        return out
