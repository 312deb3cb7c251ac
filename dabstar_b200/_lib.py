"""Loader of the C-ABI library (include/dabstar_b200.h). There is no fallback: if the CUDA library is missing or
no CUDA device is present, the product path raises."""
from __future__ import annotations

import ctypes
import os

from . import build

c_p = ctypes.c_void_p


class DabstarError(RuntimeError):
    pass


class SubCh(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("sub_ch_id", "start_cu", "size_cu", "short_form", "prot_level", "bit_rate", "start_frame")]


class DecoderCfg(ctypes.Structure):
    _fields_ = [("input_format", ctypes.c_int32), ("soft_bit_type", ctypes.c_int32), ("sync_threshold", ctypes.c_float),
                ("strongest_peak", ctypes.c_int32), ("scan_mode", ctypes.c_int32), ("keep_soft_bits", ctypes.c_int32),
                ("max_window", ctypes.c_int32), ("upload_chunk_frames", ctypes.c_int32)]


class FrameInfo(ctypes.Structure):
    _fields_ = [("sym0_pos", ctypes.c_int64), ("start_index", ctypes.c_int32), ("fbb_sym0", ctypes.c_float),
                ("fbb_data", ctypes.c_float), ("fbb_null", ctypes.c_float), ("fsync", ctypes.c_float),
                ("phase_cp", ctypes.c_float), ("clock_err", ctypes.c_float), ("fic_ratio_before", ctypes.c_int32),
                ("fic_ratio_after", ctypes.c_int32), ("fic_valid", ctypes.c_uint8 * 4)]


class SampleFormatC(ctypes.Structure):
    _fields_ = [("container", ctypes.c_int32), ("bits_per_channel", ctypes.c_int32), ("msb_first", ctypes.c_int32), ("iq_order", ctypes.c_int32)]


class TiiResultC(ctypes.Structure):
    _fields_ = [("main_id", ctypes.c_int32), ("sub_id", ctypes.c_int32), ("strength", ctypes.c_float), ("phase_deg", ctypes.c_float), ("non_etsi", ctypes.c_int32)]


class DcIqStateC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_float) for n in ("mean_i", "mean_q", "mean_ii", "mean_qq", "mean_iq")]


class FileInfoC(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int32), ("reader", ctypes.c_int32), ("sample_rate", ctypes.c_int32), ("n_channels", ctypes.c_int32),
                ("fmt", SampleFormatC), ("data_offset", ctypes.c_int64), ("n_samples", ctypes.c_int64), ("frequency_hz", ctypes.c_int32),
                ("reserved", ctypes.c_int32)]


class SuperFrameC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("first_frame", "ok", "rs_errors", "rs_corrections", "fc_corrected", "dac_rate", "sbr_flag",
                                              "aac_channel_mode", "ps_flag", "mpeg_surround", "num_aus")] + [("au_start", ctypes.c_int32 * 7), ("au_state", ctypes.c_int32 * 6)]


class Mp2FrameC(ctypes.Structure):
    _fields_ = [("first_frame", ctypes.c_int32), ("n_frames", ctypes.c_int32), ("status", ctypes.c_int32), ("header", ctypes.c_uint32),
                ("crc_stored", ctypes.c_int32), ("crc_computed", ctypes.c_int32)]


class DataGroupC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("first_frame", "last_frame", "n_packets", "status", "extension_flag", "crc_flag", "segment_flag",
                                              "user_access_flag", "type", "continuity", "repetition", "extension", "segment_last", "segment_number",
                                              "transport_id", "length_indicator", "crc_stored", "crc_computed", "length", "data_start", "data_length",
                                              "reserved")] + [("offset", ctypes.c_int64)]


class PacketStatsC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int64) for n in ("packets", "crc_errors", "bad_length", "cut", "padding", "command", "other_address", "continuity_breaks",
                                              "abandoned", "dropped")] + [("groups", ctypes.c_int64 * 5)]


class PacketCompC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("scid", "sub_ch_id", "packet_address", "dscty", "dg_flag", "ca_org")]


class FecFrameC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("first_slot", "run_slot", "first_frame", "last_frame", "status", "rows_corrected", "rows_failed",
                                              "bytes_corrected", "headers_matched", "reserved")]


class FecSchemeC(ctypes.Structure):
    _fields_ = [("sub_ch_id", ctypes.c_int32), ("scheme", ctypes.c_int32)]


class EnsembleInfoC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("eid", "change_flags", "alarm", "cif_count_hi", "cif_count_lo", "n_subch", "n_components", "restarts")]


class ServiceCompC(ctypes.Structure):
    _fields_ = [("sid", ctypes.c_uint32)] + [(n, ctypes.c_int32) for n in ("comp_index", "tmid", "type", "sub_ch_id", "primary", "ca_flag")]


class FftFrameC(ctypes.Structure):
    _fields_ = [("sym0", ctypes.c_int64), ("eval", ctypes.c_int64)] + [(n, ctypes.c_int32) for n in (
        "rec", "xslot", "f_sym0", "ph_eval", "f_data", "ph_data", "f_null", "ph_null", "n_syms", "reserved")]


# every symbol include/dabstar_b200.h declares: (name, restype)
EXPORTS = [
    ("dabstar_create", ctypes.c_int), ("dabstar_destroy", None), ("dabstar_last_error", ctypes.c_char_p),
    ("dabstar_abi_version", ctypes.c_int), ("dabstar_kernel_launches", ctypes.c_uint64),
    ("dabstar_freq_interleaver", ctypes.c_int), ("dabstar_phase_table", ctypes.c_int), ("dabstar_protection_addresses", ctypes.c_int),
    ("dabstar_ingest_convert", ctypes.c_int), ("dabstar_sample_format_bytes", ctypes.c_int),
    ("dabstar_tii_create", ctypes.c_int), ("dabstar_tii_destroy", None), ("dabstar_tii_reset", ctypes.c_int), ("dabstar_tii_set_collisions", ctypes.c_int),
    ("dabstar_tii_add", ctypes.c_int), ("dabstar_tii_process", ctypes.c_int), ("dabstar_tii_decoded", ctypes.c_int),
    ("dabstar_dc_iq_correct", ctypes.c_int), ("dabstar_file_probe", ctypes.c_int), ("dabstar_resample_count", ctypes.c_int64), ("dabstar_resample_linear", ctypes.c_int64),
    ("dabstar_dabplus_decode", ctypes.c_int),
    ("dabstar_fib_parser_create", ctypes.c_int), ("dabstar_fib_parser_destroy", None), ("dabstar_fib_parser_push", ctypes.c_int),
    ("dabstar_fib_parser_ensemble", ctypes.c_int), ("dabstar_fib_parser_subchannels", ctypes.c_int), ("dabstar_fib_parser_components", ctypes.c_int),
    ("dabstar_fft2048", ctypes.c_int), ("dabstar_viterbi", ctypes.c_int), ("dabstar_protection_deconvolve", ctypes.c_int),
    ("dabstar_fic_decode", ctypes.c_int), ("dabstar_backend_process", ctypes.c_int),
    ("dabstar_ofdm_state_create", ctypes.c_int), ("dabstar_ofdm_state_destroy", None), ("dabstar_ofdm_state_reset", ctypes.c_int),
    ("dabstar_ofdm_state_get", ctypes.c_int), ("dabstar_ofdm_state_quality", ctypes.c_int), ("dabstar_ofdm_decode_frames", ctypes.c_int),
    ("dabstar_ofdm_decode_frames_quality", ctypes.c_int),
    ("dabstar_prs_correlate", ctypes.c_int), ("dabstar_estimate_carrier_offset", ctypes.c_int), ("dabstar_cp_correlate", ctypes.c_int),
    ("dabstar_fft_frames", ctypes.c_int),
    ("dabstar_decoder_create", ctypes.c_int), ("dabstar_decoder_destroy", None), ("dabstar_decoder_set_subchannels", ctypes.c_int),
    ("dabstar_decoder_run", ctypes.c_int), ("dabstar_decoder_n_frames", ctypes.c_int), ("dabstar_decoder_frame_info", ctypes.c_int),
    ("dabstar_decoder_fib_bits", ctypes.c_int), ("dabstar_decoder_fib_packed", ctypes.c_int), ("dabstar_decoder_soft_bits", ctypes.c_int),
    ("dabstar_decoder_msc_size", ctypes.c_int64), ("dabstar_decoder_msc_copy", ctypes.c_int64), ("dabstar_decoder_msc_packed", ctypes.c_int64),
    ("dabstar_decoder_set_auto_config", ctypes.c_int), ("dabstar_decoder_subchannels", ctypes.c_int), ("dabstar_decoder_ensemble", ctypes.c_int),
    ("dabstar_decoder_enable_eti", ctypes.c_int), ("dabstar_decoder_eti_size", ctypes.c_int64), ("dabstar_decoder_eti_copy", ctypes.c_int64),
    ("dabstar_decoder_enable_tii", ctypes.c_int), ("dabstar_decoder_tii_events", ctypes.c_int), ("dabstar_decoder_tii_results", ctypes.c_int),
    ("dabstar_decoder_counters", ctypes.c_int), ("dabstar_decoder_quality", ctypes.c_int), ("dabstar_decoder_last_ms", ctypes.c_double),
    ("dabstar_decoder_set_frame_quality", ctypes.c_int), ("dabstar_decoder_frame_quality", ctypes.c_int),
    ("dabstar_decoder_stage_ms", ctypes.c_int),
    ("dabstar_decoder_set_segmentation", ctypes.c_int), ("dabstar_decoder_set_streaming", ctypes.c_int), ("dabstar_decoder_consumed", ctypes.c_int64),
    ("dabstar_decoder_state_size", ctypes.c_int64), ("dabstar_decoder_export_state", ctypes.c_int64), ("dabstar_decoder_import_state", ctypes.c_int),
    ("dabstar_decoder_warmup_frames", ctypes.c_int64), ("dabstar_decoder_heavy_ms", ctypes.c_double), ("dabstar_decoder_msc_kernel_ms", ctypes.c_int),
    ("dabstar_decoder_components", ctypes.c_int), ("dabstar_decoder_set_dabplus", ctypes.c_int), ("dabstar_decoder_superframes", ctypes.c_int),
    ("dabstar_decoder_superframe_payload", ctypes.c_int64), ("dabstar_decoder_dabplus_ms", ctypes.c_double),
    ("dabstar_decoder_dabplus_windows", ctypes.c_int),
    ("dabstar_mp2_frames", ctypes.c_int), ("dabstar_decoder_set_mp2", ctypes.c_int), ("dabstar_decoder_mp2_frames", ctypes.c_int),
    ("dabstar_decoder_mp2_payload", ctypes.c_int64), ("dabstar_decoder_mp2_ms", ctypes.c_double),
    ("dabstar_packet_groups", ctypes.c_int), ("dabstar_fib_parser_packet_components", ctypes.c_int), ("dabstar_decoder_set_packet", ctypes.c_int),
    ("dabstar_decoder_data_groups", ctypes.c_int), ("dabstar_decoder_data_group_payload", ctypes.c_int64), ("dabstar_decoder_packet_stats", ctypes.c_int),
    ("dabstar_decoder_packet_ms", ctypes.c_double), ("dabstar_decoder_packet_components", ctypes.c_int),
    ("dabstar_packet_fec", ctypes.c_int), ("dabstar_packet_groups_fec", ctypes.c_int), ("dabstar_fib_parser_fec_schemes", ctypes.c_int),
    ("dabstar_decoder_set_packet_fec", ctypes.c_int), ("dabstar_decoder_fec_frames", ctypes.c_int), ("dabstar_decoder_packet_fec_ms", ctypes.c_double),
    ("dabstar_decoder_fec_schemes", ctypes.c_int),
]

_lib = None


def library_path() -> str:
    return build.LIB_CUDA


def load() -> ctypes.CDLL:
    """Loads dabstar_b200/libdabstar_b200.so (building it with nvcc if the sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    path = build.LIB_CUDA
    if not os.path.exists(path):
        path = build.build_cuda()
    try:
        lib = ctypes.CDLL(path)
    except OSError as e:
        raise DabstarError(f"cannot load {path}: {e}. The CUDA extension is required; there is no CPU fallback.") from e
    for name, res in EXPORTS:
        getattr(lib, name).restype = res
    _lib = lib
    return lib
