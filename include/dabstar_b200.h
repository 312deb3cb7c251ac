/* dabstar_b200.h — C ABI of the B200-native DAB Mode-I baseband decode path.
 *
 * The reference (tomneda/DABstar) has no plugin/FFI layer; its boundary for this path is the public C++
 * surface of the classes that DabProcessor drives (SURVEY.md section 8b). Each entry point below names the
 * reference interface it replaces (file:line under /root/reference/src). The reference calls those
 * interfaces once per OFDM symbol; a device boundary has to be batch granular, so every call here takes
 * a batch (frames, symbols or code words) and the C++ facades in dabstar_b200/host/ restore the
 * reference's class names and per-call signatures on top of it.
 *
 * Conventions
 *   - plain pointers and sizes only; `mem` says whether data pointers are host (DABSTAR_MEM_HOST) or
 *     CUDA device pointers on the context's device (DABSTAR_MEM_DEVICE). Small descriptor arrays
 *     (offsets, sub-channel tables) are always host pointers.
 *   - every function returns 0 or a negative DABSTAR_E_* code; nothing throws across the ABI.
 *     dabstar_last_error() gives the text for the last failure on that context.
 *   - a context is single threaded; different contexts are independent; no global mutable state
 *     (unlike viterbi_spiral.cpp:40-41 / eti_generator.cpp:9-24 in the reference).
 *   - calls are synchronous unless stated: results are complete when the function returns.
 *   - there is no CPU fallback: without a CUDA device dabstar_create() fails.
 */
#ifndef DABSTAR_B200_H
#define DABSTAR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DABSTAR_ABI_VERSION 2

enum { DABSTAR_MEM_HOST = 0, DABSTAR_MEM_DEVICE = 1 };
enum { DABSTAR_FMT_CF32 = 0, DABSTAR_FMT_U8 = 1, DABSTAR_FMT_I16 = 2 };
enum
{
  DABSTAR_OK = 0,
  DABSTAR_E_INVALID = -1,   /* bad argument */
  DABSTAR_E_CUDA = -2,      /* CUDA runtime error, see dabstar_last_error */
  DABSTAR_E_NOMEM = -3,
  DABSTAR_E_UNSUPPORTED = -4
};

/* Mode-I constants (common/glob_defs.h:40-55) */
enum
{
  DABSTAR_L = 76, DABSTAR_K = 1536, DABSTAR_TU = 2048, DABSTAR_TG = 504, DABSTAR_TS = 2552, DABSTAR_TN = 2656,
  DABSTAR_TF = 196608, DABSTAR_SYM_BITS = 3072, DABSTAR_CIF_BITS = 55296, DABSTAR_FIC_BITS = 768,
  DABSTAR_FRAME_SOFT = 75 * 3072
};

typedef struct dabstar_ctx dabstar_ctx;

/* ------------------------------------------------------------------------------------------------ context */
/* stream: a cudaStream_t to run on (e.g. torch's current stream), or NULL to create a private one. */
int  dabstar_create(dabstar_ctx ** out, int device, void * stream);
void dabstar_destroy(dabstar_ctx * ctx);
const char * dabstar_last_error(const dabstar_ctx * ctx);
int  dabstar_abi_version(void);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
uint64_t dabstar_kernel_launches(const dabstar_ctx * ctx);

/* ------------------------------------------------------------------------------------------------ tables (init-only rows D0, S4, M3) */
/* FreqInterleaver::map_k_to_fft_bin for k = 0..1535 (ofdm/freq_interleaver.h:50). */
int dabstar_freq_interleaver(dabstar_ctx * ctx, int16_t out[1536]);
/* PhaseTable::mRefTable, 2048 complex floats (ofdm/phasetable.h:51). */
int dabstar_phase_table(dabstar_ctx * ctx, float out_re_im[4096]);
/* EepProtection / UepProtection viterbiBlockAddresses (protection/eep_protection.cpp:43-151,
 * uep_protection.cpp:155-196): destination index of every kept soft bit. Returns the count or <0. */
int dabstar_protection_addresses(dabstar_ctx * ctx, int short_form, int bit_rate, int prot_level, int32_t * addr, int cap);

/* ------------------------------------------------------------------------------------------------ ingest (row I1) */
/* File-reader sample conversion to complex float, as XmlReader::readElements_IQ / _QI / _I / _Q do it
 * (devices/filereaders/xml_filereader/xml_reader.cpp:254-372, 400-545, 547-676, 678-800; scaler = 2^(bits-1),
 * xml_reader.cpp:43-51,256-257), RawReader (raw_files/raw_reader.cpp:66-70: u8, (v - 127.38) / 128) and WavReader
 * (wav_files/wav_reader.cpp:164: libsndfile float read of 16-bit PCM = int16 / 32768).
 *   int8: v / 127 (IQ order in float, the other orders through double as the reference writes them);
 *   uint8: (v - 127.38) / 128; int16 / int24 / int32: v / 2^(bits_per_channel - 1), the scaler held in an i32 as the
 *   reference does, so 32 bits per channel divide by -2^31; float32: as is.
 * The decoder's native input formats (DABSTAR_FMT_U8 / I16 / CF32) are converted inside the FFT kernel; every
 * other combination goes through this call first and is then decoded as DABSTAR_FMT_CF32.
 * Reference reader defects that are NOT reproduced (they read the wrong byte, a constant, or leave the channels unswapped; each
 * is pinned against the reference's own XmlReader thread in tests/test_ingest_formats.py): uint8 with QI order indexes the table
 * with the loop counter (xml_reader.cpp:421), int8 with Q_Only sets the real part to 127 (:690), MSB int24 takes one byte from
 * offset 4*i+4 (:309, and :456 in the QI branch, which also sign-extends with 0x7F000000), float32 with QI order does not swap I
 * and Q (:525-543). int8 divides by 127 in IEEE arithmetic; the reference's -ffast-math build multiplies by the reciprocal (1 ulp). */
enum { DABSTAR_CONTAINER_INT8 = 0, DABSTAR_CONTAINER_UINT8 = 1, DABSTAR_CONTAINER_INT16 = 2, DABSTAR_CONTAINER_INT24 = 3,
       DABSTAR_CONTAINER_INT32 = 4, DABSTAR_CONTAINER_FLOAT32 = 5,
       /* RIFF/WAVE files go through libsndfile's float read in the reference (wav_reader.cpp:164): 16 / 24-bit PCM and
        * float equal the XML containers above; 8-bit PCM is (v - 128) / 128 and 32-bit PCM v / 2^31 (little endian) */
       DABSTAR_CONTAINER_UINT8_PCM = 6, DABSTAR_CONTAINER_INT32_PCM = 7 };
enum { DABSTAR_ORDER_IQ = 0, DABSTAR_ORDER_QI = 1, DABSTAR_ORDER_I_ONLY = 2, DABSTAR_ORDER_Q_ONLY = 3 };
typedef struct
{
  int32_t container;        /* DABSTAR_CONTAINER_* */
  int32_t bits_per_channel; /* significant bits (scaler 2^(bits-1)); 0 = the container's width */
  int32_t msb_first;        /* byte order of multi-byte containers: 0 LSB first, 1 MSB first */
  int32_t iq_order;         /* DABSTAR_ORDER_* */
} dabstar_sample_format;
/* src: n_samples elements (pairs, or single values for the *_ONLY orders); dst: n_samples complex floats. */
int dabstar_ingest_convert(dabstar_ctx * ctx, const void * src, const dabstar_sample_format * fmt, int64_t n_samples, float * dst, int mem);
/* Bytes per element of `src` for a format (0 if the format is invalid). */
int dabstar_sample_format_bytes(const dabstar_sample_format * fmt);

/* ------------------------------------------------------------------------------------------------ input containers (next row f4) */
/* What the file readers learn before the first sample (host code, csrc/file_probe.cu):
 *   XML / UFF: XmlDescriptor (xml_filereader/xml_descriptor.cpp:100-242) + XmlFileReader's start offset and sample count
 *              (xml_filereader.cpp:103-126,313-335);
 *   WAV / SDR: WavFileHandler (wav_files/wavfiles.cpp:61-97: 1.536..3.0 MS/s, two channels, PCM 8/16/24/32 or float);
 *   anything else: RawReader (raw_files/raw_reader.cpp:66-70): unsigned 8-bit IQ at 2.048 MS/s, no header.
 * head: the first head_bytes of the file (64 KiB is plenty); file_bytes: its total size. */
enum { DABSTAR_FILE_RAW = 0, DABSTAR_FILE_XML = 1, DABSTAR_FILE_WAV = 2 };
enum { DABSTAR_READER_XML = 0, DABSTAR_READER_WAV = 1 };
typedef struct
{
  int32_t kind;            /* DABSTAR_FILE_* */
  int32_t reader;          /* DABSTAR_READER_*: whose sample-rate conversion applies */
  int32_t sample_rate;     /* Hz */
  int32_t n_channels;
  dabstar_sample_format fmt;
  int64_t data_offset;     /* first byte of the sample data */
  int64_t n_samples;       /* complex samples (single values for the *_ONLY orders) the reader would play */
  int32_t frequency_hz;    /* centre frequency of the first data block (XML), else 0 */
  int32_t reserved;
} dabstar_file_info;
int dabstar_file_probe(const uint8_t * head, int64_t head_bytes, int64_t file_bytes, dabstar_file_info * out);

/* ------------------------------------------------------------------------------------------------ TII detection (next row f4) */
/* TiiDetector (ofdm/tii_detector.h:30-45, tii_detector.cpp) for n_detectors recordings at once, one CTA each. The reference
 * feeds it the FFT of every null symbol whose CIF counter has (count & 7) >= 4 (dab_processor.cpp:273-300), and asks for
 * the transmitter list after tiiFramesToCount of them. Results are sorted by strength, strongest first (equal strengths:
 * by sub id, then main id; the reference leaves that order to std::sort). main_id 99 marks a collision on a comb other
 * than the one set for the detailed search (tii_detector.cpp:462-471). */
typedef struct dabstar_tii dabstar_tii;
typedef struct
{
  int32_t main_id, sub_id;  /* STiiResult (tii_detector.h:14-21) */
  float   strength, phase_deg;
  int32_t non_etsi;
} dabstar_tii_result;
int  dabstar_tii_create(dabstar_ctx * ctx, int n_detectors, dabstar_tii ** out);
void dabstar_tii_destroy(dabstar_tii * t);
int  dabstar_tii_reset(dabstar_tii * t);                                /* TiiDetector::reset on every detector */
int  dabstar_tii_set_collisions(dabstar_tii * t, int on, int sub_id);    /* set_detect_collisions + set_subid_for_collision_search */
/* add_to_tii_buffer: fft = n_detectors x n_symbols x 2048 complex floats (fft order); detector d accumulates its n_symbols spectra */
int  dabstar_tii_add(dabstar_tii * t, const float * fft, int n_symbols, int mem);
/* process_tii_data(threshold_db) on every detector: out = n_detectors x cap results, counts[d] = results of detector d
 * (a count above cap means the list was cut). Host memory. */
int  dabstar_tii_process(dabstar_tii * t, int threshold_db, dabstar_tii_result * out, int cap, int32_t * counts);
/* mDecodedBufferArr of one detector: 768 complex floats (the filtered carrier-pair products) */
int  dabstar_tii_decoded(dabstar_tii * t, int detector, float * out);

/* Sample-rate conversion to 2.048 MS/s as the readers do it when the reference is built without liquid-dsp (the
 * default): per 1 ms block of rate/1000 input samples, 2048 output samples by linear interpolation between neighbours
 * (XmlReader: xml_reader.cpp:70-76,212-231; WavReader: wav_reader.cpp:66-83,196-211; the two differ in table precision
 * and by one sample of delay). in: n_in complex floats; returns the number of complex samples written (whole blocks
 * only; n_in copied unchanged when sample_rate is 2 048 000) or <0. dabstar_resample_count gives that number up front. */
int64_t dabstar_resample_count(int64_t n_in, int sample_rate, int reader);
int64_t dabstar_resample_linear(dabstar_ctx * ctx, const float * in, int64_t n_in, int sample_rate, int reader, float * out, int64_t out_cap, int mem);

/* ------------------------------------------------------------------------------------------------ DC / IQ correction (row I2, optional) */
/* SampleReader::set_dc_and_iq_correction(true, do_iq) (ofdm/sample_reader.h:66, sample_reader.cpp:216-243; off by default in
 * the reference): DC removal by two IIRs (alpha = 1 / 2 048 000) and, with do_iq, the IQ-imbalance correction by three
 * more. A pre-pass over a whole recording of complex floats (in == out allowed); the result is decoded as
 * DABSTAR_FMT_CF32. state: the filter values before the first sample, updated to those after the last (NULL: a fresh
 * SampleReader: 0, 0, 1, 1, 0). The filters are evaluated as scans in double precision, i.e. the recurrences in exact
 * arithmetic. DC removal agrees with the reference's float loop to about 1e-6 of the sample amplitude. With do_iq the
 * reference's meanII / meanQQ start at 1 and move by only ~8 float ulps per sample while they are large, so its round-off
 * is a systematic ~1 % of their decay rate: during the first seconds gainQ (the Q branch) differs by up to a few 1e-3
 * relative from this implementation; the I branch and the settled state agree as for DC removal. */
typedef struct
{
  float mean_i, mean_q, mean_ii, mean_qq, mean_iq; /* sample_reader.h:102-106 */
} dabstar_dciq_state;
int dabstar_dc_iq_correct(dabstar_ctx * ctx, const float * in, int64_t n_samples, int do_iq, dabstar_dciq_state * state, float * out, int mem);

/* ------------------------------------------------------------------------------------------------ stage taps */
/* fftwf_execute on a 2048-point plan (main/dab_processor.cpp:63,201,276,338): n transforms,
 * unnormalised, sign -1 forward / +1 backward, natural order, complex float interleaved. */
int dabstar_fft2048(dabstar_ctx * ctx, const float * in, float * out, int n, int sign, int mem);

/* ViterbiSpiral::deconvolve (support/viterbi_spiral/viterbi_spiral.h:20) for n code words.
 * soft: concatenated int16 inputs, code word i starts at soft_off[i] and holds 4*(frame_bits[i]+6) values;
 * bits: one decoded bit per byte, code word i at bits_off[i], frame_bits[i] bytes. */
int dabstar_viterbi(dabstar_ctx * ctx, const int16_t * soft, const int64_t * soft_off, const int32_t * frame_bits,
                    int n, uint8_t * bits, const int64_t * bits_off, int mem);

/* Protection::deconvolve (protection/protection.h:44) for n logical frames of ONE sub-channel profile:
 * depuncture + Viterbi, no time de-interleaving, no energy dispersal.
 * soft: n fragments of size_cu*64 int16 each (stride = size_cu*64); bits: n x 24*bit_rate bytes. */
int dabstar_protection_deconvolve(dabstar_ctx * ctx, int short_form, int bit_rate, int prot_level, int size_cu,
                                  const int16_t * soft, int n, uint8_t * bits, int mem);

/* FicDecoder::process_block x3 + get_fib_bits (decoder/fic_decoder.h:49-58) for n frames.
 * soft: n x 9216 int16 (symbols 1..3 of each frame, frame stride `frame_stride` int16);
 * fib_bits: n x 3072 bytes (4 FICs x 768, dispersal removed); crc_ok: n x 12 (one per FIB);
 * ber: n x 4 x 2 int32 {compared bits, sign errors} per FIC (ViterbiSpiral::calculate_BER). */
int dabstar_fic_decode(dabstar_ctx * ctx, const int16_t * soft, int64_t frame_stride, int n, uint8_t * fib_bits,
                       uint8_t * crc_ok, int32_t * ber, int mem);

typedef struct
{
  int32_t sub_ch_id;
  int32_t start_cu;
  int32_t size_cu;
  int32_t short_form;  /* 1: UEP, prot_level 1..5; 0: EEP, prot_level 0..3 = 1-A..4-A, 4..7 = 1-B..4-B */
  int32_t prot_level;
  int32_t bit_rate;    /* kbit/s */
  int32_t start_frame; /* frame in which the Backend is created (MscHandler::set_channel) */
} dabstar_subch;

/* Backend::process (backend/backend.h:60) for n_cifs consecutive CIFs and one sub-channel: 16-CIF time
 * de-interleave, depuncture, Viterbi, energy dispersal. cifs: n_cifs x 55296 int16. The Backend is new
 * (zero history) at CIF 0, so CIF r >= 16 emits logical frame r-16: bits holds (n_cifs-16) x 24*bit_rate
 * bytes. Returns the number of logical frames written or <0. */
int dabstar_backend_process(dabstar_ctx * ctx, const dabstar_subch * sc, const int16_t * cifs, int n_cifs,
                            uint8_t * bits, int mem);

/* OfdmDecoder (ofdm/ofdm_decoder.h:63-73) over whole frames for ONE recording.
 * state: opaque per-recording decoder state (the reference's per-carrier IIR vectors, phase reference,
 * mMeanValue), created zeroed as OfdmDecoder() does. */
typedef struct dabstar_ofdm_state dabstar_ofdm_state;
int  dabstar_ofdm_state_create(dabstar_ctx * ctx, dabstar_ofdm_state ** out);
void dabstar_ofdm_state_destroy(dabstar_ctx * ctx, dabstar_ofdm_state * st);
int  dabstar_ofdm_state_reset(dabstar_ctx * ctx, dabstar_ofdm_state * st);                 /* OfdmDecoder::reset */
/* which: 0 integAbsPhase 1 stdDevSq 2 meanPower 3 meanSigmaSq (1536 each, nominal carrier order)
 *        4 nullPower (1536, nominal carrier order k -> bin map_k_to_fft_bin(k)) 5 {meanValue, 0} */
int  dabstar_ofdm_state_get(dabstar_ctx * ctx, dabstar_ofdm_state * st, int which, float * out);
/* What OfdmDecoder reports through signal_show_lcd_data (SLcdData, ofdm/ofdm_decoder.h:53-61; ofdm_decoder.cpp:326-345,
 * _compute_noise_Power :357-371), from the current state:
 * out = { MER dB, SNR dB, mMeanValue, mMeanPowerOvrAll, noise power, sqrt(mMeanSigmaSqFreqCorr) (0 for a bare state) }.
 * mMeanPowerOvrAll is a serial IIR over the carriers of every symbol; the demapper keeps an algebraically equal
 * per-carrier form (csrc/kernels.h), so the figure agrees with the reference to float rounding (1e-4 relative). */
int  dabstar_ofdm_state_quality(dabstar_ctx * ctx, dabstar_ofdm_state * st, float out[6]);
/* fft: n_frames x 77 x 2048 complex float, rows = symbol 0 (store_reference_symbol_0), symbols 1..75
 * (decode_symbol), null symbol (store_null_symbol_without_tii when null_is_tii[f]==0);
 * clock_err: n_frames floats (iClockErr); soft: n_frames x 75 x 3072 int16. */
int  dabstar_ofdm_decode_frames(dabstar_ctx * ctx, dabstar_ofdm_state * st, const float * fft, int n_frames,
                                const float * clock_err, const uint8_t * null_is_tii, int soft_bit_type,
                                int16_t * soft, int mem);
/* The same, and quality: n_frames x 6 host floats, row f = what dabstar_ofdm_state_quality returns after frame f's null
 * symbol (field 5 is 0, as for a bare state). The last row equals dabstar_ofdm_state_quality after the call bit for bit. */
int  dabstar_ofdm_decode_frames_quality(dabstar_ctx * ctx, dabstar_ofdm_state * st, const float * fft, int n_frames,
                                        const float * clock_err, const uint8_t * null_is_tii, int soft_bit_type,
                                        int16_t * soft, int mem, float * quality);

/* PhaseReference::correlate_with_phase_ref_and_find_max_peak (ofdm/phasereference.h:53) for n windows of
 * 2048 complex samples; start_index[i] = peak index or -1. */
int dabstar_prs_correlate(dabstar_ctx * ctx, const float * samples, int n, float threshold, int strongest_peak,
                          int32_t * start_index, int mem);
/* PhaseReference::estimate_carrier_offset_from_sync_symbol_0 (ofdm/phasereference.h:54) for n FFT'd
 * symbols 0; offset_hz[i] = Hz or 100000 (IDX_NOT_FOUND). */
int dabstar_estimate_carrier_offset(dabstar_ctx * ctx, const float * fft, int n, int32_t * offset_hz, int mem);

/* ------------------------------------------------------------------------------------------------ DAB+ outer code */
/* Mp4Processor::add_to_frame for a run of logical frames of one DAB+ sub-channel (backend/audio/mp4processor.cpp:95-334):
 * super-frame synchronisation by Fire code (backend/firecode_checker.cpp), RS(120,110) over the bit_rate/8 interleaved code
 * words (ReedSolomon(8, 0435, 0, 1, 10), backend/reed_solomon.cpp:140-260), Fire-code check with 6-bit burst correction of
 * the decoded header, header fields, access-unit borders and CRCs (backend/crc.cpp:75-96). The AAC decoder stays a CPU
 * consumer of the access units.
 * frame_bits: n_frames x 24*bit_rate bytes, one bit each, exactly what Backend hands to FrameProcessor::add_to_frame
 * (dabstar_decoder_msc_copy). out: one record per super-frame the processor ATTEMPTS, in stream order (at most cap are
 * written); payload: 110*(bit_rate/8) bytes per record, the decoded super-frame (mOutVec) whatever the outcome.
 * Returns the number of attempts or <0. */
typedef struct
{
  int32_t first_frame;      /* index of the super-frame's first logical frame */
  int32_t ok;               /* _process_reed_solomon_frame succeeded: the access units below are handed on */
  int32_t rs_errors, rs_corrections, fc_corrected;
  int32_t dac_rate, sbr_flag, aac_channel_mode, ps_flag, mpeg_surround;
  int32_t num_aus;
  int32_t au_start[7];      /* access unit u occupies payload[au_start[u] .. au_start[u+1]-3], followed by its 2-byte CRC */
  int32_t au_state[6];      /* 0: length check failed (mp4processor.cpp:326), 1: CRC good, 2: CRC error */
} dabstar_superframe;
int dabstar_dabplus_decode(dabstar_ctx * ctx, const uint8_t * frame_bits, int bit_rate, int n_frames, dabstar_superframe * out, int cap,
                           uint8_t * payload, int mem);

/* ------------------------------------------------------------------------------------------------ MPEG layer II audio frames */
/* The audio frames of a run of logical frames of one DAB (MP2) sub-channel (TMId 0, ASCTy 0), checked on the device. A DAB audio
 * frame starts at the first bit of a logical frame and lasts 24 ms at 48 kHz (MPEG-1, one logical frame of 3 * bit_rate bytes) or
 * 48 ms at 24 kHz (MPEG-2 LSF, two logical frames; ETSI EN 300 401 clause 7). Every slot is classified from its 32-bit header
 * (ISO/IEC 11172-3 2.4.1.3) and its CRC-16 (x^16 + x^15 + x^2 + 1, preset 0xFFFF, over header bits 16-31, the bit allocation
 * and the SCFSI; 11172-3 2.4.3.1, allocation tables 11172-3 Annex B Table B.2a / B.2c and 13818-3 Table B.1). Status:
 *   0 OK         valid header, CRC matches
 *   1 NO_HEADER  syncword != 0xFFF, layer != II or protection_bit = 1
 *   2 MISMATCH   sampling_frequency != 01 (48 kHz / 24 kHz), bitrate_index 0 or 15, or the header's rate != the sub-channel's
 *   3 CRC_ERROR  valid header, CRC mismatch
 *   4 CUT        a 24 kHz frame whose second logical frame lies past the end of the run
 * An OK 24 kHz frame is one record covering logical frames i and i + 1; every other slot is a one-frame record. PCM decoding,
 * PAD and the DAB scale-factor CRC are left to the consumer. */
typedef struct
{
  int32_t first_frame;  /* index of the slot's first logical frame */
  int32_t n_frames;     /* logical frames it covers: 2 for an OK 24 kHz frame, else 1 */
  int32_t status;       /* 0..4, above */
  uint32_t header;      /* the slot's first 32 bits, as read */
  int32_t crc_stored, crc_computed; /* crc_check and the CRC over the protected bits; -1 where not reached */
} dabstar_mp2_frame;
/* frame_bits: n_frames x 24*bit_rate bytes, one bit each (dabstar_decoder_msc_copy). out: one record per slot, in stream order
 * (at most cap are written); payload (may be NULL; room for n_frames * 3 * bit_rate bytes): the bytes of the OK frames among
 * those records, concatenated in record order. bit_rate must be a layer II rate (MPEG-1 32..384 or LSF 8..160 kbit/s).
 * Returns the number of records or <0. */
int dabstar_mp2_frames(dabstar_ctx * ctx, const uint8_t * frame_bits, int bit_rate, int n_frames, dabstar_mp2_frame * out, int cap,
                       uint8_t * payload, int mem);

/* ------------------------------------------------------------------------------------------------ packet-mode data */
/* The data groups of one address of a run of logical frames of one packet-mode sub-channel (TMId 3), on the device (ETSI EN 300 401
 * clause 5.3.2 packets, 5.3.3 MSC data groups). Packets of 24, 48, 72 or 96 bytes (length in their first two bits) tile each
 * logical frame of 3 * bit_rate bytes; each carries a 24-bit header (length, continuity index, first / last flags, 10-bit address,
 * command flag, useful data length) and a CRC-16 over header and data field (x^16 + x^12 + x^5 + 1, preset 0xFFFF, complemented:
 * the FIB CRC). A packet is OK, a CRC error, of bad length (useful data length > packet length - 5) or cut (it would run past the
 * end of the logical frame; the rest of that frame is skipped). Address 0 is padding; command packets are counted, not assembled.
 * The CRC-good data packets of the address are assembled in stream order: a packet continues the previous one when its
 * continuity index is the previous one's plus 1 (mod 4); first opens a group (abandoning an open one), single is a group of its
 * own, intermediate keeps an open group only if it continues it, last closes an open group it continues into a record. Any
 * other packet abandons the open group or, without one, is dropped. With DG flag 0 the group is an MSC data group: its header,
 * session header and CRC are parsed and checked (status below); with DG flag 1 it is a RAW record. Sub-channels with packet-mode
 * FEC (FIG 0/14 scheme 1, the RS(204,188) outer code of clause 5.3.5) are decoded with dabstar_packet_groups_fec: their FEC
 * frames are located and corrected first (see dabstar_packet_fec), and the FEC packets are skipped. */
enum { DABSTAR_DG_OK = 0, DABSTAR_DG_NO_CRC = 1, DABSTAR_DG_CRC_ERROR = 2, DABSTAR_DG_MALFORMED = 3, DABSTAR_DG_RAW = 4 };
typedef struct
{
  int32_t first_frame, last_frame; /* logical frames of the group's first and last packet */
  int32_t n_packets;
  int32_t status;                  /* DABSTAR_DG_*: OK (CRC good), NO_CRC (CRC flag 0), CRC_ERROR, MALFORMED (headers do not fit), RAW */
  int32_t extension_flag, crc_flag, segment_flag, user_access_flag; /* data group header; -1 for RAW / where not reached */
  int32_t type, continuity, repetition;
  int32_t extension;               /* extension field, -1 if absent */
  int32_t segment_last, segment_number; /* segment field, -1 if absent */
  int32_t transport_id, length_indicator; /* user access field, -1 if absent */
  int32_t crc_stored, crc_computed;     /* data group CRC, -1 if absent */
  int32_t length;                  /* bytes of the group (the useful data of its packets) */
  int32_t data_start, data_length; /* data field inside the group (RAW: the whole group) */
  int32_t reserved;
  int64_t offset;                  /* first byte of the group in the stream's payload */
} dabstar_data_group;
/* frame_bits: n_frames x 24*bit_rate bytes, one bit each (dabstar_decoder_msc_copy); bit_rate a multiple of 8; address 1..1023.
 * out: one record per data group, in stream order (at most cap are written); payload (may be NULL; room for n_frames * 3 *
 * bit_rate bytes): the groups' bytes, concatenated in record order. Returns the number of records or <0. */
int dabstar_packet_groups(dabstar_ctx * ctx, const uint8_t * frame_bits, int bit_rate, int n_frames, int address, int dg_flag, dabstar_data_group * out,
                          int cap, uint8_t * payload, int mem);
/* per (sub-channel, address) counters of a run */
typedef struct
{
  int64_t packets;            /* CRC-good data packets with the address */
  int64_t crc_errors, bad_length, cut; /* packets of the sub-channel in these classes */
  int64_t padding;            /* CRC-good packets with address 0 */
  int64_t command;            /* CRC-good command packets with the address */
  int64_t other_address;      /* CRC-good packets with another non-zero address */
  int64_t continuity_breaks;  /* packets of the address that do not continue the previous one */
  int64_t abandoned;          /* open groups given up */
  int64_t dropped;            /* intermediate / last packets without an open group */
  int64_t groups[5];          /* groups by status (DABSTAR_DG_*) */
} dabstar_packet_stats;

/* Packet-mode FEC (EN 300 401 clause 5.3.5), on the device. An FEC frame is an Application Data Table of 2256 bytes (94 slots of 24
 * bytes holding whole packets) followed by 9 FEC packets of 24 bytes (2-byte header: length 00, continuity index, first / last
 * flags, address 1022; 22 bytes of RS data), 103 slots that start on any 24-byte slot boundary of the stream. ADT and RS data form
 * a 12 x 204 table filled column by column; each row is an RS(204,188) code word (shortened RS(255,239), field
 * x^8 + x^4 + x^3 + x^2 + 1, roots alpha^0..alpha^15) that corrects up to 8 byte errors. The runs of FEC packets are located slot
 * by slot (dabstar_b200/csrc/pfec.cuh states the rule: at least 6 of the 9 headers must fit, with their first / last flags); a
 * row with more than 8 errors is left as received. */
enum { DABSTAR_FEC_CLEAN = 0, DABSTAR_FEC_CORRECTED = 1, DABSTAR_FEC_PARTIAL = 2, DABSTAR_FEC_INCOMPLETE = 3 };
typedef struct
{
  int32_t first_slot;          /* first 24-byte slot of the frame's ADT in the stream (< 0: the frame is cut by the stream start) */
  int32_t run_slot;            /* first slot of its 9 FEC packets */
  int32_t first_frame, last_frame; /* logical frames of its first and last slot inside the stream */
  int32_t status;              /* DABSTAR_FEC_*: CLEAN, CORRECTED, PARTIAL (some rows failed), INCOMPLETE (cut by the stream's start
                                  or end, or the previous run lies inside its ADT: not corrected) */
  int32_t rows_corrected, rows_failed, bytes_corrected;
  int32_t headers_matched;     /* FEC packet headers of the run that fit (of 9) */
  int32_t reserved;
} dabstar_fec_frame;
/* The FEC pass alone: frame_bits as for dabstar_packet_groups; corrected_bits (may be NULL): the same bits after correction, in the
 * same layout; out: one record per located FEC frame, in stream order (at most cap are written). Returns the number of frames or <0. */
int dabstar_packet_fec(dabstar_ctx * ctx, const uint8_t * frame_bits, int bit_rate, int n_frames, uint8_t * corrected_bits, dabstar_fec_frame * out,
                       int cap, int mem);
/* dabstar_packet_groups with the FEC pass in front: the packets are walked on the corrected bytes, and a packet that starts on a
 * slot of a located FEC-packet run is skipped (it counts in no dabstar_packet_stats field). stats (may be NULL): the stream's
 * counters; fec_out: the FEC frame records (at most fec_cap), *n_fec (may be NULL): their number. Returns the number of groups or <0. */
int dabstar_packet_groups_fec(dabstar_ctx * ctx, const uint8_t * frame_bits, int bit_rate, int n_frames, int address, int dg_flag, dabstar_data_group * out,
                              int cap, uint8_t * payload, dabstar_packet_stats * stats, dabstar_fec_frame * fec_out, int fec_cap, int * n_fec, int mem);

/* ------------------------------------------------------------------------------------------------ multiplex configuration (FIG 0/0, 0/1, 0/2) */
/* The part of FibDecoder the decode path depends on (decoder/fib_decoder.cpp:59-106 process_FIB,
 * fib_decoder_fig0.cpp:89-113 FIG 0/0, :142-227 FIG 0/1, :229-290 FIG 0/2, fib_table.h:51 short-form table): which
 * sub-channels exist (MscHandler::set_channel), the CIF counter and the sub-channel list EtiGenerator frames. Host
 * code; current configuration (C/N = 0) only. A sub-channel that leaves the CIF or overlaps a known one makes the
 * parser drop what it collected, as FibDecoder::_restart_fib_decoding does. */
typedef struct
{
  int32_t eid, change_flags, alarm;
  int32_t cif_count_hi, cif_count_lo;   /* IFibDecoder::get_cif_count(hi, lo) */
  int32_t n_subch, n_components, restarts;
} dabstar_ensemble_info;
typedef struct
{
  uint32_t sid;
  int32_t comp_index;  /* position inside the service's FIG 0/2 entry */
  int32_t tmid;        /* 0 stream audio, 1 stream data, 3 packet data */
  int32_t type;        /* ASCTy (0 MPEG layer II, 63 DAB+) / DSCTy / SCId */
  int32_t sub_ch_id;   /* -1 for packet mode */
  int32_t primary, ca_flag;
} dabstar_service_comp;
typedef struct dabstar_fib_parser dabstar_fib_parser;
int  dabstar_fib_parser_create(dabstar_fib_parser ** out);
void dabstar_fib_parser_destroy(dabstar_fib_parser * p);
/* IFibDecoder::process_FIB (fib_decoder_if.h:81) for n_fibs CRC-good FIBs: 256 bytes each, one bit per byte. */
int  dabstar_fib_parser_push(dabstar_fib_parser * p, const uint8_t * fib_bits, int n_fibs);
/* returns 1 once a FIG 0/0 has been seen, else 0 */
int  dabstar_fib_parser_ensemble(const dabstar_fib_parser * p, dabstar_ensemble_info * out);
/* sub-channels in order of first appearance (start_frame = 0); returns the total count */
int  dabstar_fib_parser_subchannels(const dabstar_fib_parser * p, dabstar_subch * out, int cap);
int  dabstar_fib_parser_components(const dabstar_fib_parser * p, dabstar_service_comp * out, int cap);
/* FIG 0/3 (EN 300 401 clause 6.3.2): where a packet-mode component (SCId, the `type` of its FIG 0/2 TMId 3 entry) is carried.
 * Current configuration only, in order of first appearance; an entry that would cross the end of its FIG is not read (the rest
 * of that FIG is skipped). FIG 0/3 never restarts the parser and leaves the sub-channel and component lists alone. */
typedef struct
{
  int32_t scid, sub_ch_id, packet_address, dscty, dg_flag;
  int32_t ca_org; /* -1 if absent */
} dabstar_packet_comp;
int  dabstar_fib_parser_packet_components(const dabstar_fib_parser * p, dabstar_packet_comp * out, int cap);
/* FIG 0/14 (EN 300 401 clause 6.2.2): the FEC scheme of a packet-mode sub-channel: 0 none, 1 the FEC of clause 5.3.5, 2 and 3
 * reserved (treated as none). Current configuration only, first appearance of each SubChId kept; an entry that would cross the end
 * of its FIG is not read. FIG 0/14 never restarts the parser and leaves the other lists alone. */
typedef struct
{
  int32_t sub_ch_id, scheme;
} dabstar_fec_scheme;
int  dabstar_fib_parser_fec_schemes(const dabstar_fib_parser * p, dabstar_fec_scheme * out, int cap);

/* Cyclic-prefix correlation of DabProcessor::_process_ofdm_symbols_1_to_L (main/dab_processor.cpp:317-333): samples = n frames x
 * 75 x 2552 complex floats (data symbols 1..75 of a frame with their prefixes); out = n x (re, im) of
 * sum_sym sum_{i < 504} x[i + 2048] conj(x[i]); its argument, limited to +-20 degrees, is the fine AFC step (:236-251,366). */
int dabstar_cp_correlate(dabstar_ctx * ctx, const float * samples, int n, float * out_re_im, int mem);

/* The decoder's own frame FFT (sample conversion, cyclic-prefix removal, integer-Hz oscillator, 2048-point transform and
 * frequency de-interleaving in one kernel), exposed for tests. samples: n_recs recordings laid end to end in one buffer of
 * DABSTAR_FMT_* `fmt` (u8 / i16 I,Q pairs or complex floats), recording r holding rec_samples[r] samples; samples outside a
 * recording count as zero. frames: host array of n_frames descriptors; frame f writes rows 0..n_syms (and the null row 76
 * when n_syms is 75) of X slot xslot. X: n_xslots x 77 x 1536 complex floats in the demapper's pair layout (re 2p, re 2p+1,
 * im 2p, im 2p+1), filled with 0xFF bytes before the launch, so rows the kernel does not write keep that pattern.
 * max_ctas_per_sm: resident CTAs per SM of the launch (0: the launcher's choice). null_fft (may be NULL): n_frames x 2048
 * complex floats, the natural-order FFT of each frame's null symbol as the TII detector receives it.
 * Oscillator (sample_reader.cpp:276-281): sample i (0-based) of a symbol read from phase ph is multiplied by
 * e^{j 2 pi ((ph - f (i + 1)) mod 2048000) / 2048000}. Rejects an out-of-range rec / xslot, n_syms outside 0..75, a frequency
 * of 2 048 000 Hz or more in magnitude, an unknown format or a negative count with DABSTAR_E_INVALID before launching anything. */
typedef struct
{
  int64_t sym0;             /* sample index within the recording of the first useful sample of symbol 0 */
  int64_t eval;             /* sample index at which the oscillator stands at ph_eval with f_sym0 */
  int32_t rec, xslot;       /* recording index, row block of X */
  int32_t f_sym0, ph_eval;  /* integer Hz and phase of symbol 0 */
  int32_t f_data, ph_data;  /* ... before the first sample (cyclic prefix) of symbol 1 */
  int32_t f_null, ph_null;  /* ... before the first sample of the null symbol */
  int32_t n_syms;           /* data symbols present, 0..75 */
  int32_t reserved;
} dabstar_fft_frame;
int dabstar_fft_frames(dabstar_ctx * ctx, const void * samples, int fmt, const int64_t * rec_samples, int n_recs,
                       const dabstar_fft_frame * frames, int n_frames, int n_xslots, int max_ctas_per_sm, float * X,
                       float * null_fft, int mem);

/* ------------------------------------------------------------------------------------------------ whole path */
typedef struct
{
  int32_t input_format;    /* DABSTAR_FMT_* (raw_reader.cpp:66-70, xml_reader.cpp:254-372) */
  int32_t soft_bit_type;   /* ESoftBitType: 0 SOFTDEC1 (default), 1 SOFTDEC2, 2 SOFTDEC3 */
  float   sync_threshold;  /* 3.0 (dabradio.cpp:92) */
  int32_t strongest_peak;  /* PhaseReference::set_sync_on_strongest_peak */
  int32_t scan_mode;       /* DabProcessor::set_scan_mode: FIC only */
  int32_t keep_soft_bits;  /* keep 75x3072 int16 per frame for dabstar_decoder_soft_bits */
  int32_t max_window;      /* frames speculated per recording per round (0 = default 256) */
  int32_t upload_chunk_frames; /* host input is uploaded in chunks of this many frames per recording, overlapped with the decode (0 = auto) */
} dabstar_decoder_cfg;

typedef struct
{
  int64_t sym0_pos;        /* stream index of the first useful sample of symbol 0 */
  int32_t start_index;     /* PRS correlation peak */
  float   fbb_sym0, fbb_data, fbb_null, fsync, phase_cp, clock_err;
  int32_t fic_ratio_before, fic_ratio_after;
  uint8_t fic_valid[4];
} dabstar_frame_info;

typedef struct dabstar_decoder dabstar_decoder;

/* One decoder = one DabProcessor per recording (main/dab_processor.h:71), n_recordings of them in lock step. */
int  dabstar_decoder_create(dabstar_ctx * ctx, const dabstar_decoder_cfg * cfg, int n_recordings, dabstar_decoder ** out);
void dabstar_decoder_destroy(dabstar_decoder * dec);
/* DabProcessor::set_audio_channel / MscHandler::set_channel (backend/msc_handler.h:43) */
int  dabstar_decoder_set_subchannels(dabstar_decoder * dec, int recording, const dabstar_subch * sc, int n);
/* DabProcessor::run() over complete recordings. iq[r]: n_samples[r] IQ pairs in cfg.input_format. */
int  dabstar_decoder_run(dabstar_decoder * dec, const void * const * iq, const int64_t * n_samples, int mem);

int     dabstar_decoder_n_frames(const dabstar_decoder * dec, int recording);
int     dabstar_decoder_frame_info(const dabstar_decoder * dec, int recording, dabstar_frame_info * out, int cap);
/* FicDecoder::get_fib_bits per frame: n_frames x 3072 bytes, valid: n_frames x 4 */
int     dabstar_decoder_fib_bits(const dabstar_decoder * dec, int recording, uint8_t * bits, uint8_t * valid);
/* The same FIBs packed 8 bits per byte, first bit most significant: n_frames x 12 x 32 bytes, the reference's FIC dump
 * format (fic_decoder.cpp:291-308). This is how they are read back from the device; dabstar_decoder_fib_bits unpacks. */
int     dabstar_decoder_fib_packed(const dabstar_decoder * dec, int recording, uint8_t * packed);
int     dabstar_decoder_soft_bits(const dabstar_decoder * dec, int recording, int frame, int16_t * out);
int64_t dabstar_decoder_msc_size(const dabstar_decoder * dec, int recording, int sub_ch_id);
/* FrameProcessor::add_to_frame payloads (backend/frame_processor.h:43), concatenated, one bit per byte */
int64_t dabstar_decoder_msc_copy(const dabstar_decoder * dec, int recording, int sub_ch_id, uint8_t * out, int64_t cap);
/* The same payload packed 8 bits per byte, first bit most significant (3 x bit rate bytes per logical frame, as
 * eti_generator.cpp:403-411 packs a sub-channel): how it is read back from the device; dabstar_decoder_msc_copy unpacks.
 * Returns the bytes written (dabstar_decoder_msc_size / 8 in total). */
int64_t dabstar_decoder_msc_packed(const dabstar_decoder * dec, int recording, int sub_ch_id, uint8_t * out, int64_t cap);
/* Self-configuration: the recording's sub-channels and CIF counter are taken from its own FIC (dabstar_fib_parser on the
 * CRC-good FIBs in stream order) instead of dabstar_decoder_set_subchannels. Every sub-channel FIG 0/1 describes gets a
 * Backend from the frame after its first description (in the reference that moment is a GUI action); with ETI enabled the
 * generator frames the sub-channel list and FIG 0/0's CIF counter as it would sample them at symbol 4 of each frame.
 * enable = 2 adds what DabProcessor does with a real FIB decoder behind get_cif_count() (main/dab_processor.cpp:273-285): the
 * null symbol after a frame whose CIF counter has (count & 7) >= 4 is a TII symbol and does not update the null power
 * (OfdmDecoder::store_null_symbol_with_tii). The counter of frame f comes from that frame's own FIC, which the batched path
 * only knows after the window has been demapped, so the run speculates per pass: first with plain null symbols, then again
 * with the flags its own CIF counters give, until the flags used equal the flags produced (normally one extra pass). */
int     dabstar_decoder_set_auto_config(dabstar_decoder * dec, int recording, int enable);
/* sub-channels of the last run (as set, or as discovered); returns the count */
int     dabstar_decoder_subchannels(const dabstar_decoder * dec, int recording, dabstar_subch * out, int cap);
int     dabstar_decoder_ensemble(const dabstar_decoder * dec, int recording, dabstar_ensemble_info * out);
/* FIG 0/2 service components of a self-configured recording as the FIB parser holds them at the end of the run (what tells a
 * DAB+ sub-channel, TMId 0 / ASCTy 63, from an MPEG layer II one); returns the count (E_INVALID: not self-configured) */
int     dabstar_decoder_components(const dabstar_decoder * dec, int recording, dabstar_service_comp * out, int cap);
/* DAB+ outer code inside the run: Mp4Processor::add_to_frame behind BackendDriver (backend_driver.cpp:38-59) for the chosen
 * sub-channels, on the device, on the run's own MSC payload (see dabstar_dabplus_decode). sub_ch_id -1: every sub-channel the
 * recording's own FIG 0/2 lists as DAB+ (TMId 0, ASCTy 63; needs auto-config). An explicit id must name a sub-channel set with
 * dabstar_decoder_set_subchannels whose bit rate is a multiple of 8 in 8..192 (with auto-config it is looked up in the run's
 * own FIC). enable = 0 deselects it. scan_mode decodes no MSC and so no super-frames; streaming is not supported
 * (DABSTAR_E_UNSUPPORTED). */
int     dabstar_decoder_set_dabplus(dabstar_decoder * dec, int recording, int sub_ch_id, int enable);
/* records of the super-frames the processor attempted in the last run, in stream order, exactly as dabstar_dabplus_decode
 * returns them for dabstar_decoder_msc_copy's bits of that sub-channel; returns the count (E_INVALID: not DAB+-decoded) */
int     dabstar_decoder_superframes(const dabstar_decoder * dec, int recording, int sub_ch_id, dabstar_superframe * out, int cap);
/* their decoded super-frames, 110 * (bit_rate / 8) bytes each; returns bytes written (out NULL: the bytes there are) */
int64_t dabstar_decoder_superframe_payload(const dabstar_decoder * dec, int recording, int sub_ch_id, uint8_t * out, int64_t cap);
/* device time of the last run's DAB+ pass; *rounds (may be NULL): its walk / decode rounds */
double  dabstar_decoder_dabplus_ms(const dabstar_decoder * dec, int * rounds);
/* windows (five-frame candidates) of the last run's DAB+ pass: out[0] whose raw header was Fire-code checked, out[1] that went
 * through Reed-Solomon (the processor attempts about one in five of a synchronised stream) */
int     dabstar_decoder_dabplus_windows(const dabstar_decoder * dec, int64_t out[2]);
/* MPEG layer II audio frames inside the run (see dabstar_mp2_frames) for the chosen sub-channels, on the device, on the run's own
 * MSC payload. sub_ch_id -1: every sub-channel the recording's own FIG 0/2 lists as MPEG layer II (TMId 0, ASCTy 0; needs
 * auto-config). An explicit id must name a sub-channel set with dabstar_decoder_set_subchannels whose bit rate is a layer II rate
 * (with auto-config it is looked up in the run's own FIC). enable = 0 deselects it. A sub-channel may be selected for DAB+ as
 * well; both passes read the same payload. scan_mode decodes no MSC and so no frames; streaming is not supported
 * (DABSTAR_E_UNSUPPORTED: a 48 ms frame can straddle two chunks). */
int     dabstar_decoder_set_mp2(dabstar_decoder * dec, int recording, int sub_ch_id, int enable);
/* records of the last run's audio-frame slots, exactly as dabstar_mp2_frames returns them for dabstar_decoder_msc_copy's bits of
 * that sub-channel; returns the count (E_INVALID: not MP2-decoded in the last run) */
int     dabstar_decoder_mp2_frames(const dabstar_decoder * dec, int recording, int sub_ch_id, dabstar_mp2_frame * out, int cap);
/* the OK frames' bytes in record order (a playable MPEG audio elementary stream); returns bytes written (out NULL: the bytes
 * there are). A damaged frame can be read from dabstar_decoder_msc_packed at first_frame * 3 * bit_rate. */
int64_t dabstar_decoder_mp2_payload(const dabstar_decoder * dec, int recording, int sub_ch_id, uint8_t * out, int64_t cap);
/* device time of the last run's MP2 pass */
double  dabstar_decoder_mp2_ms(const dabstar_decoder * dec);
/* Packet-mode data groups inside the run (see dabstar_packet_groups) for the chosen (sub-channel, address) streams, on the device,
 * on the run's own MSC payload; a sub-channel's packets are parsed once however many of its addresses are chosen. sub_ch_id -1:
 * every packet-mode component of the recording's own FIC, that is every FIG 0/2 TMId 3 component whose SCId a FIG 0/3 entry
 * resolves to a sub-channel, with that entry's packet address and DG flag (needs auto-config; `address` is ignored). An explicit
 * id must name a sub-channel set with dabstar_decoder_set_subchannels whose bit rate is a multiple of 8 (with auto-config it is
 * looked up in the run's own FIC), and address must be 1..1023. The DG flag of an explicit selection is the one the run's own
 * FIG 0/3 gives that (sub-channel, address) with auto-config, and 0 (MSC data groups) otherwise. enable = 0 deselects it. scan_mode
 * decodes no MSC and so no groups; streaming is not supported (DABSTAR_E_UNSUPPORTED: a data group can span two chunks). */
int     dabstar_decoder_set_packet(dabstar_decoder * dec, int recording, int sub_ch_id, int address, int enable);
/* records of the last run's data groups of one stream, exactly as dabstar_packet_groups returns them for dabstar_decoder_msc_copy's
 * bits of that sub-channel; returns the count (E_INVALID: the stream was not packet-decoded in the last run) */
int     dabstar_decoder_data_groups(const dabstar_decoder * dec, int recording, int sub_ch_id, int address, dabstar_data_group * out, int cap);
/* their bytes in record order; returns bytes written (out NULL: the bytes there are) */
int64_t dabstar_decoder_data_group_payload(const dabstar_decoder * dec, int recording, int sub_ch_id, int address, uint8_t * out, int64_t cap);
int     dabstar_decoder_packet_stats(const dabstar_decoder * dec, int recording, int sub_ch_id, int address, dabstar_packet_stats * out);
/* device time of the last run's packet pass */
double  dabstar_decoder_packet_ms(const dabstar_decoder * dec);
/* FIG 0/3 packet-mode components of a self-configured recording as the FIB parser holds them at the end of the run; returns the
 * count (E_INVALID: not self-configured) */
int     dabstar_decoder_packet_components(const dabstar_decoder * dec, int recording, dabstar_packet_comp * out, int cap);
/* Packet-mode FEC (see dabstar_packet_fec) in front of the packet pass for a sub-channel, off by default. An explicit sub_ch_id
 * forces it on for that sub-channel (its bit rate must be a multiple of 8; with auto-config it is looked up in the run's own FIC);
 * -1: every sub-channel the recording's own FIG 0/14 gives scheme 1 (needs auto-config). It applies to sub-channels that also have
 * a dabstar_decoder_set_packet stream; their data groups are then those of dabstar_packet_groups_fec. The run's MSC payload
 * (dabstar_decoder_msc_copy / _packed) stays as received. enable = 0 deselects it. scan_mode decodes nothing; streaming is not
 * supported (DABSTAR_E_UNSUPPORTED). */
int     dabstar_decoder_set_packet_fec(dabstar_decoder * dec, int recording, int sub_ch_id, int enable);
/* the FEC frame records of one sub-channel in the last run, exactly as dabstar_packet_fec returns them for dabstar_decoder_msc_copy's
 * bits of that sub-channel; returns the count (E_INVALID: no FEC pass on it in the last run) */
int     dabstar_decoder_fec_frames(const dabstar_decoder * dec, int recording, int sub_ch_id, dabstar_fec_frame * out, int cap);
/* device time of the last run's FEC pass */
double  dabstar_decoder_packet_fec_ms(const dabstar_decoder * dec);
/* FIG 0/14 FEC schemes of a self-configured recording as the FIB parser holds them at the end of the run; returns the count
 * (E_INVALID: not self-configured) */
int     dabstar_decoder_fec_schemes(const dabstar_decoder * dec, int recording, dabstar_fec_scheme * out, int cap);
/* EtiGenerator (eti_handler/eti_generator.h:56-66: start_eti_generator before run / process_block per symbol): every
 * sub-channel set with dabstar_decoder_set_subchannels is decoded for every CIF through the generator's own whole-CIF
 * de-interleaver (first frame with its 17th CIF; its start-up bookkeeping, which loses the 16th CIF, is reproduced) and
 * framed as ETI(NI), 6144 bytes per CIF (eti_generator.cpp:163-199, 207-308). cif_count_hi / cif_count_lo are what
 * IFibDecoder::get_cif_count(hi, lo) returns (FIG 0/0); they are constant over the run here. Independent of scan_mode. */
int     dabstar_decoder_enable_eti(dabstar_decoder * dec, int recording, int enable, int cif_count_hi, int cif_count_lo);
int64_t dabstar_decoder_eti_size(const dabstar_decoder * dec, int recording);
int64_t dabstar_decoder_eti_copy(const dabstar_decoder * dec, int recording, uint8_t * out, int64_t cap);
/* TII (DabProcessor::set_tii_processing / set_tii_threshold / set_tii_collisions / set_tii_sub_id, main/dab_processor.h; the
 * null-symbol handling of dab_processor.cpp:273-300) for a SELF-CONFIGURED recording (dabstar_decoder_set_auto_config): the
 * null symbol after a frame is a TII symbol when the CIF counter taken from the recording's own FIG 0/0 has (count & 7) >= 4;
 * frames_to_count of them (ProcessParams::tiiFramesToCount, 5 in the reference's GUI) are accumulated per search. Settings
 * must be equal for all recordings of a decoder. One event = one process_tii_data call; frame = the frame whose null symbol
 * completed it. dabstar_decoder_tii_results returns the number of identifications of the event (out receives up to cap). */
int     dabstar_decoder_enable_tii(dabstar_decoder * dec, int recording, int enable, int frames_to_count, int threshold_db, int collisions, int sub_id);
int     dabstar_decoder_tii_events(const dabstar_decoder * dec, int recording);
int     dabstar_decoder_tii_results(const dabstar_decoder * dec, int recording, int event, dabstar_tii_result * out, int cap, int32_t * frame);
/* dabstar_ofdm_state_quality for a recording's decoder at the end of the last run (the reference shows these figures
 * every 5 frames; mMeanSigmaSqFreqCorr is replayed from the per-frame cyclic-prefix phases). */
int     dabstar_decoder_quality(const dabstar_decoder * dec, int recording, float out[6]);
/* The same figures for every frame (row D4 over time): with dabstar_decoder_set_frame_quality(dec, 1) before a run (default off;
 * applies to all recordings; the demapper then runs its capture instance and keeps 16 bytes per frame on the device),
 * dabstar_decoder_frame_quality writes up to cap records of 6 floats, in the layout of dabstar_decoder_quality, one per frame
 * dabstar_decoder_frame_info lists, and returns that frame count. Record f is what dabstar_decoder_quality would return had the
 * recording ended after frame f: the OFDM state after the frame's null symbol (which updates the noise power only for a plain,
 * non-TII null symbol). A cut trailing frame is not listed and has no record, but its symbols are demapped, so then the
 * end-of-run figures are not the last record; otherwise they are, bit for bit. Records follow the soft bits: a window replayed
 * after verification keeps those of the pass that committed it, self-configuration level 2 those of the final pass, and a
 * segment's frames carry its warm-started state. With streaming, records cover the frames of the current chunk; fields 0-4
 * continue across chunks through the imported OFDM state, while field 5 (sqrt(mMeanSigmaSqFreqCorr)) is replayed from the
 * cyclic-prefix phases of this run's frames only, as dabstar_decoder_quality does, so it starts again at every chunk.
 * dabstar_decoder_frame_quality returns DABSTAR_E_INVALID when the last run did not capture. */
int     dabstar_decoder_set_frame_quality(dabstar_decoder * dec, int enable);
int     dabstar_decoder_frame_quality(const dabstar_decoder * dec, int recording, float * out /* cap x 6 */, int cap);
/* out[0] good FIBs, [1] time-sync established count, [2] time-sync failures, [3] samples consumed,
 * [4] speculation windows run, [5] windows cut short by verification, [6] frames decoded,
 * [7] frames sent through the FFT/demap/FIC pass (exceeds [6] by replayed and partial frames) */
int     dabstar_decoder_counters(const dabstar_decoder * dec, int recording, int64_t out[8]);
/* Frames demapped a second time as the warm-up of a segment (dabstar_decoder_set_segmentation) in the last run. */
int64_t dabstar_decoder_warmup_frames(const dabstar_decoder * dec, int recording);
/* ---- long recordings (SURVEY.md 8e: "one long stream as frame batches with a warm-up prefix")
 * The reference is a stream receiver: OfdmDecoder's per-carrier IIRs (ofdm/ofdm_decoder.cpp:182-251), DabProcessor's AFC / clock
 * loops (main/dab_processor.cpp:191-265) and Backend's 16-CIF de-interleaver (backend/backend.cpp:129-161) run across all
 * frames. Three controls map that onto batches:
 *
 * dabstar_decoder_set_segmentation: inside a run, a verified window of one recording that holds at least 2 x segment_frames
 *   frames is demapped as floor(n / segment_frames) SEGMENTS in parallel instead of one serial chain. Frame positions, AFC, FFT,
 *   FIC / MSC decoding and the time de-interleaver are not affected (they see the whole window: exact); only OfdmDecoder's
 *   per-carrier state is approximated: a segment other than the first starts from reset() state warmup_frames early and
 *   discards the soft bits of those frames. The IIR constants are 0.005 per symbol (mean power, sigma, std deviation: 1e-3
 *   left after 18 frames) and 0.001 (phase integrator). segment_frames = 0 switches segments off (default).
 *
 * dabstar_decoder_set_streaming + export_state / import_state: the input of a run is a CHUNK of a longer stream. With streaming
 *   enabled a frame (or a time-sync search) the chunk does not hold completely is left for the next chunk instead of being decoded
 *   as far as the samples reach (what the reference does at the end of a file); dabstar_decoder_consumed() is the stream index
 *   of the first sample not consumed. export_state writes everything the next chunk depends on (control loops, oscillator
 *   phase, FIC success counter, OfdmDecoder state, the soft bits of the last 4 frames = 16 CIFs) into a relocatable blob;
 *   import_state on any decoder (another context, GPU or process) makes that recording's next run continue the stream: its
 *   input must begin lead_samples before the consumed position (lead > 0 gives the level estimate of a time re-synchronisation
 *   its history, sample_reader.cpp:236; 2^21 samples make it exact). Decoding a recording in chunks gives bit for bit the
 *   results of one run. dabstar_subch::start_frame counts frames of the stream; frame positions are reported as stream indices.
 *   Not available together with self-configuration, ETI or TII. */
int     dabstar_decoder_set_segmentation(dabstar_decoder * dec, int segment_frames, int warmup_frames);
int     dabstar_decoder_set_streaming(dabstar_decoder * dec, int enable);
int64_t dabstar_decoder_consumed(const dabstar_decoder * dec, int recording);
int64_t dabstar_decoder_state_size(const dabstar_decoder * dec, int recording);
/* returns the bytes written (= dabstar_decoder_state_size) or < 0 */
int64_t dabstar_decoder_export_state(dabstar_decoder * dec, int recording, void * blob, int64_t cap);
int     dabstar_decoder_import_state(dabstar_decoder * dec, int recording, const void * blob, int64_t size, int64_t lead_samples);

/* Device time of the last dabstar_decoder_run in milliseconds (CUDA events on the context's stream). */
double  dabstar_decoder_last_ms(const dabstar_decoder * dec);
/* Device time of the FFT + demap + FIC passes of the last run taken as ONE span per window, from the start of the window's
 * FFT to the end of its last kernel (unlike the per-family times below, it includes the gaps between the launches). */
double  dabstar_decoder_heavy_ms(const dabstar_decoder * dec, int with_fic /* 0: first FFT launch to last demap launch of a window */);
/* Device time and launch count per kernel family of the last run (CUDA events around every launch):
 * [0] time sync [1] PRS correlation [2] CP correlation [3] coarse AFC [4] ingest+FFT [5] demap [6] FIC Viterbi [7] MSC Viterbi */
int     dabstar_decoder_stage_ms(const dabstar_decoder * dec, double ms[8], int64_t launches[8]);
/* The MSC Viterbi time of [7] split into its two kernels: time de-interleave / depuncture gather, and trellis + chain back. */
int     dabstar_decoder_msc_kernel_ms(const dabstar_decoder * dec, double * gather_ms, double * trellis_ms);

#ifdef __cplusplus
}
#endif
#endif
