// kernels.h — host-callable launchers of the sm_100a kernels (one translation unit per kernel family).
#pragma once
#include "common.cuh"
#include "viterbi.cuh"
#include "mp2.cuh"
#include "packet.cuh"
#include "pfec.cuh"

#include <vector>

namespace dab
{
// Device-resident constant tables, built once per context (tables.cu).
struct DeviceTables
{
  float2 * w2048;        // e^{-j 2 pi m / 2048}
  float2 * prs;          // phase reference symbol, fft order
  float2 * ref_arg_conj; // coarse-AFC reference (phasereference.cpp:58-66), filled by init_ref_arg
  int16_t * bin_of_k;    // frequency interleaver: nominal carrier k -> fft index 0..2047
  int16_t * rel_of_k;    // realCarrRelIdx of carrier k (ofdm_decoder.cpp:169-180)
  uint16_t * fft_slot_w; // k_fft_frames epilogue: staging slot of output i of thread tid, [16][128] (tables.cu: host_fft_epilogue_layout)
  uint16_t * fft_slot_r; // ... and of nominal carrier k, [1536]
  uint8_t * prbs;        // energy dispersal sequence, PRBS_LEN bits (one per byte)
};

constexpr int PRBS_LEN = 24 * 1024 + 64; // the longest logical frame make_msc_profile accepts, plus slack for 8-byte loads

// Per-recording OFDM decoder state in HBM (ofdm_decoder.h:89-103), nominal carrier order.
struct OfdmStateDev
{
  float integ[K_CARR], stddev[K_CARR], mean_pow[K_CARR], mean_sigma[K_CARR], null_pow[K_CARR];
  float mean_value;
  float mean_pow_all; // unused on the device (see pow_acc)
  // mMeanPowerOvrAll (ofdm_decoder.cpp:214) is ONE IIR that walks the 1536 carriers of every symbol in turn:
  //   y <- y + b (p_k - y), b = 0.005 / 1536.
  // Over G symbols that is  y = A^G y0 + b sum_k w_k c_k  with A = (1-b)^1536, w_k = (1-b)^(1535-k) and the per-carrier
  // recurrence c_k <- A c_k + p_k, which the demapper keeps in pow_acc (one packed FMA per symbol); pow_carry = A^G y0
  // (y0 = 1 at reset()). The weighted sum is formed on the host when the figure is asked for.
  float pow_carry;
  float pad[1];
  float pow_acc[K_CARR];
};
constexpr double POW_ALL_BETA = 3.255208184782532e-06;   // (float)(0.005f / 1536.0f)
constexpr float POW_ALL_DECAY = 0.9950124713222692f;     // (1 - beta)^1536

// Per-frame signal quality (dabstar_decoder_set_frame_quality). What the capture instance of the demapper keeps of the state
// after a frame's null symbol (one per frame of a window, by descriptor index) ...
struct FrameQualSnap
{
  float stddev[K_CARR], null_pow[K_CARR], pow_acc[K_CARR];
  float pow_carry;  // A^G y0 after the frame
  float mean_value; // mMeanValue: sum |r| of the frame's last symbol / 1536
  float pad[2];
};
// ... and what k_frame_quality reduces it to (one per frame slot); the host forms the dB figures from it (engine.cu)
struct FrameQual
{
  float sum_stddev, sum_null_pow, mean_pow_all, mean_value;
};

// One serial run of the demapper: consecutive frames of one recording (a whole window, or one SEGMENT of it).
// Segments (SURVEY 8e, "frame batches with a warm-up prefix"): the per-carrier IIRs of OfdmDecoder run across all frames
// of a stream, so a segment that does not start where the recording's state was left starts from reset() state `warmup`
// frames early and throws those frames' soft bits away; only the segment that ends the window stores the state.
struct DemapWork
{
  int desc_first;  // first FrameDesc of this run (warm-up frames included)
  int n_frames;    // frames incl. warm-up
  int state_in;    // OfdmStateDev the run starts from (index into the state array)
  int state_out;   // where the state after the last frame is stored, -1: nowhere (in == out is allowed)
  int reset;       // start from OfdmDecoder::reset() state instead of state_in's vectors (after a time-sync loss; warm-started segments)
  int warmup;      // leading frames whose soft bits are not written
};

struct DipWork
{
  int rec;
  long long pos;   // position (in this run's input) where TimeSyncer::read_samples_until_end_of_level_drop starts
  long long abs0;  // stream index of the input's sample 0 (0 unless the run continues a stream): the level IIR's age
};
struct DipResult
{
  long long pos;   // stream position after the call
  int status;      // 0 established, 1 no dip, 2 no end of dip, 3 end of data
  float s_level;
};

// viterbi_kernels.cu
int viterbi_smem_bytes(int max_steps, int warps);
// fic_frames != nullptr: the jobs are the 4 FIC blocks of each of the n_jobs / 4 frame descriptors (jobs is ignored).
// step_tab: device copy of the profiles' step tables (VitProfile::tab_off). ws / ws_bytes: device workspace of the thread-per-code-word path (viterbi_ws_bytes() for one launch; a smaller
// workspace makes the launcher work in chunks, none selects the warp-per-code-word kernel).
size_t viterbi_ws_bytes(int n_jobs, int max_steps);
// hook (optional): called on the launch stream before the gather kernel (0), between gather and trellis kernel (1) and after the
// trellis kernel (2) of every chunk of the thread-per-code-word path, or before (3) and after (2) the warp-per-code-word kernel:
// lets the caller time the kernels separately.
struct VitSpanHook
{
  void (*mark)(void * user, int which, cudaStream_t stream);
  void * user;
};
cudaError_t launch_viterbi(cudaStream_t stream, const VitJob * jobs, const FrameDesc * fic_frames, int n_jobs, const VitProfile * profiles, int max_steps,
                           const int16_t * soft, uint8_t * out_bits, const uint8_t * prbs, uint8_t * crc_ok, int * ber,
                           const unsigned * step_tab, void * ws, size_t ws_bytes, unsigned long long * launch_counter, const VitSpanHook * hook = nullptr);

// bits: one decoded bit per byte (8-byte aligned, n_bytes * 8 of them) -> out: n_bytes bytes, first bit most significant
cudaError_t launch_linear_jobs(cudaStream_t stream, VitJob * jobs, int n, long long src_stride, int n_bits, int profile, unsigned long long * launch_counter);
cudaError_t launch_expand_backend_jobs(cudaStream_t stream, const BackendJobRange * ranges, int n_ranges, VitJob * jobs, unsigned long long * launch_counter);
cudaError_t launch_pack_bits(cudaStream_t stream, const uint8_t * bits, uint8_t * out, long long n_bytes, unsigned long long * launch_counter);

// dabplus_kernels.cu: the DAB+ outer code over a table of streams (one DAB+ sub-channel of one recording each)
struct SuperFrameRec
{
  int first_frame, pre_ok, ok, rs_errors, rs_corrections, fc_corrected;
  int dac_rate, sbr_flag, aac_channel_mode, ps_flag, mpeg_surround;
  int num_aus, au_start[7], au_state[6];
};
constexpr int DABPLUS_MAX_RS_DIMS = 24; // code words per super-frame at 192 kbit/s
struct DabplusStream
{
  const uint8_t * src;     // n_frames logical frames of 3 * bit_rate packed bytes
  int bit_rate, n_frames;
  long long win0;          // first of its n_frames - 4 windows (none below 5 frames) in the pass's per-window arrays
  long long att0;          // first of its n_frames - 4 slots of attempted windows (as win0)
  long long out_rec0;      // first output record (filled once the walk has converged)
  long long out_pay0;      // byte offset of its first output super-frame
};
struct DabplusEntry        // a window listed for decoding
{
  unsigned long long pay_off; // its decoded super-frame: 110 * bit_rate / 8 bytes at this offset
  int stream, window;
};
struct DabplusMeta         // running totals of the listed windows and their super-frame bytes
{
  unsigned long long entries, bytes;
};
void dabplus_host_tables(std::vector<uint8_t> & gf_blob, std::vector<uint16_t> & fc_syn);
// state: one byte per window (dabplus.cuh: SF_*), filled with SF_PRE_OK
cudaError_t launch_dabplus_scan(cudaStream_t s, const DabplusStream * st, int n_streams, long long n_windows, const void * gf_tables, uint8_t * state, unsigned long long * lc);
// att_n[i]: windows stream i attempts, listed at att[att0 ..]; those not decoded yet are appended to list at meta->entries, and
// slot[window] = their list index
cudaError_t launch_dabplus_walk(cudaStream_t s, const DabplusStream * st, int n_streams, const uint8_t * state, int * att, DabplusMeta * meta, int * att_n,
                                DabplusEntry * list, int * slot, unsigned long long * lc);
// the n_list windows at list: rec[i] for list[i], payload at list[i].pay_off, SF_DECODED / SF_OK into state; ler: n_list x 24 bytes
cudaError_t launch_dabplus_decode(cudaStream_t s, const DabplusStream * st, const DabplusEntry * list, int n_list, const void * gf_tables, const uint16_t * fc_syn,
                                  uint8_t * payload, int8_t * ler, SuperFrameRec * rec, uint8_t * state, unsigned long long * lc);
// the attempted windows' records and super-frames, n_out of them, in stream order from out_rec0 / out_pay0
cudaError_t launch_dabplus_compact(cudaStream_t s, const DabplusStream * st, int n_streams, long long n_out, const int * att, const int * slot, const DabplusEntry * list,
                                   const SuperFrameRec * rec, const uint8_t * payload, SuperFrameRec * out_rec, uint8_t * out_pay, unsigned long long * lc);

// mp2_kernels.cu: MPEG layer II audio frames over a table of streams (one MP2 sub-channel of one recording each; mp2.cuh)
struct Mp2Stream
{
  const uint8_t * src;     // n_frames logical frames of 3 * bit_rate packed bytes
  int bit_rate, n_frames;
  long long slot0;         // first of its n_frames entries in the pass's per-slot arrays (classes, CRCs, staged records)
  long long out_rec0;      // first output record (set from the walk's counts)
  long long out_pay0;      // byte offset of its first OK frame in the output payload
};
struct Mp2Count            // per stream, from the walk: records, and bytes of its OK frames
{
  long long recs, bytes;
};
// cls: class byte per slot (mp2.cuh: status | MP2_LSF), crc: (stored, computed) per slot, hdr: the slot's first 32 bits
cudaError_t launch_mp2_scan(cudaStream_t s, const Mp2Stream * st, int n_streams, long long n_slots, uint8_t * cls, int2 * crc, uint32_t * hdr, unsigned long long * lc);
// the walk of every stream (a block each): its records at stage[slot0 ..], the byte offset of each OK one inside the stream's
// payload at stage_off[slot0 ..] (-1 for the others), and its totals in cnt
cudaError_t launch_mp2_walk(cudaStream_t s, const Mp2Stream * st, int n_streams, const uint8_t * cls, const int2 * crc, const uint32_t * hdr, Mp2Rec * stage,
                            long long * stage_off, Mp2Count * cnt, unsigned long long * lc);
cudaError_t launch_mp2_compact(cudaStream_t s, const Mp2Stream * st, int n_streams, long long n_out, const Mp2Rec * stage, const long long * stage_off,
                               Mp2Rec * out_rec, uint8_t * out_pay, unsigned long long * lc);

// packet_kernels.cu: packet-mode data groups over a table of streams (packet.cuh). The packets of a sub-channel (one packet-mode
// sub-channel of one recording) are parsed once; a stream is one address of one such sub-channel.
struct PacketSub
{
  const uint8_t * src;     // n_frames logical frames of 3 * bit_rate packed bytes
  int bit_rate, n_frames;
  long long frame0;        // first of its logical frames in the pass's frame index space
  long long slot0;         // first of its n_frames * bit_rate / 8 packet slots
  const uint8_t * fec = nullptr; // packet-mode FEC: one byte per 24-byte slot, non-zero on FEC packets (src is then the corrected copy)
};
struct PacketStream
{
  int sub, address, dg_flag;
  long long stage0;        // first of its staged groups (room for one per slot of its sub-channel)
  long long out_rec0;      // first output record (set from the walk's counts)
  long long out_pay0;      // byte offset of its first group in the output payload
};
struct PacketCount         // per stream, from the walk
{
  long long groups, bytes; // groups emitted and their useful bytes
  long long packets;       // CRC-good data packets with the stream's address
  long long crc_errors, bad_length, cut; // packets of the sub-channel in those classes
  long long padding, command, other_address, continuity_breaks, abandoned, dropped;
};
struct PacketStage         // a group found by the walk: its first and last packet slot of the sub-channel
{
  int start, end, n_packets, bytes;
  long long off;           // byte offset inside the stream's payload
};
struct DgRec               // layout of dabstar_data_group
{
  int32_t first_frame, last_frame, n_packets, status;
  int32_t extension_flag, crc_flag, segment_flag, user_access_flag;
  int32_t type, continuity, repetition, extension;
  int32_t segment_last, segment_number, transport_id, length_indicator;
  int32_t crc_stored, crc_computed, length, data_start, data_length, reserved;
  int64_t offset;
};
// every frame's packets: slots[sub.slot0 + frame * bit_rate / 8 + k] (packet.cuh: packet_frame)
cudaError_t launch_packet_scan(cudaStream_t s, const PacketSub * sub, int n_subs, long long n_frames, PacketSlot * slots, unsigned long long * lc);
// the walk of every stream (a block each): its groups at stage[stage0 ..] and its counters in cnt
cudaError_t launch_packet_walk(cudaStream_t s, const PacketSub * sub, const PacketStream * st, int n_streams, const PacketSlot * slots, PacketStage * stage,
                               PacketCount * cnt, unsigned long long * lc);
// the groups' records and useful data, n_out of them, in stream order from out_rec0 / out_pay0; the MSC data group headers parsed
cudaError_t launch_packet_compact(cudaStream_t s, const PacketSub * sub, const PacketStream * st, int n_streams, long long n_out, const PacketSlot * slots,
                                  const PacketStage * stage, DgRec * out_rec, uint8_t * out_pay, unsigned long long * lc);

// pfec_kernels.cu: packet-mode FEC over a table of streams (one FEC sub-channel of one recording each; pfec.cuh). A stream's
// slots are its 24-byte slots, n_frames * bit_rate / 8 of them.
struct PfecStream
{
  const uint8_t * src;     // n_frames logical frames of 3 * bit_rate packed bytes, as received
  uint8_t * dst;           // the same bytes, copied before the pass; the corrections go here
  int bit_rate, n_frames;
  long long slot0;         // first of its slots in the pass's per-slot arrays (fit codes, run starts, FEC mask)
  long long stage0;        // first of its located runs (room for one per two slots)
  long long out0;          // first output record (set from the locate counts)
};
struct PfecStage           // a located run: its slot, its score, whether its frame is INCOMPLETE
{
  int run, score, incomplete;
};
struct PfecRec             // layout of dabstar_fec_frame
{
  int32_t first_slot, run_slot, first_frame, last_frame, status;
  int32_t rows_corrected, rows_failed, bytes_corrected, headers_matched, reserved;
};
void pfec_host_tables(std::vector<uint8_t> & blob);
// code[slot] = pfec_slot_code, then start[slot] = pfec_run_start, for every slot of every stream
cudaError_t launch_pfec_locate(cudaStream_t s, const PfecStream * st, int n_streams, long long n_slots, uint8_t * code, uint8_t * start, unsigned long long * lc);
// per stream (a block each): its runs in stream order at stage[stage0 ..], their count in cnt, and mask[slot0 + i] = 1 on the
// slots of its runs (mask zeroed by the caller)
cudaError_t launch_pfec_list(cudaStream_t s, const PfecStream * st, int n_streams, const uint8_t * code, const uint8_t * start, PfecStage * stage, int * cnt,
                             uint8_t * mask, unsigned long long * lc);
// the n_out frames (stream order from out0): rows decoded, corrections into dst, records into rec
cudaError_t launch_pfec_correct(cudaStream_t s, const PfecStream * st, int n_streams, long long n_out, const void * tables, const PfecStage * stage, PfecRec * rec,
                                unsigned long long * lc);

// ofdm_kernels.cu
cudaError_t launch_init_ref_arg(cudaStream_t s, const DeviceTables & t, unsigned long long * lc);
cudaError_t launch_fft_batch(cudaStream_t s, const DeviceTables & t, const float2 * in, float2 * out, int n, int sign, unsigned long long * lc);
// max_ctas_per_sm > 0: size the persistent grid for at most that many resident CTAs per SM (0: as many as fit); lets a caller
// run the kernel at a launch shape other than the decoder's, e.g. one CTA per SM
cudaError_t launch_fft_frames(cudaStream_t s, const DeviceTables & t, const FrameDesc * frames, int n_frames, const RecInput * recs, int fmt,
                              float2 * X, int max_ctas_per_sm, unsigned long long * lc);
cudaError_t launch_reorder_frames(cudaStream_t s, const DeviceTables & t, const float2 * fft_nat, int n_frames, float2 * X, unsigned long long * lc);
// ring: device scratch of demap_ring_bytes(n_work) bytes (exchange of the per-symbol sums between the CTAs of a recording).
// The frames of one DemapWork must occupy consecutive row blocks (xslot) of X.
// qsnap: nullptr runs the plain demapper; else the capture instance, which writes a FrameQualSnap per complete frame it writes
// soft bits for, at qsnap[descriptor index].
size_t demap_ring_bytes(int n_work);
cudaError_t launch_demap(cudaStream_t s, const DeviceTables & t, const DemapWork * work, int n_work, const FrameDesc * frames,
                         const uint8_t * null_is_tii, const float2 * X, OfdmStateDev * states, int soft_bit_type, int16_t * soft,
                         unsigned long long * ring, FrameQualSnap * qsnap, unsigned long long * lc);
// out[frames[i].slot] = the sums of qsnap[i], for every complete frame i < n_frames
cudaError_t launch_frame_quality(cudaStream_t s, const FrameDesc * frames, int n_frames, const FrameQualSnap * qsnap, FrameQual * out, unsigned long long * lc);
cudaError_t launch_cp_corr(cudaStream_t s, const FrameDesc * frames, int n_frames, const RecInput * recs, int fmt, float2 * cp, unsigned long long * lc);
cudaError_t launch_prs_corr(cudaStream_t s, const DeviceTables & t, const FrameDesc * frames, int n_frames, const RecInput * recs, int fmt,
                            float threshold_first, float threshold_rest, const uint8_t * first_flags, int strongest, int * start_index, unsigned long long * lc);
cudaError_t launch_coarse_afc(cudaStream_t s, const DeviceTables & t, const FrameDesc * frames, int n_frames, const RecInput * recs, int fmt,
                              int * offset_hz, unsigned long long * lc);
cudaError_t launch_coarse_afc_raw(cudaStream_t s, const DeviceTables & t, const float2 * fft_nat, int n, int * offset_hz, unsigned long long * lc);
// src: packed file samples (see dabstar_sample_format in the C header); lut: 256 floats for the 8-bit containers (device), else nullptr
// FFT (fft order) of the null symbol of each listed frame: out = n_frames x 2048
cudaError_t launch_fft_null(cudaStream_t s, const DeviceTables & t, const FrameDesc * frames, int n_frames, const RecInput * recs, int fmt, float2 * out,
                            unsigned long long * lc);
// tii_kernels.cu: TiiDetector (ofdm/tii_detector.cpp) for a batch of detectors
struct TiiResultDev
{
  int main_id, sub_id;
  float strength, phase_deg;
  int non_etsi;
};
cudaError_t launch_tii_add(cudaStream_t s, const float2 * fft, int n_detectors, int n_symbols, float2 * null_sum, unsigned long long * lc);
cudaError_t launch_tii_process(cudaStream_t s, int n_detectors, float2 * null_sum, float2 * decoded, const uint8_t * pattern, const uint8_t * phase_corr,
                               float threshold_factor, int collisions, int sub_id_coll, TiiResultDev * out, int cap, int * counts, unsigned long long * lc);
// dciq_kernels.cu: SampleReader's DC / IQ-imbalance correction over a whole recording (sample_reader.cpp:216-243).
// state: { meanI, meanQ, meanII, meanIQ, meanQQ }, in and out; workspace: dciq_workspace_bytes(n) device bytes.
size_t dciq_workspace_bytes(long long n);
cudaError_t launch_dc_iq_correct(cudaStream_t s, const float2 * in, long long n, bool do_iq, double alpha, double state[5], void * workspace, float2 * out,
                                 unsigned long long * lc);
// File readers' sample-rate conversion (linear interpolation per 1 ms block); base / frac: 2048-entry device tables.
cudaError_t launch_resample_linear(cudaStream_t s, const float2 * in, long long n_in, int block_in, int shift, const short * base, const float * frac,
                                   long long n_out, float2 * out, unsigned long long * lc);
cudaError_t launch_ingest_convert(cudaStream_t s, const void * src, int container, int msb_first, int iq_order, float inv_scaler, const float * lut,
                                  long long n_samples, float2 * dst, unsigned long long * lc);
cudaError_t launch_dip_search(cudaStream_t s, const DipWork * work, int n, const RecInput * recs, int fmt, DipResult * out, unsigned long long * lc);
} // namespace dab
