// kernels.h — host-callable launchers of the sm_100a kernels (one translation unit per kernel family).
#pragma once
#include "common.cuh"
#include "viterbi.cuh"

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

// dabplus_kernels.cu: one record per five-frame window of a DAB+ sub-channel
struct SuperFrameRec
{
  int first_frame, pre_ok, ok, rs_errors, rs_corrections, fc_corrected;
  int dac_rate, sbr_flag, aac_channel_mode, ps_flag, mpeg_surround;
  int num_aus, au_start[7], au_state[6];
};
void dabplus_host_tables(std::vector<uint8_t> & gf_blob, std::vector<uint16_t> & fc_syn);
// frames: n_frames x 3*bit_rate packed bytes; payload: (n_frames-4) x 110*(bit_rate/8); ler: (n_frames-4) x bit_rate/8; rec: n_frames-4
cudaError_t launch_dabplus(cudaStream_t s, const uint8_t * frames, int bit_rate, int n_frames, const void * gf_tables, const uint16_t * fc_syn,
                           uint8_t * payload, int8_t * ler, SuperFrameRec * rec, unsigned long long * lc);

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
