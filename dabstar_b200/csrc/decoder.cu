// decoder.cu — the whole-path decoder behind include/dabstar_b200.h.
//
// The decoder restates DabProcessor's control flow (main/dab_processor.cpp:110-442) as a host-side state machine
// per recording that drives BATCHED kernels: all recordings advance in lock step, and inside a recording the
// frame-to-frame dependencies (frame position from the PRS peak, AFC from the cyclic-prefix phase, coarse AFC
// gated by the FIC success counter) are handled by speculation: a window of frames is laid out assuming the PRS
// peak stays at T_g and the FIC keeps decoding, every kernel runs over the whole window, and the per-frame PRS
// peaks / FIB CRCs are verified afterwards. A window that fails verification is replayed from a state snapshot
// with the length that verified. Acquisition (first frames, or after a sync loss) runs with windows of one frame.
#include "context.h"

#include <atomic>
#include <chrono>

using namespace dab;

namespace
{
enum class RecState { WAIT_SYNC, EVAL, DONE };

struct MscOut
{
  dabstar_subch sc;
  int profile = -1;
  int first_seen = 0;   // frame whose FIC first described the sub-channel (self-configuration; 0 when set by the caller)
  long long out_off = 0, out_len = 0; // this sub-channel's decoded bits of the last run: bit range in the packed read-back buffer
};

inline int mod_fs_host(long long x)
{
  long long r = x % FS;
  return (int)(r < 0 ? r + FS : r);
}

struct Recording
{
  // TII (dab_processor.cpp:273-300): needs auto_cfg, because which null symbols carry TII follows from the CIF counter
  struct TiiCfg { bool on = false; int frames_to_count = 5, threshold_db = 8, collisions = 0, sub_id = 0; };
  // what the caller set (dabstar_decoder_set_subchannels, _set_auto_config, _enable_eti, _enable_tii) and what one pass over the
  // recording hands the next: kept by restart(), everything else belongs to one run
  struct Cfg
  {
    std::vector<MscOut> msc;   // sub-channels to decode (with auto_cfg: found in the run's FIC) and where the run put their bits
    bool auto_cfg = false;     // sub-channels and CIF counter from the recording's own FIG 0/0 and 0/1
    bool tii_nulls = false;    // auto_cfg level 2: null symbols whose CIF counter has (count & 7) >= 4 do not update the null power
    TiiCfg tii;
    std::vector<uint8_t> tii_flags; // ... per frame, as known from the previous pass over this recording (see dabstar_decoder_run)
    bool eti_on = false;       // EtiGenerator running from the first frame of the run (DabProcessor::start_eti_generator)
    int eti_cif_hi = 0, eti_cif_lo = 0; // IFibDecoder::get_cif_count(hi, lo) as the generator samples it at symbol 4
    std::vector<int> dabplus_ids; // sub-channels whose logical frames go through the DAB+ outer code (dabstar_decoder_set_dabplus)
    bool dabplus_all = false;     // ... and every sub-channel the recording's own FIG 0/2 lists as DAB+
    bool dabplus() const { return dabplus_all || !dabplus_ids.empty(); }
    std::vector<int> mp2_ids; // sub-channels whose logical frames go through the MPEG layer II frame check (dabstar_decoder_set_mp2)
    bool mp2_all = false;     // ... and every sub-channel the recording's own FIG 0/2 lists as MPEG layer II
    bool mp2() const { return mp2_all || !mp2_ids.empty(); }
    struct PacketSel { int sub_ch_id, address; };
    std::vector<PacketSel> packet_sel; // (sub-channel, address) streams whose data groups are assembled (dabstar_decoder_set_packet)
    bool packet_all = false;           // ... and every packet-mode component the recording's own FIG 0/2 and 0/3 describe
    bool packet() const { return packet_all || !packet_sel.empty(); }
    std::vector<int> fec_ids; // sub-channels whose packets go through packet-mode FEC first (dabstar_decoder_set_packet_fec)
    bool fec_all = false;     // ... and every sub-channel the recording's own FIG 0/14 gives scheme 1
  } cfg;
  // input
  const void * d_iq = nullptr;
  long long n = 0;
  // DabProcessor / SampleReader state
  RecState state = RecState::DONE;
  long long pos = 0;       // samples consumed
  int osc_phase = 0;       // SampleReader::currentPhase
  float f_sync = 0, f_bb = 0, clock_err = 0, phase_cp = 0;
  bool first_after_sync = true; // syncThreshold = mcThreshold until a frame has been processed (dab_processor.cpp:154,178)
  int fic_ratio = 0;       // 0..10
  int known_start = -2;    // PRS peak already measured for the next frame (-2 = not measured)
  bool spec_ok = false;    // the previous frame's peak was T_g: speculate the next ones
  int force_window = 0;    // replay length after a failed verification
  bool careful_spec = true;// a window that starts with a coarse-AFC frame may speculate that its FIC decodes (reset when that failed)
  int last_start = -1;     // PRS peak index of the last verified frame (-1: none since the time sync)
  bool ofdm_reset = true;  // OfdmDecoder::reset() pending
  int state_cur = 0;       // which of the recording's two OfdmStateDev buffers holds its state (a window writes the other one
                           // and the buffers swap when it is committed: a window that fails verification needs no restore)
  // stream continuation (dabstar_decoder_import_state): the next run continues a stream instead of starting one
  long long abs_pos0 = 0;  // stream index of sample 0 of this run's input
  long long abs_frames = 0;// frames of the stream decoded before this run
  int hist = 0;            // frame slots of soft-bit history in front of slot_base (the 16-CIF time de-interleaver reaches 4 frames back)
  int held_state = 0;      // ... 0: in front of a frame (EVAL), 1: in front of a time-sync search, 2: before the stream's first sample
  bool held = false;       // streaming: the run stopped in front of a frame (or a time-sync search) the chunk does not hold completely
  // bookkeeping
  long long slot_base = 0; // first frame slot of this recording in the soft-bit / FIB buffers
  int slot_cap = 0;
  int n_slots = 0;         // accepted frames (complete ones)
  int partial_syms = 0;    // data symbols of a trailing cut frame (occupies slot n_slots)
  std::vector<dabstar_frame_info> frames;
  std::vector<uint8_t> crc_ok; // 12 per frame
  std::vector<uint8_t> eti;  // ETI-NI frames of the last run, 6144 bytes each
  struct TiiEvent { int frame; std::vector<dabstar_tii_result> res; int total; };
  std::vector<TiiEvent> tii_events;  // one per process_tii_data call of the last run
  std::vector<FrameDesc> descs;      // descriptors of the accepted frames (the TII pass transforms their null symbols again)
  std::vector<int> sync_frames;      // n_slots at every successful time sync (mTiiDetector.reset(), dab_processor.cpp:150-152)
  std::vector<int> cif_hi_f, cif_lo_f; // auto_cfg: CIF counter as the FIB decoder holds it after each frame's FIC (-1: none yet)
  dabstar_ensemble_info ens{};
  std::vector<dabstar_service_comp> comps; // auto_cfg: FIG 0/2 service components as the FIB parser holds them after the run
  // an audio-decoded sub-channel: its n records from rec0 and pay_bytes bytes from pay0 in the pass's result (dec->dabplus / dec->mp2)
  struct AudioOut { int sub_ch_id, bit_rate, n; long long rec0, pay0, pay_bytes; };
  std::vector<AudioOut> dabplus_out, mp2_out;
  std::vector<dabstar_packet_comp> pcomps; // auto_cfg: FIG 0/3 packet-mode components as the FIB parser holds them after the run
  // a packet-decoded stream: its n records from rec0 and pay_bytes bytes from pay0 in dec->packet's result, and its counters
  struct PacketOut { int sub_ch_id, address, dg_flag, n; long long rec0, pay0, pay_bytes; dabstar_packet_stats stats; };
  std::vector<PacketOut> packet_out;
  std::vector<dabstar_fec_scheme> fschemes; // auto_cfg: FIG 0/14 FEC schemes as the FIB parser holds them after the run
  // a sub-channel through packet-mode FEC: its n frame records from rec0 in dec->pfec's result
  struct FecOut { int sub_ch_id, n; long long rec0; };
  std::vector<FecOut> fec_out;
  long long cnt_good_fibs = 0, cnt_sync_ok = 0, cnt_sync_fail = 0, cnt_windows = 0, cnt_cut = 0, cnt_heavy = 0, cnt_warmup = 0;
  // window scratch
  int w_first_desc = 0;
  bool w_careful = false;

  // DabProcessor::run prologue (dab_processor.cpp:110-142): a run starts from the caller's settings alone; self-configured
  // sub-channels are found again in the run's own FIC
  void restart()
  {
    Cfg keep = std::move(cfg);
    *this = Recording();
    cfg = std::move(keep);
    if (cfg.auto_cfg) cfg.msc.clear();
    for (auto & m : cfg.msc) { m.out_off = 0; m.out_len = 0; }
  }
  // CIFs of the run: four per accepted frame, and those a cut last frame holds completely
  int n_cifs() const { return 4 * n_slots + std::max(0, (partial_syms - 3) / 18); }
  // the null symbol after frame f carries TII: the CIF counter the FIB decoder holds after that frame's FIC has (count & 7) >= 4
  // (none while get_cif_count() is still 0)
  bool tii_null(int f) const { return f < (int)cif_hi_f.size() && cif_hi_f[f] >= 0 && ((cif_hi_f[f] * 250 + cif_lo_f[f]) & 7) >= 4; }
  // no PRS peak: the 2048 samples are consumed and the time sync starts over (dab_processor.cpp:397-401)
  void lose_sync() { osc_phase = mod_fs_host((long long)osc_phase - (long long)roundf(f_bb) * T_U); pos += T_U; state = RecState::WAIT_SYNC; }
  // nothing left to read: a stream holds in front of the frame the next chunk completes
  void end_input(bool streaming) { state = RecState::DONE; held = streaming; held_state = 0; }
};

// What a DabProcessor, its OfdmDecoder and its Backends' de-interleavers carry from one frame to the next
// (dab_processor.cpp:110-265, ofdm_decoder.h:89-103, backend.cpp:129-161), as one relocatable block of bytes.
struct StateBlobHdr
{
  uint32_t magic, version;
  int64_t bytes;
  int64_t stream_pos;   // stream index of the first sample the decoder has not consumed
  int64_t abs_frames;   // frames of the stream decoded so far
  int32_t rec_state;    // 0: in front of a frame, 1: in front of a time-sync search, 2: nothing decoded yet (start of a stream)
  int32_t osc_phase, fic_ratio, first_after_sync, known_start, spec_ok, careful_spec, last_start, ofdm_reset;
  float f_sync, f_bb, clock_err, phase_cp;
  int32_t hist;         // frames of soft bits that follow the OFDM state (0..4)
  int32_t reserved[7];
};
constexpr uint32_t STATE_MAGIC = 0x31534244u; // "DBS1"
int hist_frames_after(const Recording & R) { return (int)std::min<long long>(4, (long long)R.hist + R.n_slots); }

// The two directions between a recording's control state and a state blob: the blob after the run (export) ...
StateBlobHdr blob_header(const Recording & R)
{
  StateBlobHdr h;
  memset(&h, 0, sizeof(h));
  h.stream_pos = R.abs_pos0 + R.pos;
  h.abs_frames = R.abs_frames + R.n_slots;
  h.rec_state = R.held_state;
  h.osc_phase = R.osc_phase; h.fic_ratio = R.fic_ratio; h.first_after_sync = R.first_after_sync ? 1 : 0; h.known_start = R.known_start;
  h.spec_ok = R.spec_ok ? 1 : 0; h.careful_spec = R.careful_spec ? 1 : 0; h.last_start = R.last_start; h.ofdm_reset = R.ofdm_reset ? 1 : 0;
  h.f_sync = R.f_sync; h.f_bb = R.f_bb; h.clock_err = R.clock_err; h.phase_cp = R.phase_cp;
  h.hist = hist_frames_after(R);
  return h;
}
// ... and the run that continues the stream, whose input starts `lead` samples before the stream position
void resume_from(Recording & R, const StateBlobHdr & h, long long lead)
{
  R.hist = h.hist;
  R.abs_frames = h.abs_frames;
  R.abs_pos0 = h.stream_pos - lead;
  R.pos = lead;
  R.osc_phase = h.osc_phase; R.f_sync = h.f_sync; R.f_bb = h.f_bb; R.clock_err = h.clock_err; R.phase_cp = h.phase_cp; R.fic_ratio = h.fic_ratio;
  R.first_after_sync = h.first_after_sync != 0; R.known_start = h.known_start; R.spec_ok = h.spec_ok != 0; R.careful_spec = h.careful_spec != 0;
  R.last_start = h.last_start; R.ofdm_reset = h.ofdm_reset != 0;
  R.state = h.rec_state == 1 ? RecState::WAIT_SYNC : RecState::EVAL;
}

// mMeanSigmaSqFreqCorr (ofdm_decoder.cpp:296-300): at symbol 1 of every frame, from the cyclic-prefix phase the previous frame
// left behind (dab_processor.cpp:236-240,342); not touched by OfdmDecoder::reset(). Replayed over a run's frames in order.
struct SigmaReplay
{
  float sigma = 0.0f, phase = 0.0f;
  float step(const dabstar_frame_info & fi)
  {
    const float fc = phase / TWO_PI_F * 1000.0f;
    sigma += 0.2f * (fc * fc - sigma);
    phase = fi.phase_cp;
    return sigma;
  }
};

} // namespace

struct dabstar_decoder
{
  dabstar_ctx * ctx = nullptr;
  dabstar_decoder_cfg cfg{};
  std::vector<Recording> recs;
  DevBuf d_inputs;      // staged host input
  DevBuf d_recs;        // RecInput[]
  DevBuf d_soft;        // [total_slots][75*3072] int16
  DevBuf d_fib;         // [total_slots][3072]
  DevBuf d_crc;         // [total_slots][12]
  DevBuf d_ber;         // [total_slots][8] int
  DevBuf d_X;           // window: [frames][77][1536] float2
  DevBuf d_states;      // OfdmStateDev[2][n_rec]: current / next state of every recording (Recording::state_cur)
  int seg_frames = 0, seg_warmup = 0; // dabstar_decoder_set_segmentation
  bool streaming = false;             // dabstar_decoder_set_streaming
  bool frame_quality = false;         // dabstar_decoder_set_frame_quality
  bool frame_quality_run = false;     // ... as it was for the last run
  DevBuf d_qsnap;       // window: FrameQualSnap per descriptor (frame quality only)
  DevBuf d_fq;          // [total_slots] FrameQual (frame quality only)
  struct Resume                       // dabstar_decoder_import_state: what the next run of a recording starts from
  {
    bool on = false;
    StateBlobHdr hdr{};               // validated header of the imported blob
    long long lead = 0;
    std::vector<unsigned char> ofdm;  // OfdmStateDev
    std::vector<int16_t> soft;        // hist x FRAME_SOFT
  };
  std::vector<Resume> resume;
  DevBuf d_desc, d_work, d_cp, d_start, d_coarse, d_dipw, d_dipr, d_jobs, d_mscbits, d_etibits, d_etipacked;
  DevBuf d_tii_fft;   // null-symbol spectra of one TII event, fft order
  DevBuf d_mscpacked; // MSC payload packed 8 bits per byte for the read-back
  DevBuf d_fibp;      // FIB bits packed 8 per byte for the read-back (384 bytes per frame)
  DevBuf d_tii_flags; // per descriptor: the frame's null symbol is a TII symbol
  HostBuf h_mscp; // MSC payload of the last run, packed 8 bits per byte
  HostBuf h_fib, h_crc, h_fibp; // h_fib: FIB bits of the self-configuration pass (one per byte); h_fibp: all FIBs of the run, packed 8 bits per byte
  long long total_slots = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  double last_ms = 0;
  // host-input pipeline: the recordings are uploaded in time-ordered chunks on a second stream while earlier
  // chunks are being decoded; chunk_ev[c] fires when chunk c of every recording is resident
  cudaStream_t copy_stream = nullptr;
  std::vector<cudaEvent_t> chunk_ev;
  long long chunk_samples = 0;
  int n_chunks = 0, chunks_done = 0, chunks_waited = -1;
  long long cnt_rounds = 0;
  // per-stage device time of the last run: CUDA events around every kernel launch on the context's stream
  struct Span { int stage; cudaEvent_t a, b; };
  std::vector<Span> spans;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  DabplusPass dabplus; // the DAB+ outer code of the last run (Recording::dabplus_out)
  Mp2Pass mp2;         // the MPEG layer II frames of the last run (Recording::mp2_out)
  PacketPass packet;   // the packet-mode data groups of the last run (Recording::packet_out)
  PfecPass pfec;       // the packet-mode FEC frames of the last run (Recording::fec_out)
  double stage_ms[10] = { 0 };   // [8], [9]: the MSC pass split into its gather and trellis kernels (VitSpanHook)
  long long stage_launches[10] = { 0 };
  cudaEvent_t ev_get()
  {
    if (ev_used == ev_pool.size()) { cudaEvent_t e; cudaEventCreate(&e); ev_pool.push_back(e); }
    return ev_pool[ev_used++];
  }
  void span_begin(int stage, cudaStream_t s = nullptr) { Span sp{ stage, ev_get(), ev_get() }; cudaEventRecord(sp.a, s ? s : ctx->stream); spans.push_back(sp); }
  void span_end(cudaStream_t s = nullptr) { cudaEventRecord(spans.back().b, s ? s : ctx->stream); stage_launches[spans.back().stage]++; }
  // per window: FFT + demap + FIC (heavy_spans) and FFT + demap (fft_demap_spans), each as ONE span from the FFT's start to
  // the last kernel's end (dabstar_decoder_heavy_ms)
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> heavy_spans, fft_demap_spans;
  double heavy_ms = 0, fft_demap_ms = 0;
  HostBuf h_dip, h_start, h_cp, h_coarse; // pinned read-back of the control kernels' results (a pageable target makes the copy a blocking, staged one)
};
enum { ST_DIP = 0, ST_PRS = 1, ST_CP = 2, ST_COARSE = 3, ST_FFT = 4, ST_DEMAP = 5, ST_FIC = 6, ST_MSC = 7, ST_MSC_GATHER = 8, ST_MSC_TRELLIS = 9 };

// VitSpanHook of the MSC pass: a span per kernel of every chunk
static void msc_span_mark(void * user, int which, cudaStream_t stream)
{
  dabstar_decoder * dec = static_cast<dabstar_decoder *>(user);
  // 0: gather kernel begins; 1: gather ends, trellis kernel begins; 2: trellis ends; 3: the warp-per-code-word kernel (gather fused) begins
  if (which == 1 || which == 2) dec->span_end(stream);
  if (which != 2) dec->span_begin(which == 0 ? ST_MSC_GATHER : ST_MSC_TRELLIS, stream);
}

extern "C" int dabstar_decoder_create(dabstar_ctx * ctx, const dabstar_decoder_cfg * cfg, int n_recordings, dabstar_decoder ** out)
{
  if (!ctx || !cfg || !out || n_recordings <= 0) return DABSTAR_E_INVALID;
  if (cfg->input_format < 0 || cfg->input_format > 2 || cfg->soft_bit_type < 0 || cfg->soft_bit_type > 2)
    return ctx->fail(DABSTAR_E_INVALID, "bad decoder configuration");
  CK(cudaSetDevice(ctx->device));
  std::unique_ptr<dabstar_decoder> d(new dabstar_decoder);
  d->ctx = ctx;
  d->cfg = *cfg;
  if (d->cfg.max_window <= 0) d->cfg.max_window = 256;
  if (d->cfg.sync_threshold <= 0.0f) d->cfg.sync_threshold = 3.0f;
  d->recs.resize((size_t)n_recordings);
  d->resume.resize((size_t)n_recordings);
  CK(cudaEventCreate(&d->ev0));
  CK(cudaEventCreate(&d->ev1));
  CK(cudaStreamCreateWithFlags(&d->copy_stream, cudaStreamNonBlocking));
  *out = d.release();
  return 0;
}

extern "C" void dabstar_decoder_destroy(dabstar_decoder * dec)
{
  if (!dec) return;
  cudaSetDevice(dec->ctx->device);
  if (dec->ev0) cudaEventDestroy(dec->ev0);
  if (dec->ev1) cudaEventDestroy(dec->ev1);
  for (cudaEvent_t e : dec->ev_pool) cudaEventDestroy(e);
  for (cudaEvent_t e : dec->chunk_ev) cudaEventDestroy(e);
  if (dec->copy_stream) cudaStreamDestroy(dec->copy_stream);
  delete dec;
}

extern "C" int dabstar_decoder_set_subchannels(dabstar_decoder * dec, int recording, const dabstar_subch * sc, int n)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size() || n < 0 || (n > 0 && !sc)) return DABSTAR_E_INVALID;
  dabstar_ctx * ctx = dec->ctx;
  Recording & r = dec->recs[recording];
  // an ETI frame has room for 64 streams (NST is a 7-bit field next to FICF) and the sub-channels of a CIF do not overlap;
  // a list that breaks either rule would also overrun the 6144-byte ETI frame (8 + 4 NST + 4 + 96 + 3 x sum of bit rates + 8)
  if (n > 64) return ctx->fail(DABSTAR_E_INVALID, "%d sub-channels (an ensemble has at most 64)", n);
  for (int i = 0; i < n; i++)
    for (int j = 0; j < i; j++)
    {
      if (sc[i].sub_ch_id == sc[j].sub_ch_id) return ctx->fail(DABSTAR_E_INVALID, "sub-channel %d listed twice", sc[i].sub_ch_id);
      if (sc[i].start_cu < sc[j].start_cu + sc[j].size_cu && sc[j].start_cu < sc[i].start_cu + sc[i].size_cu)
        return ctx->fail(DABSTAR_E_INVALID, "sub-channels %d and %d overlap", sc[j].sub_ch_id, sc[i].sub_ch_id);
    }
  r.cfg.msc.clear();
  for (int i = 0; i < n; i++)
  {
    MscOut m;
    m.sc = sc[i];
    m.profile = get_profile(ctx, sc[i].short_form, sc[i].bit_rate, sc[i].prot_level);
    if (m.profile < 0) return ctx->fail(DABSTAR_E_INVALID, "unknown protection profile %d/%d/%d", sc[i].short_form, sc[i].bit_rate, sc[i].prot_level);
    const VitProfile & p = ctx->profiles[m.profile];
    if (sc[i].start_cu < 0 || sc[i].size_cu <= 0 || sc[i].start_cu + sc[i].size_cu > 864 || p.n_kept > sc[i].size_cu * 64 || sc[i].start_frame < 0)
      return ctx->fail(DABSTAR_E_INVALID, "sub-channel %d geometry does not fit", sc[i].sub_ch_id);
    r.cfg.msc.push_back(m);
  }
  return 0;
}

extern "C" int dabstar_decoder_set_auto_config(dabstar_decoder * dec, int recording, int enable)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  dec->recs[recording].cfg.auto_cfg = enable != 0;
  dec->recs[recording].cfg.tii_nulls = enable == 2;
  return 0;
}
extern "C" int dabstar_decoder_subchannels(const dabstar_decoder * dec, int recording, dabstar_subch * out, int cap)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size() || (!out && cap > 0)) return DABSTAR_E_INVALID;
  const std::vector<MscOut> & m = dec->recs[recording].cfg.msc;
  for (int i = 0; i < (int)m.size() && i < cap; i++) out[i] = m[i].sc;
  return (int)m.size();
}
extern "C" int dabstar_decoder_ensemble(const dabstar_decoder * dec, int recording, dabstar_ensemble_info * out)
{
  if (!dec || !out || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  *out = dec->recs[recording].ens;
  return 0;
}
extern "C" int dabstar_decoder_components(const dabstar_decoder * dec, int recording, dabstar_service_comp * out, int cap)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size() || cap < 0 || (!out && cap > 0)) return DABSTAR_E_INVALID;
  const Recording & R = dec->recs[recording];
  if (!R.cfg.auto_cfg) return dec->ctx->fail(DABSTAR_E_INVALID, "components: recording %d is not self-configured", recording);
  for (int i = 0; i < (int)R.comps.size() && i < cap; i++) out[i] = R.comps[i];
  return (int)R.comps.size();
}
// The two audio passes after the MSC pass: DAB+ super-frames (ASCTy 63) and MPEG layer II frames (ASCTy 0)
enum AudioKind { AUDIO_DABPLUS, AUDIO_MP2 };
static bool dabplus_rate_ok(int bit_rate) { return bit_rate >= 8 && bit_rate <= 192 && bit_rate % 8 == 0; }
static bool audio_rate_ok(AudioKind k, int bit_rate) { return k == AUDIO_MP2 ? mp2_rate_ok(bit_rate) : dabplus_rate_ok(bit_rate); }
static int set_audio(dabstar_decoder * dec, int recording, int sub_ch_id, int enable, AudioKind kind)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  dabstar_ctx * ctx = dec->ctx;
  Recording::Cfg & c = dec->recs[recording].cfg;
  const char * what = kind == AUDIO_MP2 ? "MP2" : "DAB+";
  if (sub_ch_id < -1 || sub_ch_id > 63) return ctx->fail(DABSTAR_E_INVALID, "%s: sub-channel id %d", what, sub_ch_id);
  if (enable && dec->streaming)
    return ctx->fail(DABSTAR_E_UNSUPPORTED, "%s across stream chunks are not supported", kind == AUDIO_MP2 ? "MPEG audio frames" : "DAB+ super-frames");
  std::vector<int> & ids = kind == AUDIO_MP2 ? c.mp2_ids : c.dabplus_ids;
  bool & all = kind == AUDIO_MP2 ? c.mp2_all : c.dabplus_all;
  if (!enable)
  {
    if (sub_ch_id == -1) all = false;
    else ids.erase(std::remove(ids.begin(), ids.end(), sub_ch_id), ids.end());
    return 0;
  }
  if (sub_ch_id == -1)
  {
    if (!c.auto_cfg) return ctx->fail(DABSTAR_E_INVALID, "%s: sub-channel -1 (the recording's own FIG 0/2) needs self-configuration", what);
    all = true;
    return 0;
  }
  if (!c.auto_cfg) // with self-configuration the sub-channel is looked up in the run's FIC
  {
    const MscOut * m = nullptr;
    for (const MscOut & x : c.msc) if (x.sc.sub_ch_id == sub_ch_id) m = &x;
    if (!m) return ctx->fail(DABSTAR_E_INVALID, "%s: recording %d has no sub-channel %d", what, recording, sub_ch_id);
    if (!audio_rate_ok(kind, m->sc.bit_rate)) return ctx->fail(DABSTAR_E_INVALID, "%s: sub-channel %d has %d kbit/s, which %s", what, sub_ch_id, m->sc.bit_rate,
                                                               kind == AUDIO_MP2 ? "no layer II frame has" : "is not a multiple of 8 in 8..192");
  }
  if (std::find(ids.begin(), ids.end(), sub_ch_id) == ids.end()) ids.push_back(sub_ch_id);
  return 0;
}
extern "C" int dabstar_decoder_set_dabplus(dabstar_decoder * dec, int recording, int sub_ch_id, int enable)
{
  return set_audio(dec, recording, sub_ch_id, enable, AUDIO_DABPLUS);
}
extern "C" int dabstar_decoder_set_mp2(dabstar_decoder * dec, int recording, int sub_ch_id, int enable)
{
  return set_audio(dec, recording, sub_ch_id, enable, AUDIO_MP2);
}
extern "C" int dabstar_decoder_set_packet(dabstar_decoder * dec, int recording, int sub_ch_id, int address, int enable)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  dabstar_ctx * ctx = dec->ctx;
  Recording::Cfg & c = dec->recs[recording].cfg;
  if (sub_ch_id < -1 || sub_ch_id > 63) return ctx->fail(DABSTAR_E_INVALID, "packet mode: sub-channel id %d", sub_ch_id);
  if (sub_ch_id >= 0 && (address < 1 || address > 1023)) return ctx->fail(DABSTAR_E_INVALID, "packet mode: address %d is not 1..1023", address);
  if (enable && dec->streaming) return ctx->fail(DABSTAR_E_UNSUPPORTED, "packet-mode data groups across stream chunks are not supported");
  auto same = [&](const Recording::Cfg::PacketSel & x) { return x.sub_ch_id == sub_ch_id && x.address == address; };
  if (!enable)
  {
    if (sub_ch_id == -1) c.packet_all = false;
    else c.packet_sel.erase(std::remove_if(c.packet_sel.begin(), c.packet_sel.end(), same), c.packet_sel.end());
    return 0;
  }
  if (sub_ch_id == -1)
  {
    if (!c.auto_cfg) return ctx->fail(DABSTAR_E_INVALID, "packet mode: sub-channel -1 (the recording's own FIG 0/2 and 0/3) needs self-configuration");
    c.packet_all = true;
    return 0;
  }
  if (!c.auto_cfg) // with self-configuration the sub-channel is looked up in the run's FIC
  {
    const MscOut * m = nullptr;
    for (const MscOut & x : c.msc) if (x.sc.sub_ch_id == sub_ch_id) m = &x;
    if (!m) return ctx->fail(DABSTAR_E_INVALID, "packet mode: recording %d has no sub-channel %d", recording, sub_ch_id);
    if (m->sc.bit_rate < 8 || m->sc.bit_rate % 8) return ctx->fail(DABSTAR_E_INVALID, "packet mode: sub-channel %d has %d kbit/s, not a multiple of 8", sub_ch_id, m->sc.bit_rate);
  }
  if (std::find_if(c.packet_sel.begin(), c.packet_sel.end(), same) == c.packet_sel.end()) c.packet_sel.push_back({ sub_ch_id, address });
  return 0;
}
extern "C" int dabstar_decoder_set_packet_fec(dabstar_decoder * dec, int recording, int sub_ch_id, int enable)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  dabstar_ctx * ctx = dec->ctx;
  Recording::Cfg & c = dec->recs[recording].cfg;
  if (sub_ch_id < -1 || sub_ch_id > 63) return ctx->fail(DABSTAR_E_INVALID, "packet-mode FEC: sub-channel id %d", sub_ch_id);
  if (enable && dec->streaming) return ctx->fail(DABSTAR_E_UNSUPPORTED, "packet-mode FEC across stream chunks is not supported");
  if (!enable)
  {
    if (sub_ch_id == -1) c.fec_all = false;
    else c.fec_ids.erase(std::remove(c.fec_ids.begin(), c.fec_ids.end(), sub_ch_id), c.fec_ids.end());
    return 0;
  }
  if (sub_ch_id == -1)
  {
    if (!c.auto_cfg) return ctx->fail(DABSTAR_E_INVALID, "packet-mode FEC: sub-channel -1 (the recording's own FIG 0/14) needs self-configuration");
    c.fec_all = true;
    return 0;
  }
  if (!c.auto_cfg) // with self-configuration the sub-channel is looked up in the run's FIC
  {
    const MscOut * m = nullptr;
    for (const MscOut & x : c.msc) if (x.sc.sub_ch_id == sub_ch_id) m = &x;
    if (!m) return ctx->fail(DABSTAR_E_INVALID, "packet-mode FEC: recording %d has no sub-channel %d", recording, sub_ch_id);
    if (m->sc.bit_rate < 8 || m->sc.bit_rate % 8) return ctx->fail(DABSTAR_E_INVALID, "packet-mode FEC: sub-channel %d has %d kbit/s, not a multiple of 8", sub_ch_id, m->sc.bit_rate);
  }
  if (std::find(c.fec_ids.begin(), c.fec_ids.end(), sub_ch_id) == c.fec_ids.end()) c.fec_ids.push_back(sub_ch_id);
  return 0;
}
extern "C" int dabstar_decoder_enable_eti(dabstar_decoder * dec, int recording, int enable, int cif_count_hi, int cif_count_lo)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  if (enable && (cif_count_hi < 0 || cif_count_lo < 0)) return dec->ctx->fail(DABSTAR_E_INVALID, "negative CIF count"); // the generator waits for a valid count (eti_generator.cpp:158-162)
  Recording & r = dec->recs[recording];
  r.cfg.eti_on = enable != 0;
  r.cfg.eti_cif_hi = cif_count_hi;
  r.cfg.eti_cif_lo = cif_count_lo;
  return 0;
}
extern "C" int64_t dabstar_decoder_eti_size(const dabstar_decoder * dec, int recording)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  return (int64_t)dec->recs[recording].eti.size();
}
extern "C" int64_t dabstar_decoder_eti_copy(const dabstar_decoder * dec, int recording, uint8_t * out, int64_t cap)
{
  if (!dec || !out || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  const std::vector<uint8_t> & e = dec->recs[recording].eti;
  const int64_t n = std::min<int64_t>(cap, (int64_t)e.size());
  if (n > 0) memcpy(out, e.data(), (size_t)n);
  return n;
}

namespace
{
// ---- ETI-NI framing (eti_handler/eti_generator.cpp:169-199 frame tail, :207-308 _init_eti)
// CRC of ETS 300 799: x^16 + x^12 + x^5 + 1, register preset to all ones, remainder complemented (backend/crc.cpp:75-96)
uint16_t eti_crc(const uint8_t * p, int n)
{
  unsigned reg = 0xffffu;
  for (int i = 0; i < n; i++)
  {
    reg ^= (unsigned)p[i] << 8;
    for (int b = 0; b < 8; b++) reg = (reg & 0x8000u) ? ((reg << 1) ^ 0x1021u) : (reg << 1);
    reg &= 0xffffu;
  }
  return (uint16_t)(~reg & 0xffffu);
}

// Header of one ETI(NI) frame: SYNC, FC, one STC per stream, EOH. Returns the offset of the MST field.
int eti_header(uint8_t * f, int cif_hi, int cif_lo, int minor, const std::vector<MscOut> & streams)
{
  int o = 0;
  cif_lo += minor;
  if (cif_lo >= 250) { cif_lo %= 250; cif_hi++; }
  if (cif_hi >= 20) cif_hi = 20;
  f[o++] = 0xFF;                                                       // ERR
  static const uint8_t fsync[2][3] = { { 0x07, 0x3a, 0xb6 }, { 0xf8, 0xc5, 0x49 } };
  for (int i = 0; i < 3; i++) f[o++] = fsync[cif_lo & 1][i];
  f[o++] = (uint8_t)cif_lo;                                            // FCT
  const int nst = (int)streams.size();
  int fl = nst + 1 + 24;                                               // STC + EOH + FIC in 32-bit words (mode I)
  for (const MscOut & m : streams) fl += (m.sc.bit_rate * 3) / 4;
  f[o++] = (uint8_t)(0x80 | nst);                                      // FICF, NST
  const int fp = (cif_hi * 250 + cif_lo) % 8;
  f[o++] = (uint8_t)((fp << 5) | (0x01 << 3) | ((fl & 0x700) >> 8));   // FP, MID = mode I, FL
  f[o++] = (uint8_t)(fl & 0xff);
  for (const MscOut & m : streams)
  {
    const int tpl = m.sc.short_form ? (0x10 | (m.sc.prot_level - 1)) : (0x20 | m.sc.prot_level);
    const int stl = m.sc.bit_rate * 3 / 8;
    f[o++] = (uint8_t)((m.sc.sub_ch_id << 2) | ((m.sc.start_cu & 0x300) >> 8));
    f[o++] = (uint8_t)(m.sc.start_cu & 0xff);
    f[o++] = (uint8_t)((tpl << 2) | ((stl & 0x300) >> 8));
    f[o++] = (uint8_t)(stl & 0xff);
  }
  f[o++] = 0xFF; f[o++] = 0xFF;                                        // MNSC
  const uint16_t hcrc = eti_crc(f + 4, o - 4);
  f[o++] = (uint8_t)(hcrc >> 8);
  f[o++] = (uint8_t)(hcrc & 0xff);
  return o;
}

// Host restatement of the per-frame control bookkeeping (dab_processor.cpp:191-265, 389-414).
struct FrameCtl
{
  FrameDesc desc;
  dabstar_frame_info info;
};

void ctl_begin_frame(Recording & r, int start_index, int n_syms, FrameCtl & fc)
{
  memset(&fc, 0, sizeof(fc));
  fc.desc.eval = r.pos;
  fc.desc.f_sym0 = (int)roundf(r.f_bb);
  fc.desc.ph_eval = r.osc_phase;
  fc.desc.sym0 = r.pos + start_index;
  fc.desc.n_syms = n_syms;
  fc.info.sym0_pos = r.abs_pos0 + fc.desc.sym0;
  fc.info.start_index = start_index;
  fc.info.fbb_sym0 = r.f_bb;
  fc.info.fic_ratio_before = r.fic_ratio * 10;
  r.osc_phase = mod_fs_host((long long)r.osc_phase - (long long)fc.desc.f_sym0 * (T_U + start_index));
  r.pos += T_U + start_index;
}

// correction: result of the coarse AFC (only when the FIC ratio was below 30 %), or 0 with ran_coarse = false
void ctl_after_coarse(Recording & r, bool ran_coarse, int correction, FrameCtl & fc)
{
  if (ran_coarse)
  {
    if (correction != 100000)
    {
      r.f_sync += (float)correction;
      if (fabsf(r.f_sync) > 35000.0f) r.f_sync = 0.0f;
    }
    if (correction != 0) r.clock_err = 0.0f;
    r.f_bb = r.f_sync;
  }
  fc.desc.f_data = (int)roundf(r.f_bb);
  fc.desc.ph_data = r.osc_phase;
  fc.desc.clock_err = r.clock_err;
  fc.info.fbb_data = r.f_bb;
  fc.info.clock_err = r.clock_err;
}

// Phase of the cyclic-prefix sum after the derotation by the integer frequency f (dab_processor.cpp:326-333; the kernel sums the
// RAW samples, the derotated sum differs by the constant factor e^{-j 2 pi f / 1000}): the one expensive, state-independent part
// of the per-frame recurrence once f is known.
float cp_phase(float2 cp_raw, int f)
{
  // (the integer frequency changes rarely: a small direct-mapped cache of the two trigonometric values, same expressions)
  struct Rot { int f; bool set; double c, s; };
  static thread_local Rot rot_cache[64] = {};
  Rot & rc = rot_cache[(unsigned)f & 63u];
  if (!rc.set || rc.f != f)
  {
    const double ang = -2.0 * M_PI * (double)f / 1000.0;
    rc = Rot{ f, true, cos(ang), sin(ang) };
  }
  const double cr = rc.c, sr = rc.s;
  const float re = (float)((double)cp_raw.x * cr - (double)cp_raw.y * sr), im = (float)((double)cp_raw.x * sr + (double)cp_raw.y * cr);
  return atan2f(im, re);
}

// spec_f / spec_ph: cp_phase(cp_raw, spec_f) computed ahead (by the pool, for the integer frequency the window started with);
// used when the frame's frequency turns out to be that one
void ctl_finish_frame(Recording & r, float2 cp_raw, bool ran_coarse, int correction, FrameCtl & fc, int spec_f = INT32_MIN, float spec_ph = 0.0f)
{
  const int n_syms = fc.desc.n_syms;
  r.osc_phase = mod_fs_host((long long)r.osc_phase - (long long)fc.desc.f_data * ((long long)n_syms * T_S));
  r.pos += (long long)n_syms * T_S;
  if (n_syms < 75) return; // recording ends inside this frame
  float ph = fc.desc.f_data == spec_f ? spec_ph : cp_phase(cp_raw, fc.desc.f_data);
  const float lim = 20.0f * RAD_PER_DEG_F;
  ph = ph > lim ? lim : (ph < -lim ? -lim : ph);
  r.phase_cp = ph;
  r.f_sync += ph / TWO_PI_F * 1000.0f;
  r.f_bb = r.f_sync;
  fc.desc.f_null = (int)roundf(r.f_bb);
  fc.desc.ph_null = r.osc_phase;
  r.osc_phase = mod_fs_host((long long)r.osc_phase - (long long)fc.desc.f_null * T_N);
  r.pos += T_N;
  fc.info.fbb_null = r.f_bb;
  fc.info.fsync = r.f_sync;
  fc.info.phase_cp = ph;
  if (!ran_coarse || correction == 0)
  {
    const int sample_count = fc.info.start_index + T_U + 75 * T_S + T_N;
    float ce = (float)FS * ((float)sample_count / (float)T_F - 1.0f);
    ce = ce > 307.2f ? 307.2f : (ce < -307.2f ? -307.2f : ce);
    r.clock_err += 0.1f * (ce - r.clock_err);
  }
}

struct CtlSnapshot
{
  long long pos; int osc_phase; float f_sync, f_bb, clock_err, phase_cp; int fic_ratio;
};
CtlSnapshot take(const Recording & r) { return { r.pos, r.osc_phase, r.f_sync, r.f_bb, r.clock_err, r.phase_cp, r.fic_ratio }; }
void restore(Recording & r, const CtlSnapshot & s)
{
  r.pos = s.pos; r.osc_phase = s.osc_phase; r.f_sync = s.f_sync; r.f_bb = s.f_bb; r.clock_err = s.clock_err; r.phase_cp = s.phase_cp; r.fic_ratio = s.fic_ratio;
}
} // namespace

namespace
{
// The window of one recording in a round, grown by the layout passes
struct Plan
{
  int rec, want;
  std::vector<FrameCtl> fr; // verified frames of this window
  bool open;
  int next_start;           // measured PRS peak of the frame after fr (-2: not measured)
  int event;                // 1: the frame after the window has no PRS peak (time sync lost)
  int t_first, t_frames;    // this pass: descriptors of the tail being laid out
  int t_last_syms;          // symbols of the last of them (< 75: the recording ends inside it)
};

// (plan, first frame, end frame) pieces of at most 1024 of the frames(plan) frames of every plan: one long recording is a single
// plan, the pool works on pieces
template <typename F> std::vector<std::array<int, 3>> pool_pieces(const std::vector<Plan> & plans, F frames)
{
  std::vector<std::array<int, 3>> pieces;
  for (size_t pi = 0; pi < plans.size(); pi++)
    for (int j0 = 0, n = frames(plans[pi]); j0 < n; j0 += 1024) pieces.push_back({ (int)pi, j0, std::min(n, j0 + 1024) });
  return pieces;
}

// ETI frames of a recording: n_out frames whose streams start at bit_off of the packed ETI payload
struct EtiRef { int rec; long long bit_off; int n_out; };

// One pass of dabstar_decoder_run over all recordings (DESIGN.md §4): rounds of time sync, window layout and the heavy pass until
// every recording is done, then self-configuration, TII, MSC and ETI. Each phase below is one step of that sequence.
struct Run
{
  dabstar_decoder * const dec;
  dabstar_ctx * const ctx;
  const cudaStream_t st;
  const int n_rec, fmt;
  const bool host_in;
  const float thr0;
  const bool trace = getenv("DABSTAR_TRACE") != nullptr; // per-round progress on stderr (debug aid), read once per run
  // X budget: bound the frames of one round so the window spectrum buffer stays below ~12 GB
  const long long x_frame_bytes = (long long)sizeof(float2) * X_ROWS * K_CARR;
  const long long max_round_frames;
  std::chrono::steady_clock::time_point t_run0;
  std::vector<RecInput> rin;
  const RecInput * d_rin = nullptr;
  // the round: control records of the frames being laid out (then of the round's frames, in round order), each recording's
  // control state when its window opened, and the windows
  std::vector<FrameCtl> ctl;
  std::vector<CtlSnapshot> snaps;
  std::vector<int> win_recs;
  std::vector<Plan> plans;
  int n_desc = 0;                                 // frames of the round
  cudaEvent_t wake_ev = nullptr;                  // end of the round's demapper launch
  long long eti_bits = 0;                         // decoded bits of all ETI streams
  // a layout pass: control state after every tail frame, before every plan's tail, and the tail frames that follow a time sync
  std::vector<CtlSnapshot> after, before_tail;
  std::vector<uint8_t> first_flags;

  Run(dabstar_decoder * d, int mem)
    : dec(d), ctx(d->ctx), st(d->ctx->stream), n_rec((int)d->recs.size()), fmt(d->cfg.input_format), host_in(mem == DABSTAR_MEM_HOST),
      thr0(d->cfg.sync_threshold), max_round_frames(std::max<long long>(n_rec, (12LL << 30) / x_frame_bytes)), snaps((size_t)n_rec)
  {
  }
  double elapsed_ms() const { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_run0).count(); }
  void tr(const char * what) const
  {
    if (trace) fprintf(stderr, "[dabstar]   %-28s t=%.3f ms\n", what, elapsed_ms());
  }
  // the decode stream must not read samples at or beyond `upto` before their chunk has landed
  cudaError_t need_upto(long long upto)
  {
    if (!host_in) return cudaSuccess;
    int c = (int)std::min<long long>(dec->n_chunks - 1, std::max<long long>(0, (upto - 1) / dec->chunk_samples));
    if (c <= dec->chunks_waited) return cudaSuccess;
    dec->chunks_waited = c;
    return cudaStreamWaitEvent(st, dec->chunk_ev[c], 0);
  }
  // samples known to be resident (polled, never blocks)
  long long resident_upto()
  {
    if (!host_in) return (long long)1 << 62;
    while (dec->chunks_done < dec->n_chunks && cudaEventQuery(dec->chunk_ev[dec->chunks_done]) == cudaSuccess) dec->chunks_done++;
    (void)cudaGetLastError(); // cudaErrorNotReady from the poll is not an error
    if (dec->chunks_done >= dec->n_chunks) return (long long)1 << 62;
    return (long long)dec->chunks_done * dec->chunk_samples;
  }
  // ---- inputs
  // Host input is uploaded in time-ordered chunks on the copy stream; the decode stream waits for the chunk a kernel
  // reads (need_upto), and windows are sized to what has arrived, so the PCIe transfer overlaps the decode.
  int stage_inputs(const void * const * iq, const int64_t * n_samples)
  {
    dec->spans.clear();
    dec->heavy_spans.clear();
    dec->fft_demap_spans.clear();
    dec->heavy_ms = dec->fft_demap_ms = 0;
    dec->ev_used = 0;
    for (int i = 0; i < 10; i++) { dec->stage_ms[i] = 0; dec->stage_launches[i] = 0; }
    CK(cudaEventRecord(dec->ev0, st));
    ctx->host_pool().prewake(); // the first region of the run is less than a wake-up away
    t_run0 = std::chrono::steady_clock::now();
    const size_t bps = fmt == FMT_U8 ? 2 : (fmt == FMT_I16 ? 4 : 8);
    rin.resize((size_t)n_rec);
    dec->n_chunks = 0;
    dec->chunks_done = 0;
    dec->chunks_waited = -1;
    dec->cnt_rounds = 0;
    if (host_in)
    {
      long long max_n = 0;
      for (int r = 0; r < n_rec; r++) max_n = std::max<long long>(max_n, n_samples[r]);
      const size_t dstride = ((size_t)max_n * bps + 255) & ~(size_t)255; // uniform device stride: a chunk of all recordings is one 2D copy
      CK(dec->d_inputs.reserve(dstride * (size_t)n_rec));
      for (int r = 0; r < n_rec; r++) rin[r] = { dec->d_inputs.as<char>() + dstride * (size_t)r, (long long)n_samples[r] };
      // recordings at a constant host stride (rows of one array) and of equal length go as one cudaMemcpy2DAsync per chunk
      bool uniform = n_rec > 1;
      const ptrdiff_t hstride = n_rec > 1 ? (const char *)iq[1] - (const char *)iq[0] : 0;
      for (int r = 0; r < n_rec && uniform; r++)
        uniform = n_samples[r] == n_samples[0] && (const char *)iq[r] - (const char *)iq[0] == hstride * (ptrdiff_t)r && hstride >= (ptrdiff_t)((size_t)n_samples[0] * bps);
      long long chunk_frames = (long long)((128LL << 20) / ((long long)n_rec * (long long)bps * T_F));
      chunk_frames = std::min<long long>(64, std::max<long long>(4, chunk_frames));
      if (dec->cfg.upload_chunk_frames > 0) chunk_frames = dec->cfg.upload_chunk_frames;
      dec->chunk_samples = chunk_frames * T_F;
      dec->n_chunks = (int)std::max<long long>(1, (max_n + dec->chunk_samples - 1) / dec->chunk_samples);
      while ((int)dec->chunk_ev.size() < dec->n_chunks)
      {
        cudaEvent_t e;
        CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        dec->chunk_ev.push_back(e);
      }
      CK(cudaStreamWaitEvent(dec->copy_stream, dec->ev0, 0)); // earlier work on the decode stream may still read d_inputs
      for (int c = 0; c < dec->n_chunks; c++)
      {
        const long long lo = (long long)c * dec->chunk_samples;
        if (uniform)
        {
          const long long hi = std::min<long long>(n_samples[0], lo + dec->chunk_samples);
          if (lo < hi)
            CK(cudaMemcpy2DAsync((char *)rin[0].iq + (size_t)lo * bps, dstride, (const char *)iq[0] + (size_t)lo * bps, (size_t)hstride, (size_t)(hi - lo) * bps, (size_t)n_rec,
                                 cudaMemcpyHostToDevice, dec->copy_stream));
        }
        else
          for (int r = 0; r < n_rec; r++)
          {
            const long long hi = std::min<long long>(n_samples[r], lo + dec->chunk_samples);
            if (lo < hi)
              CK(cudaMemcpyAsync((char *)rin[r].iq + (size_t)lo * bps, (const char *)iq[r] + (size_t)lo * bps, (size_t)(hi - lo) * bps, cudaMemcpyHostToDevice, dec->copy_stream));
          }
        CK(cudaEventRecord(dec->chunk_ev[c], dec->copy_stream));
      }
    }
    else for (int r = 0; r < n_rec; r++) rin[r] = { iq[r], (long long)n_samples[r] };
    CK(dec->d_recs.reserve(sizeof(RecInput) * (size_t)n_rec));
    UP(dec->d_recs.p, rin.data(), sizeof(RecInput) * (size_t)n_rec);
    d_rin = dec->d_recs.as<RecInput>();
    return 0;
  }
  // ---- per-recording reset (DabProcessor::run prologue, dab_processor.cpp:110-142), or continuation of a stream; slot buffers
  int reset_recordings()
  {
    dec->total_slots = 0;
    for (int r = 0; r < n_rec; r++)
    {
      Recording & R = dec->recs[r];
      R.restart();
      R.d_iq = rin[r].iq;
      R.n = rin[r].n;
      const dabstar_decoder::Resume & rs = dec->resume[r];
      if ((dec->streaming || rs.on) && (R.cfg.dabplus() || R.cfg.mp2()))
        return ctx->fail(DABSTAR_E_UNSUPPORTED, "recording %d: DAB+ super-frames / MPEG audio frames across stream chunks are not supported", r);
      if ((dec->streaming || rs.on) && R.cfg.packet())
        return ctx->fail(DABSTAR_E_UNSUPPORTED, "recording %d: packet-mode data groups across stream chunks are not supported", r);
      if (rs.on)
      {
        if (R.cfg.eti_on || R.cfg.auto_cfg || R.cfg.tii.on) return ctx->fail(DABSTAR_E_UNSUPPORTED, "stream continuation with ETI / self-configuration / TII is not supported");
        if (rs.lead > R.n) return ctx->fail(DABSTAR_E_INVALID, "recording %d: %lld lead samples, %lld samples given", r, rs.lead, R.n);
        resume_from(R, rs.hdr, rs.lead);
      }
      R.slot_base = dec->total_slots + R.hist;
      // a frame consumes T_u + start_index + 75 T_s + T_n samples with start_index >= T_g - 250 (phasereference.cpp:136-139):
      // fewer than T_F when the sample clock runs fast or after a re-sync
      R.slot_cap = (int)(R.n / (T_U + (T_G - 250) + 75LL * T_S + T_N)) + 2;
      dec->total_slots += R.hist + R.slot_cap;
      R.frames.reserve((size_t)R.slot_cap);
      R.descs.reserve((size_t)R.slot_cap);
      R.crc_ok.reserve((size_t)R.slot_cap * 12);
      if (!rs.on)
      {
        R.pos = 20LL * T_U; // 20 reads of T_u samples for the level estimate, no mixing (f = 0)
        R.state = R.pos <= R.n ? RecState::WAIT_SYNC : RecState::DONE;
        if (R.state == RecState::DONE && dec->streaming) { R.pos = 0; R.held = true; R.held_state = 2; } // the chunk is shorter than the level estimate's 20 reads
        R.ofdm_reset = true;
      }
    }
    CK(dec->d_soft.reserve(sizeof(int16_t) * (size_t)dec->total_slots * FRAME_SOFT));
    CK(dec->d_fib.reserve((size_t)dec->total_slots * 3072));
    CK(dec->d_crc.reserve((size_t)dec->total_slots * 12));
    CK(dec->d_ber.reserve(sizeof(int) * (size_t)dec->total_slots * 8));
    dec->frame_quality_run = dec->frame_quality;
    if (dec->frame_quality) CK(dec->d_fq.reserve(sizeof(FrameQual) * (size_t)dec->total_slots));
    CK(dec->d_states.reserve(sizeof(OfdmStateDev) * 2 * (size_t)n_rec));
    if (int e = ofdm_state_init(ctx, dec->d_states.as<OfdmStateDev>(), true, 2 * n_rec)) return e;
    for (int r = 0; r < n_rec; r++)
    {
      dabstar_decoder::Resume & rs = dec->resume[r];
      if (!rs.on) continue;
      // the stream's OFDM decoder state and the soft bits of its last frames (history of the time de-interleaver)
      Recording & R = dec->recs[r];
      CK(cudaMemcpyAsync(dec->d_states.as<OfdmStateDev>() + r, rs.ofdm.data(), sizeof(OfdmStateDev), cudaMemcpyHostToDevice, st));
      if (R.hist > 0)
        CK(cudaMemcpyAsync(dec->d_soft.as<int16_t>() + (size_t)(R.slot_base - R.hist) * FRAME_SOFT, rs.soft.data(), sizeof(int16_t) * (size_t)R.hist * FRAME_SOFT,
                           cudaMemcpyHostToDevice, st));
      SYNC(); // (pageable source)
      rs.on = false; // consumed: a further run without a new import starts a new stream
    }
    CK(cudaMemsetAsync(dec->d_crc.p, 0, (size_t)dec->total_slots * 12, st));
    return 0;
  }
  // ---- time sync for recordings without frame lock
  int time_sync()
  {
    std::vector<DipWork> dw;
    for (int r = 0; r < n_rec; r++)
    {
      Recording & R = dec->recs[r];
      if (R.state != RecState::WAIT_SYNC) continue;
      R.ofdm_reset = true;       // dab_processor.cpp:149
      R.first_after_sync = true; // syncThreshold = mcThreshold
      R.known_start = -2;
      R.spec_ok = false;
      R.last_start = -1;
      dw.push_back({ r, R.pos, R.abs_pos0 });
    }
    if (dw.empty()) return 0;
    CK(dec->d_dipw.reserve(sizeof(DipWork) * dw.size()));
    CK(dec->d_dipr.reserve(sizeof(DipResult) * dw.size()));
    UP(dec->d_dipw.p, dw.data(), sizeof(DipWork) * dw.size());
    {
      long long upto = 0; // the search reads at most T_F + T_N + 70 samples (timesyncer.cpp:66-85) plus one scan block
      for (auto & w : dw) upto = std::max(upto, w.pos + T_F + T_N + 70 + 4096);
      CK(need_upto(upto));
    }
    dec->span_begin(ST_DIP);
    CK(launch_dip_search(st, dec->d_dipw.as<DipWork>(), (int)dw.size(), d_rin, fmt, dec->d_dipr.as<DipResult>(), &ctx->launches));
    dec->span_end();
    CK(dec->h_dip.reserve(sizeof(DipResult) * dw.size()));
    const DipResult * dr = dec->h_dip.as<DipResult>();
    CK(cudaMemcpyAsync(dec->h_dip.p, dec->d_dipr.p, sizeof(DipResult) * dw.size(), cudaMemcpyDeviceToHost, st));
    SYNC();
    tr("time sync done");
    for (size_t i = 0; i < dw.size(); i++)
    {
      Recording & R = dec->recs[dw[i].rec];
      if (dr[i].status == 3 && dec->streaming)
      {
        // the chunk ends inside the search: the next chunk repeats it from where it started
        R.state = RecState::DONE;
        R.held = true;
        R.held_state = 1;
        continue;
      }
      R.pos = dr[i].pos;
      R.clock_err = 0.0f; // dab_processor.cpp:158
      if (dr[i].status == 0) { R.state = RecState::EVAL; R.cnt_sync_ok++; R.sync_frames.push_back(R.n_slots); }
      else if (dr[i].status == 3) R.state = RecState::DONE;
      else R.cnt_sync_fail++;
    }
    return 0;
  }
  // ---- open this round's windows; true when a recording still waits for its time sync
  bool open_windows()
  {
    ctl.clear();
    win_recs.clear();
    bool any_wait = false;
    for (int r = 0; r < n_rec; r++)
    {
      Recording & R = dec->recs[r];
      if (R.state == RecState::WAIT_SYNC) { any_wait = true; continue; }
      if (R.state != RecState::EVAL) continue;
      if (R.pos + T_U > R.n) { R.end_input(dec->streaming); continue; } // the eval read hits the end of the data
      R.w_careful = (R.fic_ratio * 10 < 30) || (R.known_start == -2 && !R.spec_ok);
      R.w_first_desc = (int)ctl.size();
      snaps[r] = take(R);
      win_recs.push_back(r);
    }
    return any_wait;
  }
  // PRS peaks of n frames (descriptors d_fd, first-frame-after-sync flags d_first) into pinned memory; synchronises the stream
  int prs_peaks(const FrameDesc * d_fd, int n, const uint8_t * d_first, const int ** start)
  {
    CK(dec->d_start.reserve(sizeof(int) * (size_t)n));
    dec->span_begin(ST_PRS);
    CK(launch_prs_corr(st, ctx->tab, d_fd, n, d_rin, fmt, thr0, 2.0f * thr0, d_first, dec->cfg.strongest_peak, dec->d_start.as<int>(), &ctx->launches));
    dec->span_end();
    CK(dec->h_start.reserve(sizeof(int) * (size_t)n));
    *start = dec->h_start.as<int>();
    CK(cudaMemcpyAsync(dec->h_start.p, dec->d_start.p, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, st));
    SYNC();
    return 0;
  }
  // ---- step A: measure the PRS peak of the first frame where it is not known and not speculated
  int probe_first_peaks()
  {
    std::vector<FrameDesc> fd;
    std::vector<uint8_t> first;
    for (int r : win_recs)
    {
      Recording & R = dec->recs[r];
      if (!(R.w_careful && R.known_start == -2)) continue;
      FrameDesc d;
      memset(&d, 0, sizeof(d));
      d.rec = r; d.eval = R.pos; d.f_sym0 = (int)roundf(R.f_bb); d.ph_eval = R.osc_phase;
      fd.push_back(d);
      first.push_back(R.first_after_sync ? 1 : 0);
    }
    if (fd.empty()) return 0;
    CK(dec->d_desc.reserve(sizeof(FrameDesc) * fd.size() + fd.size() + 64));
    uint8_t * dfirst = dec->d_desc.as<uint8_t>() + sizeof(FrameDesc) * fd.size();
    UP(dec->d_desc.p, fd.data(), sizeof(FrameDesc) * fd.size());
    UP(dfirst, first.data(), first.size());
    {
      long long upto = 0;
      for (auto & d : fd) upto = std::max(upto, (long long)d.eval + T_U);
      CK(need_upto(upto));
    }
    const int * si = nullptr;
    if (int e = prs_peaks(dec->d_desc.as<FrameDesc>(), (int)fd.size(), dfirst, &si)) return e;
    for (size_t i = 0; i < fd.size(); i++)
    {
      Recording & R = dec->recs[fd[i].rec];
      if (si[i] < 0) R.lose_sync();
      else R.known_start = si[i];
    }
    win_recs.erase(std::remove_if(win_recs.begin(), win_recs.end(), [&](int r) { return dec->recs[r].state != RecState::EVAL; }), win_recs.end());
    return 0;
  }
  // ---- frame layout. A window is grown in passes: lay out the frames that follow the verified ones assuming the PRS
  //      peak stays at T_g, run the cheap kernels on them (CP correlation, PRS correlation; coarse AFC for a careful
  //      frame), resolve the scalar AFC / clock recurrences on the host, and keep the frames up to the first one whose
  //      measured peak differs from the layout. That frame's peak is now known, so the next pass continues from it.
  //      The expensive kernels run once per round, over verified frames only.
  int layout()
  {
    plans.clear();
    for (int r : win_recs)
    {
      Recording & R = dec->recs[r];
      int want = R.force_window > 0 ? R.force_window : ((R.w_careful && !R.careful_spec) ? 1 : dec->cfg.max_window);
      want = (int)std::min<long long>(want, std::max<long long>(1, max_round_frames / std::max<size_t>(1, win_recs.size())));
      want = std::min(want, R.slot_cap - R.n_slots);
      plans.push_back({ r, want, {}, true, R.known_start, 0, 0, 0, 75 });
      plans.back().fr.reserve((size_t)std::max(want, 1));
    }
    const long long resident = resident_upto();
    tr("  plans made");
    for (bool first_pass = true;; first_pass = false)
    {
      long long window_end = 0;
      const int n_tail = lay_out_tail(resident, window_end);
      if (n_tail == 0) break;
      if (trace) fprintf(stderr, "[dabstar]     pass: %d tail frames\n", n_tail);
      tr("  tail laid out");
      CK(need_upto(window_end));
      CK(dec->d_desc.reserve(sizeof(FrameDesc) * (size_t)n_tail + (size_t)n_tail + 64));
      if (int e = upload_descs(n_tail)) return e;
      std::vector<int> coarse((size_t)n_tail, 0);
      if (int e = cp_and_coarse(n_tail, first_pass, coarse)) return e;
      recurrences(n_tail, coarse);
      if (int e = upload_descs(n_tail)) return e;
      tr("  recurrences done");
      bool any_open = false;
      if (int e = verify_peaks(n_tail, any_open)) return e;
      tr("layout pass done");
      if (!any_open) break;
    }
    return 0;
  }
  // Tail layout of the open plans: positions first (a few integer operations per frame), then the descriptors of all plans
  // filled in by the pool. Returns the number of tail frames; window_end: the last sample they reach.
  int lay_out_tail(long long resident, long long & window_end)
  {
    window_end = 0;
    int n_laid = 0;
    for (auto & pl : plans)
    {
      if (!pl.open) continue;
      Recording & R = dec->recs[pl.rec];
      const int s0 = pl.next_start >= 0 ? pl.next_start : T_G;
      long long p = R.pos;
      // host input still in flight: stay within what has arrived, but always reach into the chunk being copied
      const long long lim = host_in ? std::max(resident, (snaps[pl.rec].pos / dec->chunk_samples + 1) * dec->chunk_samples) : ((long long)1 << 62);
      pl.t_first = n_laid;
      pl.t_frames = 0;
      pl.t_last_syms = 75;
      int room = pl.want - (int)pl.fr.size();
      {
        // the peak of the frame after one whose peak was off T_g is not speculated (a detection that was a sample early is
        // followed by one a sample late): probe that frame alone. A MEASURED peak (next_start) is a known start: the frames
        // behind it are laid out at T_g straight away.
        const int prev = pl.fr.empty() ? R.last_start : pl.fr.back().info.start_index;
        if (pl.next_start < 0 && prev != T_G) room = std::min(room, 1);
      }
      for (int j = 0; j < room; j++)
      {
        const int s = j == 0 ? s0 : T_G;
        if (p + T_U + s > R.n) break;                          // eval window + rest of symbol 0 not available
        const long long after_sym0 = p + T_U + s;
        const long long avail = R.n - after_sym0;
        if (!(pl.fr.empty() && j == 0) && std::min<long long>(R.n, after_sym0 + 75LL * T_S + T_N) > lim) break;
        pl.t_frames++;
        if (avail >= 75LL * T_S + T_N) { p = after_sym0 + 75LL * T_S + T_N; continue; }
        if (dec->streaming) { pl.t_frames--; break; } // a chunk of a longer stream: the frame is left for the next chunk
        // the recording ends inside this frame: the reference still decodes the symbols it could read
        pl.t_last_syms = (int)std::min<long long>(75, avail / T_S);
        p = after_sym0 + (long long)pl.t_last_syms * T_S;
        break;
      }
      if (pl.t_frames == 0) { pl.open = false; continue; }
      n_laid += pl.t_frames;
      window_end = std::max(window_end, p);
    }
    ctl.resize((size_t)n_laid);
    tr("  positions walked");
    const auto pieces = pool_pieces(plans, [](const Plan & pl) { return pl.open ? pl.t_frames : 0; });
    ctx->host_pool().parallel_for((int)pieces.size(), [&](int k) {
      Plan & pl = plans[(size_t)pieces[(size_t)k][0]];
      const Recording & R = dec->recs[pl.rec];
      const int s0 = pl.next_start >= 0 ? pl.next_start : T_G;
      for (int j = pieces[(size_t)k][1]; j < pieces[(size_t)k][2]; j++)
      {
        const int s = j == 0 ? s0 : T_G;
        // frame 0 starts at R.pos; frame j > 0 behind frame 0 (peak s0) and j - 1 frames with the peak at T_g
        const long long p = j == 0 ? R.pos : R.pos + (T_U + s0 + 75LL * T_S + T_N) + (long long)(j - 1) * (T_U + T_G + 75LL * T_S + T_N);
        FrameCtl & fc = ctl[(size_t)(pl.t_first + j)];
        memset(&fc.desc, 0, sizeof(fc.desc));
        fc.desc.rec = pl.rec;
        fc.desc.eval = p;
        fc.desc.sym0 = p + s;
        fc.desc.n_syms = j == pl.t_frames - 1 ? pl.t_last_syms : 75;
        fc.desc.slot = (int)(R.slot_base + R.n_slots + (int)pl.fr.size() + j);
        fc.desc.xslot = pl.t_first + j;
      }
    });
    return (int)ctl.size();
  }
  // descriptors go from the control records straight into the pinned staging area, a share per pool thread
  int upload_descs(int n)
  {
    unsigned char * stage = nullptr;
    if (int r_ = upload_begin(ctx, sizeof(FrameDesc) * (size_t)n, &stage)) return r_;
    FrameDesc * o = reinterpret_cast<FrameDesc *>(stage);
    const int parts = std::max(1, std::min(n / 512, 16));
    ctx->host_pool().parallel_for(parts, [&](int k) {
      for (int i = (int)((long long)n * k / parts); i < (int)((long long)n * (k + 1) / parts); i++) o[i] = ctl[(size_t)i].desc;
    });
    return upload_commit(ctx, dec->d_desc.p, stage, sizeof(FrameDesc) * (size_t)n);
  }
  // CP correlation on raw samples (all tail frames, into dec->h_cp) and coarse AFC (first frame of a careful window)
  int cp_and_coarse(int n_tail, bool first_pass, std::vector<int> & coarse)
  {
    CK(dec->d_cp.reserve(sizeof(float2) * (size_t)n_tail));
    dec->span_begin(ST_CP);
    CK(launch_cp_corr(st, dec->d_desc.as<FrameDesc>(), n_tail, d_rin, fmt, dec->d_cp.as<float2>(), &ctx->launches));
    dec->span_end();
    CK(dec->h_cp.reserve(sizeof(float2) * (size_t)n_tail));
    CK(cudaMemcpyAsync(dec->h_cp.p, dec->d_cp.p, sizeof(float2) * (size_t)n_tail, cudaMemcpyDeviceToHost, st));
    if (first_pass)
    {
      // coarse AFC needs symbol 0 derotated with the CURRENT f_bb / phase, which are known for the first frame of a window
      std::vector<FrameDesc> cf;
      std::vector<int> idx;
      for (auto & pl : plans)
      {
        Recording & R = dec->recs[pl.rec];
        if (!pl.open || !(R.fic_ratio * 10 < 30)) continue;
        FrameDesc d = ctl[pl.t_first].desc;
        d.f_sym0 = (int)roundf(R.f_bb);
        d.ph_eval = R.osc_phase;
        cf.push_back(d);
        idx.push_back(pl.t_first);
      }
      if (!cf.empty())
      {
        CK(dec->d_work.reserve(sizeof(FrameDesc) * cf.size()));
        CK(dec->d_coarse.reserve(sizeof(int) * cf.size()));
        UP(dec->d_work.p, cf.data(), sizeof(FrameDesc) * cf.size());
        dec->span_begin(ST_COARSE);
        CK(launch_coarse_afc(st, ctx->tab, dec->d_work.as<FrameDesc>(), (int)cf.size(), d_rin, fmt, dec->d_coarse.as<int>(), &ctx->launches));
        dec->span_end();
        CK(dec->h_coarse.reserve(sizeof(int) * cf.size()));
        const int * res = dec->h_coarse.as<int>();
        CK(cudaMemcpyAsync(dec->h_coarse.p, dec->d_coarse.p, sizeof(int) * cf.size(), cudaMemcpyDeviceToHost, st));
        SYNC();
        for (size_t i = 0; i < idx.size(); i++) coarse[idx[i]] = res[i];
      }
    }
    SYNC();
    tr("  cp synced");
    return 0;
  }
  // scalar recurrences (dab_processor.cpp:205-251), with the control state after every frame
  void recurrences(int n_tail, const std::vector<int> & coarse)
  {
    dab::HostPool & pool = ctx->host_pool();
    const float2 * cp = dec->h_cp.as<float2>();
    after.assign((size_t)n_tail, CtlSnapshot());
    before_tail.assign(plans.size(), CtlSnapshot());
    first_flags.assign((size_t)n_tail, 0);
    // The recurrence of a recording is serial over its frames, but its one expensive step (atan2f of the rotated CP sum) depends
    // on the state only through the INTEGER frequency, which moves rarely: the pool computes the phases of all tail frames for
    // the frequency each plan starts with, the serial pass takes them where the frequency still is that one. (One long
    // recording has a single plan: without this the pass ran 1.0 ms per 9984 frames on one thread.)
    std::vector<float> spec_ph((size_t)n_tail);
    std::vector<int> spec_f(plans.size(), INT32_MIN);
    std::vector<int> plan_of((size_t)n_tail, -1);
    for (size_t pi = 0; pi < plans.size(); pi++)
    {
      if (!plans[pi].open) continue;
      spec_f[pi] = (int)roundf(dec->recs[plans[pi].rec].f_bb);
      for (int j = 0; j < plans[pi].t_frames; j++) plan_of[(size_t)(plans[pi].t_first + j)] = (int)pi;
    }
    {
      const int parts = std::max(1, std::min(n_tail / 256, 4 * (pool.workers() + 1)));
      pool.parallel_for(parts, [&](int k) {
        for (int i = (int)((long long)n_tail * k / parts); i < (int)((long long)n_tail * (k + 1) / parts); i++)
          if (plan_of[(size_t)i] >= 0) spec_ph[(size_t)i] = cp_phase(cp[i], spec_f[(size_t)plan_of[(size_t)i]]);
      });
    }
    pool.parallel_for((int)plans.size(), [&](int pi) {
      Plan & pl = plans[(size_t)pi];
      if (!pl.open) return;
      Recording & R = dec->recs[pl.rec];
      before_tail[(size_t)pi] = take(R);
      const int s0 = pl.next_start >= 0 ? pl.next_start : T_G;
      if (pl.fr.empty() && R.first_after_sync) first_flags[pl.t_first] = 1;
      for (int j = 0; j < pl.t_frames; j++)
      {
        const int i = pl.t_first + j;
        const int slot = ctl[i].desc.slot, n_syms = ctl[i].desc.n_syms;
        FrameCtl fc;
        ctl_begin_frame(R, j == 0 ? s0 : T_G, n_syms, fc);
        const bool ran_coarse = pl.fr.empty() && (j == 0) && (R.fic_ratio * 10 < 30);
        ctl_after_coarse(R, ran_coarse, coarse[i], fc);
        ctl_finish_frame(R, cp[i], ran_coarse, coarse[i], fc, spec_f[(size_t)pi], spec_ph[(size_t)i]);
        fc.desc.rec = pl.rec;
        fc.desc.slot = slot;
        fc.desc.xslot = i;
        ctl[i] = fc;
        after[i] = take(R);
      }
    });
  }
  // PRS peak of every tail frame; a plan keeps its tail up to the first frame whose peak differs from the layout and rewinds
  // its recording's control state to there
  int verify_peaks(int n_tail, bool & any_open)
  {
    uint8_t * d_first = dec->d_desc.as<uint8_t>() + sizeof(FrameDesc) * (size_t)n_tail;
    UP(d_first, first_flags.data(), (size_t)n_tail);
    const int * start = nullptr;
    if (int e = prs_peaks(dec->d_desc.as<FrameDesc>(), n_tail, d_first, &start)) return e;
    tr("  prs synced");
    std::atomic<int> n_open{ 0 };
    ctx->host_pool().parallel_for((int)plans.size(), [&](int pi_) {
      const size_t pi = (size_t)pi_;
      Plan & pl = plans[pi];
      if (!pl.open) return;
      Recording & R = dec->recs[pl.rec];
      int valid = 0;
      for (int j = 0; j < pl.t_frames; j++)
      {
        const int expect = j == 0 ? (pl.next_start >= 0 ? pl.next_start : T_G) : T_G;
        if (!(j == 0 && pl.next_start >= 0) && start[pl.t_first + j] != expect) break;
        valid++;
      }
      for (int j = 0; j < valid; j++) pl.fr.push_back(ctl[pl.t_first + j]);
      if (valid > 0) pl.next_start = -2;
      if (valid == pl.t_frames)
      {
        // everything laid out in this pass verified; the next pass closes the plan when there is no room or no data left
        // (a pass may have been limited to one probe frame)
        if ((int)pl.fr.size() >= pl.want || pl.fr.back().desc.n_syms < 75) pl.open = false;
        else n_open.fetch_add(1, std::memory_order_relaxed);
        return;
      }
      restore(R, valid > 0 ? after[pl.t_first + valid - 1] : before_tail[pi]);
      const int sj = start[pl.t_first + valid];
      if (sj < 0) { pl.event = 1; pl.open = false; }
      else { pl.next_start = sj; n_open.fetch_add(1, std::memory_order_relaxed); R.cnt_cut++; }
    });
    any_open = n_open.load() > 0;
    return 0;
  }
  // ---- this round's verified frames (a recording without any lost its time sync or has nothing left to read); their descriptors
  int collect_frames()
  {
    n_desc = 0;
    std::vector<Plan> kept;
    for (auto & pl : plans)
    {
      Recording & R = dec->recs[pl.rec];
      if (pl.fr.empty())
      {
        if (pl.event == 1) { R.cnt_windows++; R.lose_sync(); }
        else R.end_input(dec->streaming);
        continue;
      }
      R.w_first_desc = n_desc;
      n_desc += (int)pl.fr.size();
      kept.push_back(std::move(pl));
    }
    plans.swap(kept);
    if (plans.empty()) return 0;
    // the round's frames in round order: control records and the device's descriptor list
    dec->cnt_rounds++;
    ctl.resize((size_t)n_desc);
    CK(dec->d_desc.reserve(sizeof(FrameDesc) * (size_t)n_desc + 64));
    unsigned char * desc_stage = nullptr;
    if (int r_ = upload_begin(ctx, sizeof(FrameDesc) * (size_t)n_desc, &desc_stage)) return r_;
    const auto pieces = pool_pieces(plans, [](const Plan & pl) { return (int)pl.fr.size(); });
    ctx->host_pool().parallel_for((int)pieces.size(), [&](int k) {
      Plan & pl = plans[(size_t)pieces[(size_t)k][0]];
      const int base = dec->recs[pl.rec].w_first_desc;
      FrameDesc * o = reinterpret_cast<FrameDesc *>(desc_stage);
      for (int j = pieces[(size_t)k][1]; j < pieces[(size_t)k][2]; j++)
      {
        pl.fr[(size_t)j].desc.xslot = base + j;
        ctl[(size_t)(base + j)] = pl.fr[(size_t)j];
        o[base + j] = pl.fr[(size_t)j].desc;
      }
    });
    if (trace)
      fprintf(stderr, "[dabstar] round %lld t=%.3f ms: %zu recordings, %d frames, chunks resident %d/%d waited %d\n", dec->cnt_rounds,
              elapsed_ms(), plans.size(), n_desc, dec->chunks_done, dec->n_chunks, dec->chunks_waited);
    return upload_commit(ctx, dec->d_desc.p, desc_stage, sizeof(FrameDesc) * (size_t)n_desc);
  }
  // ---- heavy pass: FFT (+ingest, derotation, de-interleave) -> demap -> FIC, one launch of each over the whole round
  int heavy_pass()
  {
    const FrameDesc * d_fd = dec->d_desc.as<FrameDesc>();
    CK(dec->d_X.reserve((size_t)x_frame_bytes * (size_t)n_desc));
    FrameQualSnap * d_qsnap = nullptr;
    if (dec->frame_quality)
    {
      CK(dec->d_qsnap.reserve(sizeof(FrameQualSnap) * (size_t)n_desc));
      d_qsnap = dec->d_qsnap.as<FrameQualSnap>();
    }
    if (int e = sync_profiles(ctx)) return e;
    if (int e = reserve_viterbi_ws(ctx, 4 * n_desc, FIC_OUT + 6)) return e;
    // demapper runs: one per segment of a recording's window. Segment s > 0 starts from reset() state `seg_warmup` frames
    // early (their spectra are in the window's buffer anyway) and discards those frames' soft bits; the segment that ends
    // the window writes the recording's OTHER state buffer, and the buffers swap when the window is committed: a window
    // that fails verification leaves the recording's state untouched.
    std::vector<DemapWork> wk;
    for (auto & pl : plans)
    {
      Recording & R = dec->recs[pl.rec];
      const int n = (int)pl.fr.size();
      const int s_in = pl.rec + R.state_cur * n_rec, s_out = pl.rec + (R.state_cur ^ 1) * n_rec;
      int n_seg = 1;
      if (dec->seg_frames > 0 && n >= 2 * dec->seg_frames) n_seg = n / dec->seg_frames;
      for (int sg = 0; sg < n_seg; sg++)
      {
        const int b = (int)((long long)n * sg / n_seg), e = (int)((long long)n * (sg + 1) / n_seg);
        const int w = sg == 0 ? 0 : std::min(dec->seg_warmup, b);
        const bool from_state = b - w == 0; // reaches back to the window's first frame: continue from the recording's state (exact)
        if (sg > 0) R.cnt_warmup += w;
        wk.push_back({ R.w_first_desc + b - w, e - b + w, s_in, sg == n_seg - 1 ? s_out : -1, from_state ? (R.ofdm_reset ? 1 : 0) : 1, w });
      }
    }
    CK(dec->d_work.reserve(sizeof(DemapWork) * wk.size() + 64));
    DemapWork * d_wk = dec->d_work.as<DemapWork>();
    UP(d_wk, wk.data(), sizeof(DemapWork) * wk.size());
    // TII null symbols (self-configuration level 2): flags per descriptor, from the previous pass's CIF counters
    const uint8_t * d_tii = nullptr;
    {
      std::vector<uint8_t> tii;
      for (auto & pl : plans)
      {
        Recording & R = dec->recs[pl.rec];
        if (R.cfg.tii_flags.empty()) continue;
        if (tii.empty()) tii.assign((size_t)n_desc, 0);
        for (int j = 0; j < (int)pl.fr.size(); j++)
        {
          const size_t f = (size_t)R.n_slots + (size_t)j;
          if (f < R.cfg.tii_flags.size()) tii[(size_t)R.w_first_desc + (size_t)j] = R.cfg.tii_flags[f];
        }
      }
      if (!tii.empty())
      {
        CK(dec->d_tii_flags.reserve(tii.size()));
        UP(dec->d_tii_flags.p, tii.data(), tii.size());
        d_tii = dec->d_tii_flags.as<uint8_t>();
      }
    }
    CK(ctx->demap_ring.reserve(demap_ring_bytes((int)wk.size())));

    cudaEvent_t h0 = dec->ev_get(), h1 = dec->ev_get(), hd = dec->ev_get();
    CK(cudaEventRecord(h0, st));
    dec->span_begin(ST_FFT, st);
    CK(launch_fft_frames(st, ctx->tab, d_fd, n_desc, d_rin, fmt, dec->d_X.as<float2>(), 0, &ctx->launches));
    dec->span_end(st);
    dec->span_begin(ST_DEMAP, st);
    CK(launch_demap(st, ctx->tab, d_wk, (int)wk.size(), d_fd, d_tii, dec->d_X.as<float2>(), dec->d_states.as<OfdmStateDev>(), dec->cfg.soft_bit_type,
                    dec->d_soft.as<int16_t>(), ctx->demap_ring.as<unsigned long long>(), d_qsnap, &ctx->launches));
    dec->span_end(st);
    CK(cudaEventRecord(hd, st));
    // the 4 FIC blocks of every frame of the window, straight from the descriptors (no job list)
    dec->span_begin(ST_FIC, st);
    CK(launch_viterbi(st, nullptr, d_fd, 4 * n_desc, ctx->d_profiles.as<VitProfile>(), FIC_OUT + 6, dec->d_soft.as<int16_t>(), dec->d_fib.as<uint8_t>(),
                      ctx->tab.prbs, dec->d_crc.as<uint8_t>(), dec->d_ber.as<int>(), ctx->d_step_tab.as<unsigned>(), ctx->vit_ws.p, ctx->vit_ws.cap, &ctx->launches));
    dec->span_end(st);
    if (d_qsnap)
    {
      // every frame's snapshot is in: reduce them into the per-slot records (a rolled-back frame's slot is written again
      // by the window that commits it, as its soft bits are)
      dec->span_begin(ST_DEMAP, st);
      CK(launch_frame_quality(st, d_fd, n_desc, d_qsnap, dec->d_fq.as<FrameQual>(), &ctx->launches));
      dec->span_end(st);
    }
    CK(cudaEventRecord(h1, st));
    dec->heavy_spans.push_back({ h0, h1 });
    dec->fft_demap_spans.push_back({ h0, hd });
    wake_ev = hd;
    return 0;
  }
  // ---- read back the FIB CRC flags, 12 per frame in round order
  // (one copy of the slot range this round touched: a copy per recording costs more in launch overhead than the bytes saved)
  int read_crc(std::vector<uint8_t> & crc)
  {
    crc.assign((size_t)n_desc * 12, 0);
    long long s_lo = (long long)1 << 62, s_hi = -1;
    for (auto & pl : plans)
    {
      const long long s0 = ctl[dec->recs[pl.rec].w_first_desc].desc.slot;
      s_lo = std::min(s_lo, s0);
      s_hi = std::max(s_hi, s0 + (long long)pl.fr.size());
    }
    CK(dec->h_crc.reserve((size_t)(s_hi - s_lo) * 12));
    CK(cudaMemcpyAsync(dec->h_crc.p, dec->d_crc.as<uint8_t>() + (size_t)s_lo * 12, (size_t)(s_hi - s_lo) * 12, cudaMemcpyDeviceToHost, st));
    // the pool's workers went to sleep during the FFT and the demapper: have them polling again when the FIC decode ends
    if (wake_ev) { CK(cudaEventSynchronize(wake_ev)); ctx->host_pool().prewake(); }
    SYNC();
    for (auto & pl : plans)
    {
      Recording & R = dec->recs[pl.rec];
      memcpy(crc.data() + (size_t)R.w_first_desc * 12, dec->h_crc.as<uint8_t>() + (size_t)(ctl[R.w_first_desc].desc.slot - s_lo) * 12, pl.fr.size() * 12);
    }
    return 0;
  }
  // ---- accept: the FIC success ratio must not have fallen below 30 % at a frame start (that frame needs the coarse AFC)
  // (the OFDM state of a rolled-back recording is still in its current buffer: nothing to restore on the device)
  void accept(const std::vector<uint8_t> & crc)
  {
    ctx->host_pool().parallel_for((int)plans.size(), [&](int pi) {
      Plan & pl = plans[(size_t)pi];
      Recording & R = dec->recs[pl.rec];
      R.cnt_windows++;
      R.cnt_heavy += (int)pl.fr.size();
      const int base = R.w_first_desc;
      int ratio = snaps[pl.rec].fic_ratio;
      int valid = 0;
      std::vector<int> ratio_after((size_t)(int)pl.fr.size()), ratio_before((size_t)(int)pl.fr.size());
      for (int j = 0; j < (int)pl.fr.size(); j++)
      {
        const int i = base + j;
        if (j > 0 && ratio * 10 < 30) break; // this frame needed the coarse AFC: replay it as the first frame of a careful window
        ratio_before[j] = ratio;
        const int n_fic = std::min(4, ctl[i].desc.n_syms * SYM_BITS / FIC_IN);
        for (int b = 0; b < n_fic; b++)
          for (int q = 0; q < 3; q++)
          {
            if (crc[(size_t)i * 12 + 3 * b + q]) { if (ratio < 10) ratio++; }
            else if (ratio > 0) ratio--;
          }
        ratio_after[j] = ratio;
        valid++;
      }
      if (valid == (int)pl.fr.size())
      {
        // whole window verified: commit
        for (int j = 0; j < (int)pl.fr.size(); j++)
        {
          const int i = base + j;
          const bool complete = ctl[i].desc.n_syms == 75;
          ctl[i].info.fic_ratio_before = ratio_before[j] * 10;
          ctl[i].info.fic_ratio_after = ratio_after[j] * 10;
          const int n_fic = std::min(4, ctl[i].desc.n_syms * SYM_BITS / FIC_IN);
          for (int b = 0; b < 4; b++)
          {
            bool ok = b < n_fic;
            for (int q = 0; q < 3 && ok; q++) ok = crc[(size_t)i * 12 + 3 * b + q] != 0;
            ctl[i].info.fic_valid[b] = ok ? 1 : 0;
            for (int q = 0; q < 3; q++) if (b < n_fic && crc[(size_t)i * 12 + 3 * b + q]) R.cnt_good_fibs++;
          }
          if (complete)
          {
            R.frames.push_back(ctl[i].info);
            R.descs.push_back(ctl[i].desc);
            R.crc_ok.insert(R.crc_ok.end(), crc.begin() + (size_t)i * 12, crc.begin() + (size_t)i * 12 + 12);
            R.n_slots++;
          }
          else { R.partial_syms = ctl[i].desc.n_syms; R.state = RecState::DONE; }
        }
        R.fic_ratio = ratio;
        R.state_cur ^= 1; // the demapper wrote the state after this window into the other buffer
        R.last_start = pl.fr.back().info.start_index;
        if (ratio * 10 >= 30) R.careful_spec = true;
        R.ofdm_reset = false;
        R.force_window = 0;
        R.known_start = -2;
        R.spec_ok = true;
        R.first_after_sync = false;
        if (pl.event == 1 && R.state == RecState::EVAL) R.lose_sync(); // the frame after this window has no PRS peak
        else if (pl.next_start >= 0) { R.known_start = pl.next_start; R.spec_ok = false; } // already measured for the next window
      }
      else
      {
        // the FIC ratio fell below 30 % inside the window: roll back and replay the prefix that needs no coarse AFC
        R.cnt_cut++;
        restore(R, snaps[pl.rec]);
        R.careful_spec = false;
        if (valid > 0) R.force_window = valid;
        else { R.force_window = 0; R.spec_ok = false; } // careful mode follows from the ratio
      }
    });
  }
  // ---- self-configuration: sub-channels and CIF counter from the recording's own FIC (FIG 0/0, 0/1)
  // FibDecoder::process_FIB sees the CRC-good FIBs in stream order; a Backend is taken to exist from the frame after the one
  // whose FIC first described its sub-channel (in the reference that moment is a GUI action), EtiGenerator samples the
  // sub-channel list and the CIF counter at symbol 4 of every frame, i.e. after that frame's own FIC.
  int self_configure()
  {
    bool any = false;
    for (int r = 0; r < n_rec; r++) any = any || (dec->recs[r].cfg.auto_cfg && dec->recs[r].n_slots > 0);
    if (!any) return 0;
    CK(dec->h_fib.reserve((size_t)dec->total_slots * 3072));
    for (int r = 0; r < n_rec; r++)
    {
      Recording & R = dec->recs[r];
      const int fs = std::min(R.slot_cap, R.n_slots + (R.partial_syms > 3 ? 1 : 0));
      if (R.cfg.auto_cfg && fs > 0)
        CK(cudaMemcpyAsync(dec->h_fib.as<uint8_t>() + (size_t)R.slot_base * 3072, dec->d_fib.as<uint8_t>() + (size_t)R.slot_base * 3072, (size_t)fs * 3072, cudaMemcpyDeviceToHost, st));
    }
    SYNC();
    for (int r = 0; r < n_rec; r++)
    {
      Recording & R = dec->recs[r];
      if (!R.cfg.auto_cfg || R.n_slots == 0) continue;
      dabstar_fib_parser * fp = nullptr;
      if (dabstar_fib_parser_create(&fp) != 0) return ctx->fail(DABSTAR_E_NOMEM, "fib parser");
      R.cfg.msc.clear();
      R.cif_hi_f.assign((size_t)R.n_slots + 1, -1);
      R.cif_lo_f.assign((size_t)R.n_slots + 1, -1);
      int known = 0;
      const int n_f = (int)(R.crc_ok.size() / 12);
      for (int f = 0; f < n_f && f <= R.n_slots; f++)
      {
        const uint8_t * fb = dec->h_fib.as<uint8_t>() + ((size_t)R.slot_base + f) * 3072;
        for (int k = 0; k < 12; k++)
          if (R.crc_ok[(size_t)12 * f + k]) dabstar_fib_parser_push(fp, fb + (size_t)(k / 3) * 768 + (size_t)(k % 3) * 256, 1);
        dabstar_ensemble_info e;
        if (dabstar_fib_parser_ensemble(fp, &e) == 1) { R.cif_hi_f[f] = e.cif_count_hi; R.cif_lo_f[f] = e.cif_count_lo; }
        if (e.restarts > 0 && e.n_subch < known) { R.cfg.msc.clear(); known = 0; } // the parser dropped its database
        std::vector<dabstar_subch> all((size_t)std::max(1, e.n_subch));
        dabstar_fib_parser_subchannels(fp, all.data(), (int)all.size());
        for (int i = known; i < e.n_subch; i++)
        {
          MscOut m;
          m.sc = all[i];
          m.sc.start_frame = f + 1;
          m.first_seen = f;
          m.profile = get_profile(ctx, m.sc.short_form, m.sc.bit_rate, m.sc.prot_level);
          if (m.profile < 0 || ctx->profiles[m.profile].n_kept > m.sc.size_cu * 64) continue; // described but not decodable (unknown profile)
          R.cfg.msc.push_back(m);
        }
        known = e.n_subch;
        R.ens = e;
      }
      for (int f = n_f; f <= R.n_slots; f++) { R.cif_hi_f[f] = f > 0 ? R.cif_hi_f[f - 1] : -1; R.cif_lo_f[f] = f > 0 ? R.cif_lo_f[f - 1] : -1; }
      R.comps.resize((size_t)std::max(0, dabstar_fib_parser_components(fp, nullptr, 0)));
      dabstar_fib_parser_components(fp, R.comps.data(), (int)R.comps.size());
      R.pcomps.resize((size_t)std::max(0, dabstar_fib_parser_packet_components(fp, nullptr, 0)));
      dabstar_fib_parser_packet_components(fp, R.pcomps.data(), (int)R.pcomps.size());
      R.fschemes.resize((size_t)std::max(0, dabstar_fib_parser_fec_schemes(fp, nullptr, 0)));
      dabstar_fib_parser_fec_schemes(fp, R.fschemes.data(), (int)R.fschemes.size());
      dabstar_fib_parser_destroy(fp);
    }
    return sync_profiles(ctx);
  }
  // ---- TII (dab_processor.cpp:273-300) for self-configured recordings: the null symbols that carry TII (Recording::tii_null)
  // are transformed again (the demapper's spectrum buffer is per window), accumulated tiiFramesToCount at a time and searched;
  // a time re-synchronisation resets the detector and the counter (dab_processor.cpp:150-152).
  int tii_pass()
  {
    struct Seg { std::vector<int> frames; bool reset_before; };
    std::map<int, std::vector<Seg>> per_rec;
    for (int r = 0; r < n_rec; r++)
    {
      Recording & R = dec->recs[r];
      R.tii_events.clear();
      if (!R.cfg.tii.on || !R.cfg.auto_cfg || R.n_slots == 0) continue;
      const int need = std::max(1, R.cfg.tii.frames_to_count);
      std::vector<int> acc;
      bool reset_pending = false;
      size_t si = 0;
      for (int f = 0; f < R.n_slots; f++)
      {
        while (si < R.sync_frames.size() && R.sync_frames[si] <= f) { acc.clear(); reset_pending = true; si++; }
        if (!R.tii_null(f)) continue;
        acc.push_back(f);
        if ((int)acc.size() >= need) { per_rec[r].push_back({ acc, reset_pending }); acc.clear(); reset_pending = false; }
      }
    }
    if (per_rec.empty()) return 0;
    // recordings with more events first: event e then concerns the first n_e detectors
    std::vector<int> order;
    for (auto & kv : per_rec) order.push_back(kv.first);
    std::sort(order.begin(), order.end(), [&](int a, int b) { return per_rec[a].size() != per_rec[b].size() ? per_rec[a].size() > per_rec[b].size() : a < b; });
    dabstar_tii * det = nullptr;
    if (int e = dabstar_tii_create(ctx, (int)order.size(), &det)) return e;
    std::unique_ptr<dabstar_tii, void (*)(dabstar_tii *)> guard(det, dabstar_tii_destroy);
    const Recording::TiiCfg & tc = dec->recs[order[0]].cfg.tii;
    const int need = std::max(1, tc.frames_to_count), cap = 128;
    for (int r : order)
    {
      const Recording::TiiCfg & t = dec->recs[r].cfg.tii;
      if (std::max(1, t.frames_to_count) != need || t.threshold_db != tc.threshold_db || t.collisions != tc.collisions || t.sub_id != tc.sub_id)
        return ctx->fail(DABSTAR_E_INVALID, "TII settings must be the same for every recording of a decoder");
    }
    dabstar_tii_set_collisions(det, tc.collisions, tc.sub_id);
    std::vector<dabstar_tii_result> res((size_t)order.size() * cap);
    std::vector<int32_t> cnt(order.size());
    for (size_t ev = 0; ev < per_rec[order[0]].size(); ev++)
    {
      int n_act = 0;
      while (n_act < (int)order.size() && per_rec[order[n_act]].size() > ev) n_act++;
      std::vector<FrameDesc> fd;
      for (int a = 0; a < n_act; a++)
      {
        const Seg & sg = per_rec[order[a]][ev];
        if (sg.reset_before)
        {
          CK(cudaMemsetAsync(det->null_sum.as<float2>() + (size_t)a * T_U, 0, sizeof(float2) * T_U, st));
          CK(cudaMemsetAsync(det->decoded.as<float2>() + (size_t)a * 768, 0, sizeof(float2) * 768, st));
        }
        for (int f : sg.frames) fd.push_back(dec->recs[order[a]].descs[f]);
      }
      CK(dec->d_desc.reserve(sizeof(FrameDesc) * fd.size()));
      UP(dec->d_desc.p, fd.data(), sizeof(FrameDesc) * fd.size());
      CK(dec->d_tii_fft.reserve(sizeof(float2) * fd.size() * T_U));
      CK(launch_fft_null(st, ctx->tab, dec->d_desc.as<FrameDesc>(), (int)fd.size(), d_rin, fmt, dec->d_tii_fft.as<float2>(), &ctx->launches));
      const int n_keep = det->n;
      det->n = n_act; // the first n_act detectors take part in this event
      int e = dabstar_tii_add(det, dec->d_tii_fft.as<float>(), need, DABSTAR_MEM_DEVICE);
      if (e == 0) e = dabstar_tii_process(det, tc.threshold_db, res.data(), cap, cnt.data());
      det->n = n_keep;
      if (e) return e;
      for (int a = 0; a < n_act; a++)
      {
        Recording & R = dec->recs[order[a]];
        Recording::TiiEvent te;
        te.frame = per_rec[order[a]][ev].frames.back();
        te.total = cnt[a];
        te.res.assign(res.begin() + (size_t)a * cap, res.begin() + (size_t)a * cap + std::min(cnt[a], cap));
        R.tii_events.push_back(std::move(te));
      }
    }
    return 0;
  }
  // ---- MSC: all logical frames of all sub-channels in one batch per profile size
  // One job per sub-channel and CIF (several hundred thousand for a full ensemble), grouped by code-word length (one launch
  // per length: shared-memory footprint). The host only lists one range per Backend; the jobs are written on the device.
  // The decoded bits are laid out group by group (code-word length), so that a group's payload can be packed and copied
  // to the host while the next group is decoded; nothing on the host waits between the groups.
  int msc_pass()
  {
    struct Group { std::vector<BackendJobRange> ranges; std::vector<MscOut *> outs; int n_jobs = 0; long long bits = 0, bit_base = 0; int job_base = 0; };
    std::map<int, Group> groups;
    for (int r = 0; r < n_rec; r++)
    {
      Recording & R = dec->recs[r];
      const int n_cifs = R.n_cifs();
      for (size_t c = 0; c < R.cfg.msc.size(); c++)
      {
        MscOut & m = R.cfg.msc[c];
        const VitProfile & p = ctx->profiles[m.profile];
        // start_frame counts the frames of the STREAM; CIF indices here are relative to this run's first frame, and a run
        // that continues a stream finds the CIFs of the last R.hist frames in front of its own (negative indices)
        const long long g_abs = 4LL * ((long long)m.sc.start_frame - R.abs_frames);
        const int g_start = (int)std::max<long long>(g_abs, -4LL * R.hist);
        const int g_first = std::max(g_start + 16, 0);
        const int n_out = std::max(0, n_cifs - g_first);
        m.out_off = 0;
        m.out_len = (long long)n_out * p.n_bits;
        if (n_out == 0) continue;
        Group & g = groups[p.n_bits + 6];
        // out / job_first are relative to the group here; the group's bases are added below
        g.ranges.push_back(BackendJobRange{ R.slot_base * FRAME_SOFT, g.bits, m.profile, p.n_bits, g_start, g_first, n_out, m.sc.start_cu * 64, g.n_jobs, 0 });
        g.outs.push_back(&m);
        g.n_jobs += n_out;
        g.bits += (long long)n_out * p.n_bits;
      }
    }
    long long out_total = 0;
    int jobs_total = 0;
    std::vector<BackendJobRange> all_ranges;
    for (auto & kv : groups)
    {
      Group & g = kv.second;
      g.bit_base = out_total;
      g.job_base = jobs_total;
      for (size_t i = 0; i < g.ranges.size(); i++)
      {
        g.ranges[i].out += g.bit_base;
        g.ranges[i].job_first += g.job_base;
        g.outs[i]->out_off = g.ranges[i].out;
      }
      all_ranges.insert(all_ranges.end(), g.ranges.begin(), g.ranges.end());
      out_total += g.bits;
      jobs_total += g.n_jobs;
    }
    tr("msc ranges built");
    if (out_total == 0) return 0;
    CK(dec->d_mscbits.reserve((size_t)out_total));
    CK(dec->d_mscpacked.reserve((size_t)(out_total / 8)));
    CK(dec->h_mscp.reserve((size_t)(out_total / 8)));
    if (int e = sync_profiles(ctx)) return e;
    // every Backend's jobs of every group in one array, written by one launch
    CK(dec->d_jobs.reserve(sizeof(VitJob) * (size_t)jobs_total + sizeof(BackendJobRange) * all_ranges.size() + 256));
    VitJob * d_jobs = dec->d_jobs.as<VitJob>();
    BackendJobRange * d_ranges = reinterpret_cast<BackendJobRange *>(reinterpret_cast<unsigned char *>(d_jobs) + ((sizeof(VitJob) * (size_t)jobs_total + 255) & ~(size_t)255));
    UP(d_ranges, all_ranges.data(), sizeof(BackendJobRange) * all_ranges.size());
    CK(launch_expand_backend_jobs(st, d_ranges, (int)all_ranges.size(), d_jobs, &ctx->launches));
    {
      // one workspace for all groups (they run one after the other on the stream), sized for the largest product
      size_t need_jobs = 0;
      int need_steps = 0;
      for (auto & kv : groups)
        if (viterbi_ws_bytes(kv.second.n_jobs, kv.first) > viterbi_ws_bytes((int)need_jobs, need_steps)) { need_jobs = (size_t)kv.second.n_jobs; need_steps = kv.first; }
      if (int e = reserve_viterbi_ws(ctx, (int)need_jobs, need_steps)) return e;
    }
    // the payload leaves the device packed 8 bits per byte (every logical frame is a whole number of bytes: 24 x bit rate
    // bits), one copy per group into pinned memory on the copy stream; dabstar_decoder_msc_copy unpacks a sub-channel on
    // request. One pageable copy per sub-channel and recording of the bits as bytes cost 220 ms per 10 000 full-ensemble
    // frames, 7 x the kernels.
    // Longest code words first: a group's copy runs under the next group's kernels, only the last group's copy is exposed, and
    // the groups of long code words carry most of the payload (full ensemble: 46 of 141 MB per 9984 frames in the 128 kbit/s group).
    for (auto it = groups.rbegin(); it != groups.rend(); ++it)
    {
      auto & kv = *it;
      Group & g = kv.second;
      {
        const VitSpanHook hook{ msc_span_mark, dec }; // one span per kernel (gather / trellis) instead of one around the launch
        CK(launch_viterbi(st, d_jobs + g.job_base, nullptr, g.n_jobs, ctx->d_profiles.as<VitProfile>(), kv.first, dec->d_soft.as<int16_t>(), dec->d_mscbits.as<uint8_t>(), ctx->tab.prbs,
                          nullptr, nullptr, ctx->d_step_tab.as<unsigned>(), ctx->vit_ws.p, ctx->vit_ws.cap, &ctx->launches, &hook));
      }
      CK(launch_pack_bits(st, dec->d_mscbits.as<uint8_t>() + g.bit_base, dec->d_mscpacked.as<uint8_t>() + g.bit_base / 8, g.bits / 8, &ctx->launches));
      cudaEvent_t ev = dec->ev_get();
      CK(cudaEventRecord(ev, st));
      CK(cudaStreamWaitEvent(dec->copy_stream, ev, 0));
      CK(cudaMemcpyAsync(dec->h_mscp.as<uint8_t>() + g.bit_base / 8, dec->d_mscpacked.as<uint8_t>() + g.bit_base / 8, (size_t)(g.bits / 8), cudaMemcpyDeviceToHost, dec->copy_stream));
    }
    tr("msc enqueued");
    return 0;
  }
  // the run's final synchronisation of `st` covers the payload copies of the MSC pass
  int join_copies()
  {
    cudaEvent_t ev = dec->ev_get();
    CK(cudaEventRecord(ev, dec->copy_stream));
    CK(cudaStreamWaitEvent(st, ev, 0));
    return 0;
  }
  // ---- ETI: every sub-channel of every CIF through EtiGenerator's own de-interleaver (eti_generator.cpp:90-204)
  // The generator's ring holds 16 whole CIFs and, unlike Backend, emits with its 17th CIF but loses the 16th from the
  // history while `Minor` is still -1 (the CIF is stored, index_Out does not advance, the next CIF overwrites it). Seen
  // from ETI frame n (n = 0 is CIF 16 of the run) de-interleaver row m therefore reads entry n - 1 + m of the CIF sequence
  // 0..14, 16, 17, ...; entry -1 (row 0 of frame 0) is the slot about to be overwritten, which still holds CIF 15.
  int eti_jobs(std::vector<EtiRef> & eti_refs)
  {
    std::map<int, std::vector<VitJob>> by_steps;
    long long & bits_total = eti_bits;
    for (int r = 0; r < n_rec; r++)
    {
      Recording & R = dec->recs[r];
      R.eti.clear();
      if (!R.cfg.eti_on || R.cfg.msc.empty()) continue;
      const int n_out = std::max(0, R.n_cifs() - 16);
      if (n_out == 0) continue;
      eti_refs.push_back({ r, bits_total, n_out });
      for (int n = 0; n < n_out; n++)
        for (MscOut & m : R.cfg.msc)
        {
          if (m.first_seen > 4 + (n >> 2)) continue; // not yet in the FIB decoder's list when the generator sampled it
          const VitProfile & p = ctx->profiles[m.profile];
          VitJob j;
          memset(&j, 0, sizeof(j));
          j.src = R.slot_base * FRAME_SOFT;
          j.out = bits_total;
          j.profile = m.profile;
          j.src_mode = VIT_SRC_TIME_DEINTERLEAVE;
          j.flags = VIT_FLAG_PRBS;
          j.cif_first = n - 1;
          j.row_mask = 0xffff;
          j.frag_off = m.sc.start_cu * 64;
          j.skip_plus1 = 15 + 1;
          by_steps[p.n_bits + 6].push_back(j);
          bits_total += p.n_bits;
        }
    }
    if (bits_total == 0) return 0;
    CK(dec->d_etibits.reserve((size_t)bits_total));
    CK(dec->d_etipacked.reserve((size_t)(bits_total / 8)));
    for (auto & kv : by_steps)
    {
      dec->span_begin(ST_MSC);
      if (int e = run_viterbi_jobs(ctx, kv.second, kv.first, dec->d_soft.as<int16_t>(), dec->d_etibits.as<uint8_t>(), nullptr, nullptr, dec->d_jobs)) return e;
      dec->span_end();
      SYNC(); // d_jobs is reused by the next group
    }
    dec->span_begin(ST_MSC);
    CK(launch_pack_bits(st, dec->d_etibits.as<uint8_t>(), dec->d_etipacked.as<uint8_t>(), bits_total / 8, &ctx->launches));
    dec->span_end();
    return 0;
  }
  // ---- the run's read-back (FIB bits of all accepted frames, the ETI payload; its last synchronisation), ETI frames, timings
  // The decoded FIBs leave the device packed 8 bits per byte (32 bytes per FIB, the reference's FIC dump format,
  // fic_decoder.cpp:291-308): 3.8 MB instead of 30.6 MB per 10 000 frames; dabstar_decoder_fib_bits unpacks on request.
  int finish(const std::vector<EtiRef> & eti_refs)
  {
    std::vector<uint8_t> eti_packed;
    if (dec->total_slots > 0)
    {
      const long long n_bytes = (long long)dec->total_slots * 384;
      CK(dec->d_fibp.reserve((size_t)n_bytes));
      CK(dec->h_fibp.reserve((size_t)n_bytes));
      CK(launch_pack_bits(st, dec->d_fib.as<uint8_t>(), dec->d_fibp.as<uint8_t>(), n_bytes, &ctx->launches));
      CK(cudaMemcpyAsync(dec->h_fibp.p, dec->d_fibp.p, (size_t)n_bytes, cudaMemcpyDeviceToHost, st));
    }
    if (!eti_refs.empty())
    {
      eti_packed.resize((size_t)(eti_bits / 8));
      CK(cudaMemcpyAsync(eti_packed.data(), dec->d_etipacked.p, eti_packed.size(), cudaMemcpyDeviceToHost, st));
    }
    CK(cudaEventRecord(dec->ev1, st));
    SYNC();
    if (trace) fprintf(stderr, "[dabstar] run done t=%.3f ms\n", elapsed_ms());
    // ETI(NI) frames: header, FIC of the frame the CIF belongs to, the streams, EOF and TIST, padding (eti_generator.cpp:163-199)
    for (const EtiRef & er : eti_refs)
    {
      Recording & R = dec->recs[er.rec];
      R.eti.assign((size_t)er.n_out * 6144, 0x55);
      const uint8_t * src = eti_packed.data() + er.bit_off / 8;
      for (int n = 0; n < er.n_out; n++)
      {
        uint8_t * f = R.eti.data() + (size_t)n * 6144;
        const int fr = 4 + (n >> 2);
        std::vector<MscOut> streams; // the sub-channel list as sampled at symbol 4 of the CIF's frame
        size_t need = 8 + 4 + 96 + 8;
        for (const MscOut & m : R.cfg.msc) if (m.first_seen <= fr) { streams.push_back(MscOut()); streams.back().sc = m.sc; need += 4 + 3 * (size_t)m.sc.bit_rate; }
        if (streams.size() > 64 || need > 6144) return ctx->fail(DABSTAR_E_INVALID, "ETI frame overflow: %zu streams, %zu bytes", streams.size(), need);
        const bool own = R.cfg.auto_cfg && fr < (int)R.cif_hi_f.size() && R.cif_hi_f[fr] >= 0;
        int o = eti_header(f, own ? R.cif_hi_f[fr] : R.cfg.eti_cif_hi, own ? R.cif_lo_f[fr] : R.cfg.eti_cif_lo, n & 3, streams);
        const int base = o;
        // fibVector: the four FICs of the frame as the FIC decoder left them at symbol 4, whether their CRCs passed or not
        memcpy(f + o, dec->h_fibp.as<uint8_t>() + ((size_t)R.slot_base + 4 + (size_t)(n >> 2)) * 384 + (size_t)(n & 3) * 96, 96);
        o += 96;
        for (const MscOut & m : streams)
        {
          const int nb = 3 * m.sc.bit_rate;
          memcpy(f + o, src, (size_t)nb);
          src += nb;
          o += nb;
        }
        const uint16_t crc = eti_crc(f + base, o - base);
        f[o++] = (uint8_t)(crc >> 8); f[o++] = (uint8_t)(crc & 0xff);
        for (int i = 0; i < 6; i++) f[o++] = 0xFF;                       // RFU, TIST (time stamp not used)
      }
    }
    // device time of the run, of each stage and of the heavy passes
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, dec->ev0, dec->ev1));
    dec->last_ms = ms;
    for (auto & sp : dec->spans) dec->stage_ms[sp.stage] += event_ms(sp.a, sp.b);
    for (auto & hs : dec->heavy_spans) dec->heavy_ms += event_ms(hs.first, hs.second);
    for (auto & hs : dec->fft_demap_spans) dec->fft_demap_ms += event_ms(hs.first, hs.second);
    return 0;
  }
  // time between two recorded events; 0 when there is none
  static float event_ms(cudaEvent_t a, cudaEvent_t b)
  {
    float t = 0;
    return cudaEventElapsedTime(&t, a, b) == cudaSuccess ? t : 0.0f;
  }
};
} // namespace

// ---- packet mode: the data groups of every selected (sub-channel, address) stream on the same packed MSC payload (run_packet).
// Each selected sub-channel's packets are parsed once; first_frame / last_frame count its logical frames as msc_copy lists them.
// Sub-channels with packet-mode FEC go through run_packet_fec first; their packets are then parsed from the corrected copies.
static int packet_phase(dabstar_decoder * dec)
{
  dabstar_ctx * ctx = dec->ctx;
  PacketPass & pp = dec->packet;
  PfecPass & pf = dec->pfec;
  pp.subs.clear();
  pp.streams.clear();
  pf.streams.clear();
  std::vector<std::pair<int, int>> owner; // (recording, sub-channel) of every stream
  std::vector<std::pair<int, int>> fec_owner; // (recording, sub-channel) of every FEC stream
  std::vector<int> fec_sub;                   // ... and its index in pp.subs
  for (int r = 0; r < (int)dec->recs.size(); r++)
  {
    Recording & R = dec->recs[r];
    R.packet_out.clear();
    R.fec_out.clear();
    if (!R.cfg.packet()) continue;
    for (const MscOut & m : R.cfg.msc)
    {
      const int id = m.sc.sub_ch_id, br = m.sc.bit_rate;
      if (br < 8 || br % 8) continue;
      // the (address, DG flag) pairs chosen on this sub-channel: explicit ones (DG flag from the run's FIG 0/3 when it lists the
      // pair, else 0), then the FIG 0/2 TMId 3 components FIG 0/3 puts here
      std::vector<std::pair<int, int>> sel;
      auto fig03 = [&](int address) {
        for (const dabstar_packet_comp & p : R.pcomps) if (p.sub_ch_id == id && p.packet_address == address) return p.dg_flag;
        return 0;
      };
      auto add = [&](int address, int dg) {
        for (const auto & x : sel) if (x.first == address) return;
        sel.push_back({ address, dg });
      };
      for (const Recording::Cfg::PacketSel & x : R.cfg.packet_sel)
        if (x.sub_ch_id == id) add(x.address, R.cfg.auto_cfg ? fig03(x.address) : 0);
      if (R.cfg.packet_all && R.cfg.auto_cfg)
        for (const dabstar_service_comp & c : R.comps)
          if (c.tmid == 3)
            for (const dabstar_packet_comp & p : R.pcomps)
              if (p.scid == c.type && p.sub_ch_id == id && p.packet_address >= 1) add(p.packet_address, p.dg_flag);
      if (sel.empty()) continue;
      const int sub = (int)pp.subs.size();
      pp.subs.push_back(PacketSub{ dec->d_mscpacked.as<uint8_t>() + m.out_off / 8, br, (int)(m.out_len / (24 * br)), 0, 0 });
      bool fec = std::find(R.cfg.fec_ids.begin(), R.cfg.fec_ids.end(), id) != R.cfg.fec_ids.end();
      if (R.cfg.fec_all && R.cfg.auto_cfg)
        for (const dabstar_fec_scheme & x : R.fschemes) fec = fec || (x.sub_ch_id == id && x.scheme == 1);
      if (fec)
      {
        pf.streams.push_back(PfecStream{ pp.subs.back().src, nullptr, br, pp.subs.back().n_frames, 0, 0, 0 });
        fec_owner.push_back({ r, id });
        fec_sub.push_back(sub);
      }
      for (const auto & x : sel)
      {
        pp.streams.push_back(PacketStream{ sub, x.first, x.second, 0, 0, 0 });
        owner.push_back({ r, id });
      }
    }
  }
  if (pp.streams.empty()) return 0;
  if (!pf.streams.empty())
  {
    if (int e = run_packet_fec(ctx, ctx->stream, pf)) return e;
    for (size_t i = 0; i < pf.streams.size(); i++)
    {
      PacketSub & sb = pp.subs[(size_t)fec_sub[i]];
      sb.src = pf.streams[i].dst;
      sb.fec = pf.mask + pf.streams[i].slot0;
      dec->recs[fec_owner[i].first].fec_out.push_back({ fec_owner[i].second, pf.n_out[i], pf.streams[i].out0 });
    }
  }
  if (int e = run_packet(ctx, ctx->stream, pp)) return e;
  for (size_t i = 0; i < pp.streams.size(); i++)
  {
    const PacketStream & st = pp.streams[i];
    const PacketCount & c = pp.n_out[i];
    dec->recs[owner[i].first].packet_out.push_back({ owner[i].second, st.address, st.dg_flag, (int)c.groups, st.out_rec0, st.out_pay0, c.bytes,
                             packet_stats_public(c, pp.rec + st.out_rec0, c.groups) });
  }
  return 0;
}

// ---- audio: the outer code behind every selected sub-channel's Backend, on the packed MSC payload the MSC pass left on the
// device, one stream per recording and sub-channel and kind: DAB+ super-frames (Mp4Processor, mp4processor.cpp:95-334;
// run_dabplus) and MPEG layer II frames (run_mp2). A sub-channel may be selected for both; the passes read the same payload.
// Record first_frame counts the logical frames of the sub-channel's output of the run, as dabstar_decoder_msc_copy lists them.
static int audio_phase(dabstar_decoder * dec)
{
  dabstar_ctx * ctx = dec->ctx;
  DabplusPass & dp = dec->dabplus;
  Mp2Pass & mp = dec->mp2;
  dp.streams.clear();
  mp.streams.clear();
  std::vector<std::pair<int, const MscOut *>> owner[2];
  for (int r = 0; r < (int)dec->recs.size(); r++)
  {
    Recording & R = dec->recs[r];
    R.dabplus_out.clear();
    R.mp2_out.clear();
    if (!R.cfg.dabplus() && !R.cfg.mp2()) continue;
    for (const MscOut & m : R.cfg.msc)
    {
      const int id = m.sc.sub_ch_id, br = m.sc.bit_rate, n = (int)(m.out_len / (24 * br));
      const uint8_t * src = dec->d_mscpacked.as<uint8_t>() + m.out_off / 8;
      for (AudioKind k : { AUDIO_DABPLUS, AUDIO_MP2 })
      {
        const std::vector<int> & ids = k == AUDIO_MP2 ? R.cfg.mp2_ids : R.cfg.dabplus_ids;
        bool on = std::find(ids.begin(), ids.end(), id) != ids.end();
        if ((k == AUDIO_MP2 ? R.cfg.mp2_all : R.cfg.dabplus_all) && R.cfg.auto_cfg)
          for (const dabstar_service_comp & c : R.comps) on = on || (c.tmid == 0 && c.type == (k == AUDIO_MP2 ? 0 : 63) && c.sub_ch_id == id);
        if (!on || !audio_rate_ok(k, br)) continue;
        if (k == AUDIO_MP2) mp.streams.push_back(Mp2Stream{ src, br, n, 0, 0, 0 });
        else dp.streams.push_back(DabplusStream{ src, br, n, 0, 0, 0, 0 });
        owner[k].push_back({ r, &m });
      }
    }
  }
  if (!dp.streams.empty())
  {
    if (int e = run_dabplus(ctx, ctx->stream, dp)) return e;
    for (size_t i = 0; i < owner[AUDIO_DABPLUS].size(); i++)
    {
      const MscOut & m = *owner[AUDIO_DABPLUS][i].second;
      const int n = dp.n_out[i];
      dec->recs[owner[AUDIO_DABPLUS][i].first].dabplus_out.push_back({ m.sc.sub_ch_id, m.sc.bit_rate, n, dp.streams[i].out_rec0, dp.streams[i].out_pay0,
                                                                      (long long)n * 110 * (m.sc.bit_rate / 8) });
    }
  }
  if (!mp.streams.empty())
  {
    if (int e = run_mp2(ctx, ctx->stream, mp)) return e;
    for (size_t i = 0; i < owner[AUDIO_MP2].size(); i++)
    {
      const MscOut & m = *owner[AUDIO_MP2][i].second;
      dec->recs[owner[AUDIO_MP2][i].first].mp2_out.push_back({ m.sc.sub_ch_id, m.sc.bit_rate, (int)mp.n_out[i].recs, mp.streams[i].out_rec0, mp.streams[i].out_pay0,
                                                              mp.n_out[i].bytes });
    }
  }
  return packet_phase(dec);
}
// With self-configuration level 2 the recordings may be decoded again (dabstar_decoder_run): the audio phase then runs once, after the final pass.
static bool audio_after_passes(const dabstar_decoder * dec)
{
  for (const Recording & R : dec->recs) if (R.cfg.auto_cfg && R.cfg.tii_nulls) return true;
  return false;
}

static int decoder_run_pass(dabstar_decoder * dec, const void * const * iq, const int64_t * n_samples, int mem)
{
  if (!dec || !iq || !n_samples) return DABSTAR_E_INVALID;
  dabstar_ctx * ctx = dec->ctx;
  CK(cudaSetDevice(ctx->device));
  Run run(dec, mem);
  if (int e = run.stage_inputs(iq, n_samples)) return e;
  if (int e = run.reset_recordings()) return e;
  run.tr("setup done");
  while (true)
  {
    if (int e = run.time_sync()) return e;
    const bool any_wait = run.open_windows();
    if (run.win_recs.empty()) { if (any_wait) continue; break; }
    run.tr("  windows opened");
    if (int e = run.probe_first_peaks()) return e;
    if (run.win_recs.empty()) continue;
    if (int e = run.layout()) return e;
    if (int e = run.collect_frames()) return e;
    if (run.plans.empty()) continue;
    if (int e = run.heavy_pass()) return e;
    run.tr("heavy pass enqueued");
    std::vector<uint8_t> crc;
    if (int e = run.read_crc(crc)) return e;
    run.tr("heavy pass done");
    run.accept(crc);
  }
  if (int e = run.self_configure()) return e;
  if (int e = run.tii_pass()) return e;
  if (!dec->cfg.scan_mode)
  {
    if (int e = run.msc_pass()) return e;
    if (!audio_after_passes(dec))
      if (int e = audio_phase(dec)) return e; // on `st`, beside the MSC payload copies
    if (int e = run.join_copies()) return e;
  }
  std::vector<EtiRef> eti_refs;
  if (int e = run.eti_jobs(eti_refs)) return e;
  run.tr("rounds done");
  return run.finish(eti_refs);
}

// ------------------------------------------------------------------------------------------------ results
// DabProcessor::run() for every recording. With self-configuration level 2 the demapper has to know, at the null symbol of
// frame f, the CIF counter that frame's own FIC carried (dab_processor.cpp:273-285), which the batched path only learns after
// the window has been demapped. The run therefore speculates at the granularity of a pass: the first pass treats every null
// symbol as a plain one, the CIF counters it decodes give the flags, and the recordings are decoded again with them until the
// flags a pass used equal the flags it produced (one extra pass unless a FIG 0/0 is lost exactly where it matters).
extern "C" int dabstar_decoder_run(dabstar_decoder * dec, const void * const * iq, const int64_t * n_samples, int mem)
{
  if (!dec || !iq || !n_samples) return DABSTAR_E_INVALID;
  for (auto & R : dec->recs) { R.cfg.tii_flags.clear(); R.dabplus_out.clear(); R.mp2_out.clear(); R.packet_out.clear(); R.fec_out.clear(); }
  dec->dabplus.ms = 0;
  dec->dabplus.rounds = 0;
  dec->dabplus.scanned = dec->dabplus.decoded = 0;
  dec->mp2.ms = 0;
  dec->mp2.slots = 0;
  dec->packet.ms = 0;
  dec->packet.slots = 0;
  dec->pfec.ms = 0;
  dec->pfec.slots = 0;
  int rc = decoder_run_pass(dec, iq, n_samples, mem);
  double total_ms = dec->last_ms;
  for (int pass = 1; rc == 0 && pass <= 3; pass++)
  {
    bool again = false;
    for (auto & R : dec->recs)
    {
      if (!R.cfg.auto_cfg || !R.cfg.tii_nulls || R.n_slots == 0) continue;
      std::vector<uint8_t> flags((size_t)R.n_slots, 0);
      for (int f = 0; f < R.n_slots; f++) flags[f] = R.tii_null(f) ? 1 : 0;
      bool any = false;
      for (uint8_t v : flags) any = any || v;
      std::vector<uint8_t> used = R.cfg.tii_flags;
      used.resize(flags.size(), 0);
      if (any && used != flags) again = true;
      R.cfg.tii_flags = std::move(flags);
    }
    if (!again) break;
    // the recordings are resident on the device after the first pass
    std::vector<const void *> dptr(dec->recs.size());
    for (size_t r = 0; r < dec->recs.size(); r++) dptr[r] = dec->recs[r].d_iq;
    rc = decoder_run_pass(dec, dptr.data(), n_samples, DABSTAR_MEM_DEVICE);
    total_ms += dec->last_ms;
  }
  if (rc == 0 && !dec->cfg.scan_mode && audio_after_passes(dec))
  {
    rc = audio_phase(dec);
    total_ms += dec->dabplus.ms + dec->mp2.ms + dec->pfec.ms + dec->packet.ms;
  }
  dec->last_ms = total_ms;
  return rc;
}

extern "C" int dabstar_decoder_n_frames(const dabstar_decoder * dec, int recording)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  return dec->recs[recording].n_slots;
}
extern "C" int dabstar_decoder_frame_info(const dabstar_decoder * dec, int recording, dabstar_frame_info * out, int cap)
{
  if (!dec || !out || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  const Recording & R = dec->recs[recording];
  const int n = std::max(0, std::min<int>(cap, (int)R.frames.size()));
  for (int i = 0; i < n; i++) out[i] = R.frames[i];
  return n;
}
extern "C" int dabstar_decoder_fib_bits(const dabstar_decoder * dec, int recording, uint8_t * bits, uint8_t * valid)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  const Recording & R = dec->recs[recording];
  if (bits && R.n_slots > 0)
  {
    const uint8_t * p = dec->h_fibp.as<uint8_t>() + (size_t)R.slot_base * 384;
    const size_t n = (size_t)R.n_slots * 384;
    for (size_t i = 0; i < n; i++)
    {
      const unsigned v = p[i];
      uint8_t * o = bits + 8 * i;
      o[0] = (uint8_t)(v >> 7); o[1] = (v >> 6) & 1; o[2] = (v >> 5) & 1; o[3] = (v >> 4) & 1; o[4] = (v >> 3) & 1; o[5] = (v >> 2) & 1; o[6] = (v >> 1) & 1; o[7] = v & 1;
    }
  }
  if (valid) for (int i = 0; i < R.n_slots; i++) memcpy(valid + 4 * i, R.frames[i].fic_valid, 4);
  return R.n_slots;
}
extern "C" int dabstar_decoder_fib_packed(const dabstar_decoder * dec, int recording, uint8_t * packed)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  const Recording & R = dec->recs[recording];
  if (packed && R.n_slots > 0) memcpy(packed, dec->h_fibp.as<uint8_t>() + (size_t)R.slot_base * 384, (size_t)R.n_slots * 384);
  return R.n_slots;
}
extern "C" int dabstar_decoder_soft_bits(const dabstar_decoder * dec, int recording, int frame, int16_t * out)
{
  if (!dec || !out || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  const Recording & R = dec->recs[recording];
  if (frame < 0 || frame >= R.n_slots) return DABSTAR_E_INVALID;
  if (cudaSetDevice(dec->ctx->device) != cudaSuccess) return DABSTAR_E_CUDA;
  if (cudaMemcpy(out, dec->d_soft.as<int16_t>() + (size_t)(R.slot_base + frame) * FRAME_SOFT, sizeof(int16_t) * FRAME_SOFT, cudaMemcpyDeviceToHost) != cudaSuccess)
    return DABSTAR_E_CUDA;
  return 0;
}
static const MscOut * find_msc(const dabstar_decoder * dec, int recording, int sub_ch_id)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return nullptr;
  for (const auto & m : dec->recs[recording].cfg.msc) if (m.sc.sub_ch_id == sub_ch_id) return &m;
  return nullptr;
}
extern "C" int64_t dabstar_decoder_msc_size(const dabstar_decoder * dec, int recording, int sub_ch_id)
{
  const MscOut * m = find_msc(dec, recording, sub_ch_id);
  return m ? (int64_t)m->out_len : 0;
}
extern "C" int64_t dabstar_decoder_msc_copy(const dabstar_decoder * dec, int recording, int sub_ch_id, uint8_t * out, int64_t cap)
{
  const MscOut * m = find_msc(dec, recording, sub_ch_id);
  if (!m || !out || cap <= 0) return 0;
  const int64_t n = std::min<int64_t>(cap, (int64_t)m->out_len);
  const uint8_t * p = dec->h_mscp.as<uint8_t>() + m->out_off / 8; // (out_off is a multiple of 8: whole logical frames precede it)
  const int64_t whole = n >> 3;
  for (int64_t b = 0; b < whole; b++)
  {
    const unsigned v = p[b];
    uint8_t * o = out + 8 * b;
    o[0] = (uint8_t)(v >> 7); o[1] = (v >> 6) & 1; o[2] = (v >> 5) & 1; o[3] = (v >> 4) & 1; o[4] = (v >> 3) & 1; o[5] = (v >> 2) & 1; o[6] = (v >> 1) & 1; o[7] = v & 1;
  }
  for (int64_t i = 8 * whole; i < n; i++) out[i] = (uint8_t)((p[i >> 3] >> (7 - (i & 7))) & 1u);
  return n;
}
static const Recording::AudioOut * find_audio(const dabstar_decoder * dec, int recording, int sub_ch_id, AudioKind kind)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return nullptr;
  const Recording & R = dec->recs[recording];
  for (const auto & d : kind == AUDIO_MP2 ? R.mp2_out : R.dabplus_out) if (d.sub_ch_id == sub_ch_id) return &d;
  return nullptr;
}
extern "C" int dabstar_decoder_superframes(const dabstar_decoder * dec, int recording, int sub_ch_id, dabstar_superframe * out, int cap)
{
  if (!dec || cap < 0 || (!out && cap > 0)) return DABSTAR_E_INVALID;
  const Recording::AudioOut * d = find_audio(dec, recording, sub_ch_id, AUDIO_DABPLUS);
  if (!d) return dec->ctx->fail(DABSTAR_E_INVALID, "superframes: recording %d sub-channel %d was not DAB+-decoded in the last run", recording, sub_ch_id);
  for (int i = 0; i < d->n && i < cap; i++) out[i] = superframe_public(dec->dabplus.rec[d->rec0 + i]);
  return d->n;
}
extern "C" int64_t dabstar_decoder_superframe_payload(const dabstar_decoder * dec, int recording, int sub_ch_id, uint8_t * out, int64_t cap)
{
  if (!dec || cap < 0) return DABSTAR_E_INVALID;
  const Recording::AudioOut * d = find_audio(dec, recording, sub_ch_id, AUDIO_DABPLUS);
  if (!d) return dec->ctx->fail(DABSTAR_E_INVALID, "superframe_payload: recording %d sub-channel %d was not DAB+-decoded in the last run", recording, sub_ch_id);
  if (!out) return d->pay_bytes;
  const int64_t n = std::min(cap, (int64_t)d->pay_bytes);
  if (n > 0) memcpy(out, dec->dabplus.payload + d->pay0, (size_t)n);
  return n;
}
extern "C" double dabstar_decoder_dabplus_ms(const dabstar_decoder * dec, int * rounds)
{
  if (!dec) return 0.0;
  if (rounds) *rounds = dec->dabplus.rounds;
  return dec->dabplus.ms;
}
extern "C" int dabstar_decoder_mp2_frames(const dabstar_decoder * dec, int recording, int sub_ch_id, dabstar_mp2_frame * out, int cap)
{
  if (!dec || cap < 0 || (!out && cap > 0)) return DABSTAR_E_INVALID;
  const Recording::AudioOut * d = find_audio(dec, recording, sub_ch_id, AUDIO_MP2);
  if (!d) return dec->ctx->fail(DABSTAR_E_INVALID, "mp2_frames: recording %d sub-channel %d was not MP2-decoded in the last run", recording, sub_ch_id);
  for (int i = 0; i < d->n && i < cap; i++) out[i] = mp2_public(dec->mp2.rec[d->rec0 + i]);
  return d->n;
}
extern "C" int64_t dabstar_decoder_mp2_payload(const dabstar_decoder * dec, int recording, int sub_ch_id, uint8_t * out, int64_t cap)
{
  if (!dec || cap < 0) return DABSTAR_E_INVALID;
  const Recording::AudioOut * d = find_audio(dec, recording, sub_ch_id, AUDIO_MP2);
  if (!d) return dec->ctx->fail(DABSTAR_E_INVALID, "mp2_payload: recording %d sub-channel %d was not MP2-decoded in the last run", recording, sub_ch_id);
  if (!out) return d->pay_bytes;
  const int64_t n = std::min(cap, (int64_t)d->pay_bytes);
  if (n > 0) memcpy(out, dec->mp2.payload + d->pay0, (size_t)n);
  return n;
}
extern "C" double dabstar_decoder_mp2_ms(const dabstar_decoder * dec)
{
  return dec ? dec->mp2.ms : 0.0;
}
static const Recording::PacketOut * find_packet(const dabstar_decoder * dec, int recording, int sub_ch_id, int address)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return nullptr;
  for (const auto & d : dec->recs[recording].packet_out) if (d.sub_ch_id == sub_ch_id && d.address == address) return &d;
  return nullptr;
}
extern "C" int dabstar_decoder_data_groups(const dabstar_decoder * dec, int recording, int sub_ch_id, int address, dabstar_data_group * out, int cap)
{
  if (!dec || cap < 0 || (!out && cap > 0)) return DABSTAR_E_INVALID;
  const Recording::PacketOut * d = find_packet(dec, recording, sub_ch_id, address);
  if (!d) return dec->ctx->fail(DABSTAR_E_INVALID, "data_groups: recording %d sub-channel %d address %d was not packet-decoded in the last run", recording, sub_ch_id, address);
  for (int i = 0; i < d->n && i < cap; i++) out[i] = data_group_public(dec->packet.rec[d->rec0 + i]);
  return d->n;
}
extern "C" int64_t dabstar_decoder_data_group_payload(const dabstar_decoder * dec, int recording, int sub_ch_id, int address, uint8_t * out, int64_t cap)
{
  if (!dec || cap < 0) return DABSTAR_E_INVALID;
  const Recording::PacketOut * d = find_packet(dec, recording, sub_ch_id, address);
  if (!d) return dec->ctx->fail(DABSTAR_E_INVALID, "data_group_payload: recording %d sub-channel %d address %d was not packet-decoded in the last run", recording, sub_ch_id, address);
  if (!out) return d->pay_bytes;
  const int64_t n = std::min(cap, (int64_t)d->pay_bytes);
  if (n > 0) memcpy(out, dec->packet.payload + d->pay0, (size_t)n);
  return n;
}
extern "C" int dabstar_decoder_packet_stats(const dabstar_decoder * dec, int recording, int sub_ch_id, int address, dabstar_packet_stats * out)
{
  if (!dec || !out) return DABSTAR_E_INVALID;
  const Recording::PacketOut * d = find_packet(dec, recording, sub_ch_id, address);
  if (!d) return dec->ctx->fail(DABSTAR_E_INVALID, "packet_stats: recording %d sub-channel %d address %d was not packet-decoded in the last run", recording, sub_ch_id, address);
  *out = d->stats;
  return 0;
}
extern "C" double dabstar_decoder_packet_ms(const dabstar_decoder * dec)
{
  return dec ? dec->packet.ms : 0.0;
}
extern "C" int dabstar_decoder_fec_frames(const dabstar_decoder * dec, int recording, int sub_ch_id, dabstar_fec_frame * out, int cap)
{
  if (!dec || cap < 0 || (!out && cap > 0) || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  for (const auto & d : dec->recs[recording].fec_out)
    if (d.sub_ch_id == sub_ch_id)
    {
      for (int i = 0; i < d.n && i < cap; i++) out[i] = fec_frame_public(dec->pfec.rec[d.rec0 + i]);
      return d.n;
    }
  return dec->ctx->fail(DABSTAR_E_INVALID, "fec_frames: recording %d sub-channel %d had no FEC pass in the last run", recording, sub_ch_id);
}
extern "C" double dabstar_decoder_packet_fec_ms(const dabstar_decoder * dec)
{
  return dec ? dec->pfec.ms : 0.0;
}
extern "C" int dabstar_decoder_fec_schemes(const dabstar_decoder * dec, int recording, dabstar_fec_scheme * out, int cap)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size() || cap < 0 || (!out && cap > 0)) return DABSTAR_E_INVALID;
  const Recording & R = dec->recs[recording];
  if (!R.cfg.auto_cfg) return dec->ctx->fail(DABSTAR_E_INVALID, "fec_schemes: recording %d is not self-configured", recording);
  for (int i = 0; i < (int)R.fschemes.size() && i < cap; i++) out[i] = R.fschemes[i];
  return (int)R.fschemes.size();
}
extern "C" int dabstar_decoder_packet_components(const dabstar_decoder * dec, int recording, dabstar_packet_comp * out, int cap)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size() || cap < 0 || (!out && cap > 0)) return DABSTAR_E_INVALID;
  const Recording & R = dec->recs[recording];
  if (!R.cfg.auto_cfg) return dec->ctx->fail(DABSTAR_E_INVALID, "packet_components: recording %d is not self-configured", recording);
  for (int i = 0; i < (int)R.pcomps.size() && i < cap; i++) out[i] = R.pcomps[i];
  return (int)R.pcomps.size();
}
extern "C" int dabstar_decoder_dabplus_windows(const dabstar_decoder * dec, int64_t out[2])
{
  if (!dec || !out) return DABSTAR_E_INVALID;
  out[0] = dec->dabplus.scanned;
  out[1] = dec->dabplus.decoded;
  return 0;
}
extern "C" int64_t dabstar_decoder_msc_packed(const dabstar_decoder * dec, int recording, int sub_ch_id, uint8_t * out, int64_t cap)
{
  const MscOut * m = find_msc(dec, recording, sub_ch_id);
  if (!m || !out || cap <= 0) return 0; // (a negative cap would reach memcpy as a huge size)
  const int64_t n = std::min<int64_t>(cap, (int64_t)(m->out_len / 8));
  if (n > 0) memcpy(out, dec->h_mscp.as<uint8_t>() + m->out_off / 8, (size_t)n);
  return n;
}
extern "C" int dabstar_decoder_counters(const dabstar_decoder * dec, int recording, int64_t out[8])
{
  if (!dec || !out || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  const Recording & R = dec->recs[recording];
  out[0] = R.cnt_good_fibs; out[1] = R.cnt_sync_ok; out[2] = R.cnt_sync_fail; out[3] = R.pos;
  out[4] = R.cnt_windows; out[5] = R.cnt_cut; out[6] = R.n_slots; out[7] = R.cnt_heavy;
  return 0;
}
extern "C" int dabstar_decoder_quality(const dabstar_decoder * dec, int recording, float out[6])
{
  if (!dec || !out || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  if (dec->d_states.cap < sizeof(OfdmStateDev) * 2 * dec->recs.size()) return DABSTAR_E_INVALID; // no run yet
  dabstar_ctx * ctx = dec->ctx;
  CK(cudaSetDevice(ctx->device));
  const Recording & R = dec->recs[recording];
  SigmaReplay sr;
  for (const auto & fi : R.frames) sr.step(fi);
  return quality_from_state(ctx, dec->d_states.as<OfdmStateDev>() + recording + (size_t)R.state_cur * dec->recs.size(), sr.sigma, out);
}
extern "C" int dabstar_decoder_set_frame_quality(dabstar_decoder * dec, int enable)
{
  if (!dec) return DABSTAR_E_INVALID;
  dec->frame_quality = enable != 0;
  return 0;
}
extern "C" int dabstar_decoder_frame_quality(const dabstar_decoder * dec, int recording, float * out, int cap)
{
  if (!dec || !out || cap < 0 || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  if (!dec->frame_quality_run) return dec->ctx->fail(DABSTAR_E_INVALID, "frame_quality: the last run did not capture it (dabstar_decoder_set_frame_quality)");
  dabstar_ctx * ctx = dec->ctx;
  CK(cudaSetDevice(ctx->device));
  const Recording & R = dec->recs[recording];
  const int n = std::min(cap, R.n_slots);
  std::vector<FrameQual> fq((size_t)n);
  CK(cudaStreamSynchronize(ctx->stream));
  if (n > 0) CK(cudaMemcpy(fq.data(), dec->d_fq.as<FrameQual>() + R.slot_base, sizeof(FrameQual) * (size_t)n, cudaMemcpyDeviceToHost));
  SigmaReplay sr;
  for (int f = 0; f < n; f++) quality_from_sums(fq[(size_t)f], sr.step(R.frames[(size_t)f]), out + 6 * (size_t)f);
  return R.n_slots;
}
extern "C" int dabstar_decoder_enable_tii(dabstar_decoder * dec, int recording, int enable, int frames_to_count, int threshold_db, int collisions, int sub_id)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  if (enable && (frames_to_count < 1 || sub_id < 0 || sub_id > 23)) return dec->ctx->fail(DABSTAR_E_INVALID, "TII: frames_to_count %d, sub id %d", frames_to_count, sub_id);
  Recording & R = dec->recs[recording];
  R.cfg.tii.on = enable != 0;
  if (enable) { R.cfg.tii.frames_to_count = frames_to_count; R.cfg.tii.threshold_db = threshold_db; R.cfg.tii.collisions = collisions ? 1 : 0; R.cfg.tii.sub_id = sub_id; }
  return 0;
}
extern "C" int dabstar_decoder_tii_events(const dabstar_decoder * dec, int recording)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  return (int)dec->recs[recording].tii_events.size();
}
extern "C" int dabstar_decoder_tii_results(const dabstar_decoder * dec, int recording, int event, dabstar_tii_result * out, int cap, int32_t * frame)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  const Recording & R = dec->recs[recording];
  if (event < 0 || event >= (int)R.tii_events.size() || cap < 0 || (cap > 0 && !out)) return DABSTAR_E_INVALID;
  const Recording::TiiEvent & te = R.tii_events[event];
  if (frame) *frame = te.frame;
  const int n = std::min<int>(cap, (int)te.res.size());
  for (int i = 0; i < n; i++) out[i] = te.res[i];
  return (int)te.res.size();
}
extern "C" double dabstar_decoder_last_ms(const dabstar_decoder * dec) { return dec ? dec->last_ms : 0.0; }
extern "C" double dabstar_decoder_heavy_ms(const dabstar_decoder * dec, int with_fic) { return dec ? (with_fic ? dec->heavy_ms : dec->fft_demap_ms) : 0.0; }
extern "C" int dabstar_decoder_stage_ms(const dabstar_decoder * dec, double ms[8], int64_t launches[8])
{
  if (!dec || !ms || !launches) return DABSTAR_E_INVALID;
  for (int i = 0; i < 8; i++) { ms[i] = dec->stage_ms[i]; launches[i] = dec->stage_launches[i]; }
  ms[ST_MSC] += dec->stage_ms[ST_MSC_GATHER] + dec->stage_ms[ST_MSC_TRELLIS]; // the MSC pass as a whole, as before
  return 0;
}
extern "C" int dabstar_decoder_msc_kernel_ms(const dabstar_decoder * dec, double * gather_ms, double * trellis_ms)
{
  if (!dec || !gather_ms || !trellis_ms) return DABSTAR_E_INVALID;
  *gather_ms = dec->stage_ms[ST_MSC_GATHER];
  *trellis_ms = dec->stage_ms[ST_MSC_TRELLIS];
  return 0;
}

// ------------------------------------------------------------------------------------------------ long recordings: segments, stream continuation
extern "C" int dabstar_decoder_set_segmentation(dabstar_decoder * dec, int segment_frames, int warmup_frames)
{
  if (!dec || segment_frames < 0 || warmup_frames < 0) return DABSTAR_E_INVALID;
  dec->seg_frames = segment_frames;
  dec->seg_warmup = warmup_frames;
  return 0;
}
extern "C" int dabstar_decoder_set_streaming(dabstar_decoder * dec, int enable)
{
  if (!dec) return DABSTAR_E_INVALID;
  dec->streaming = enable != 0;
  return 0;
}
extern "C" int64_t dabstar_decoder_warmup_frames(const dabstar_decoder * dec, int recording)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  return (int64_t)dec->recs[recording].cnt_warmup;
}
extern "C" int64_t dabstar_decoder_consumed(const dabstar_decoder * dec, int recording)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  const Recording & R = dec->recs[recording];
  return (int64_t)(R.abs_pos0 + R.pos);
}

extern "C" int64_t dabstar_decoder_state_size(const dabstar_decoder * dec, int recording)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  return (int64_t)(sizeof(StateBlobHdr) + sizeof(OfdmStateDev) + sizeof(int16_t) * (size_t)hist_frames_after(dec->recs[recording]) * FRAME_SOFT);
}

extern "C" int64_t dabstar_decoder_export_state(dabstar_decoder * dec, int recording, void * blob, int64_t cap)
{
  if (!dec || !blob || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  dabstar_ctx * ctx = dec->ctx;
  const Recording & R = dec->recs[recording];
  if (dec->d_states.cap < sizeof(OfdmStateDev) * 2 * dec->recs.size()) return ctx->fail(DABSTAR_E_INVALID, "export_state: no run yet");
  if (R.partial_syms > 0 || (R.state == RecState::DONE && !R.held && R.pos > 0))
    return ctx->fail(DABSTAR_E_INVALID, "export_state: the run decoded into the end of its input; enable dabstar_decoder_set_streaming for chunked input");
  const int64_t need = dabstar_decoder_state_size(dec, recording);
  if (cap < need) return ctx->fail(DABSTAR_E_INVALID, "export_state: %lld bytes needed, %lld given", (long long)need, (long long)cap);
  CK(cudaSetDevice(ctx->device));
  StateBlobHdr h = blob_header(R);
  h.magic = STATE_MAGIC; h.version = 1; h.bytes = need;
  unsigned char * o = static_cast<unsigned char *>(blob);
  memcpy(o, &h, sizeof(h));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(o + sizeof(h), dec->d_states.as<OfdmStateDev>() + recording + (size_t)R.state_cur * dec->recs.size(), sizeof(OfdmStateDev), cudaMemcpyDeviceToHost));
  if (h.hist > 0)
    CK(cudaMemcpy(o + sizeof(h) + sizeof(OfdmStateDev), dec->d_soft.as<int16_t>() + (size_t)(R.slot_base + R.n_slots - h.hist) * FRAME_SOFT,
                  sizeof(int16_t) * (size_t)h.hist * FRAME_SOFT, cudaMemcpyDeviceToHost));
  return need;
}

extern "C" int dabstar_decoder_import_state(dabstar_decoder * dec, int recording, const void * blob, int64_t size, int64_t lead_samples)
{
  if (!dec || !blob || recording < 0 || recording >= (int)dec->recs.size() || lead_samples < 0) return DABSTAR_E_INVALID;
  dabstar_ctx * ctx = dec->ctx;
  StateBlobHdr h;
  if (size < (int64_t)sizeof(h)) return ctx->fail(DABSTAR_E_INVALID, "import_state: truncated blob");
  memcpy(&h, blob, sizeof(h));
  if (h.magic != STATE_MAGIC || h.version != 1 || h.bytes > size || h.hist < 0 || h.hist > 4 ||
      h.bytes != (int64_t)(sizeof(h) + sizeof(OfdmStateDev) + sizeof(int16_t) * (size_t)h.hist * FRAME_SOFT) || h.rec_state < 0 || h.rec_state > 2)
    return ctx->fail(DABSTAR_E_INVALID, "import_state: not a state blob of this library version");
  if (lead_samples > h.stream_pos) return ctx->fail(DABSTAR_E_INVALID, "import_state: %lld lead samples in front of stream position %lld", (long long)lead_samples, (long long)h.stream_pos);
  dabstar_decoder::Resume & rs = dec->resume[recording];
  rs = dabstar_decoder::Resume();
  if (h.rec_state == 2) return 0; // nothing had been decoded: the next run starts the stream
  rs.on = true;
  rs.hdr = h;
  rs.lead = lead_samples;
  const unsigned char * in = static_cast<const unsigned char *>(blob) + sizeof(h);
  rs.ofdm.assign(in, in + sizeof(OfdmStateDev));
  rs.soft.resize((size_t)h.hist * FRAME_SOFT);
  if (h.hist > 0) memcpy(rs.soft.data(), in + sizeof(OfdmStateDev), sizeof(int16_t) * rs.soft.size());
  return 0;
}
