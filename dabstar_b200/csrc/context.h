// context.h — what the stage taps (engine.cu) and the whole-path decoder (decoder.cu) share: buffers, the context, the
// staging helpers and the error macros.
#pragma once
#include "../../include/dabstar_b200.h"
#include "kernels.h"
#include "hostpool.h"

#include <algorithm>
#include <array>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

struct DevBuf
{
  void * p = nullptr;
  size_t cap = 0;
  ~DevBuf() { if (p) cudaFree(p); }
  cudaError_t reserve(size_t bytes)
  {
    if (bytes <= cap) return cudaSuccess;
    if (p) { cudaFree(p); p = nullptr; cap = 0; }
    const size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  template <typename T> T * as() const { return static_cast<T *>(p); }
};

// pinned host memory for result read-back (pageable memory makes cudaMemcpyAsync synchronous and ~3x slower)
struct HostBuf
{
  void * p = nullptr;
  size_t cap = 0;
  ~HostBuf() { if (p) cudaFreeHost(p); }
  cudaError_t reserve(size_t bytes)
  {
    if (bytes <= cap) return cudaSuccess;
    if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
    cudaError_t e = cudaHostAlloc(&p, bytes + bytes / 8 + 256, cudaHostAllocMapped | cudaHostAllocPortable);
    if (e == cudaSuccess) cap = bytes + bytes / 8 + 256;
    return e;
  }
  template <typename T> T * as() const { return static_cast<T *>(p); }
};

// The DAB+ outer code over a table of streams (run_dabplus): device work buffers, and the result in pinned host memory
struct DabplusPass
{
  std::vector<dab::DabplusStream> streams; // the caller sets src (device, packed frames), bit_rate and n_frames
  // results of the last run_dabplus: per stream the attempted super-frames' records and decoded bytes, in stream order
  std::vector<int> n_out;
  const dab::SuperFrameRec * rec = nullptr; // sum(n_out) records ...
  const uint8_t * payload = nullptr;        // ... and their super-frames (stream i's at streams[i].out_pay0)
  long long scanned = 0, decoded = 0;       // windows whose raw header was checked / that went through Reed-Solomon
  int rounds = 0;                           // walks (a walk that lists nothing new ends the pass)
  double ms = 0;                            // device time of the pass
  DevBuf d_streams, d_state, d_att, d_meta, d_list, d_slot, d_ler, d_rec, d_pay, d_out;
  HostBuf h_meta, h_out;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  ~DabplusPass()
  {
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
  }
};

// MPEG layer II audio frames over a table of streams (run_mp2): device work buffers, and the result in pinned host memory
struct Mp2Pass
{
  std::vector<dab::Mp2Stream> streams; // the caller sets src (device, packed frames), bit_rate and n_frames
  // results of the last run_mp2: per stream its records and the bytes of its OK frames, in stream order
  std::vector<dab::Mp2Count> n_out;
  const dab::Mp2Rec * rec = nullptr; // sum(n_out.recs) records (stream i's from streams[i].out_rec0) ...
  const uint8_t * payload = nullptr; // ... and the OK frames' bytes (stream i's at streams[i].out_pay0)
  long long slots = 0;               // logical frames classified
  double ms = 0;                     // device time of the pass
  DevBuf d_streams, d_cls, d_crc, d_hdr, d_stage, d_stage_off, d_cnt, d_out;
  HostBuf h_cnt, h_out;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  ~Mp2Pass()
  {
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
  }
};

// Packet-mode data groups over a table of sub-channels and (sub-channel, address) streams (run_packet): device work buffers, and
// the result in pinned host memory
struct PacketPass
{
  std::vector<dab::PacketSub> subs;       // the caller sets src (device, packed frames), bit_rate and n_frames
  std::vector<dab::PacketStream> streams; // ... and sub, address and dg_flag
  // results of the last run_packet: per stream its counters, records and group bytes, in stream order
  std::vector<dab::PacketCount> n_out;
  const dab::DgRec * rec = nullptr;       // sum(n_out.groups) records (stream i's from streams[i].out_rec0) ...
  const uint8_t * payload = nullptr;      // ... and the groups' bytes (stream i's at streams[i].out_pay0)
  long long slots = 0;                    // packet slots parsed
  double ms = 0;                          // device time of the pass
  DevBuf d_subs, d_streams, d_slots, d_stage, d_cnt, d_out;
  HostBuf h_cnt, h_out;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  ~PacketPass()
  {
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
  }
};

// Packet-mode FEC over a table of streams (run_packet_fec): device work buffers, the corrected copies and the FEC mask the packet
// pass reads, and the frame records in pinned host memory
struct PfecPass
{
  std::vector<dab::PfecStream> streams; // the caller sets src (device, packed frames, all in one allocation), bit_rate and n_frames;
                                        // the pass sets dst
  // results of the last run_packet_fec: per stream its frame records, in stream order
  std::vector<int> n_out;
  const dab::PfecRec * rec = nullptr;   // sum(n_out) records (stream i's from streams[i].out0)
  const uint8_t * mask = nullptr;       // device: one byte per slot (stream i's from streams[i].slot0), 1 on FEC packets
  long long slots = 0;                  // 24-byte slots scanned
  double ms = 0;                        // device time of the pass
  std::vector<uint8_t> tables;          // GF(2^8) tables (pfec.cuh: PfecTables), uploaded once to d_tab
  DevBuf d_streams, d_copy, d_code, d_start, d_mask, d_stage, d_cnt, d_rec, d_tab;
  HostBuf h_cnt, h_rec;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  ~PfecPass()
  {
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
  }
};

struct dabstar_ctx
{
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::string err;
  unsigned long long launches = 0;
  dab::DeviceTables tab{};
  std::vector<int16_t> h_bin_signed;
  std::vector<float2> h_prs;
  std::vector<dab::VitProfile> profiles; // [0] = FIC
  std::map<long long, int> profile_index;
  DevBuf d_profiles;
  std::vector<uint32_t> step_tab;   // vit_step_entry of every profile, back to back (VitProfile::tab_off)
  DevBuf d_step_tab;
  bool profiles_dirty = true;
  DevBuf scratch[8];
  DevBuf demap_ring;    // exchange ring of the sliced demapper
  DevBuf vit_ws;        // symbols + decision words of the thread-per-code-word Viterbi
  DevBuf d_gf, d_fc_syn; // DAB+ outer code: GF(2^8) / Fire code tables (built on first use)
  DabplusPass dabplus;   // dabstar_dabplus_decode's pass
  Mp2Pass mp2;           // dabstar_mp2_frames's pass
  PacketPass packet;     // dabstar_packet_groups's pass
  PfecPass pfec;         // dabstar_packet_fec's and dabstar_packet_groups_fec's FEC pass
  HostBuf arena;        // pinned staging of small uploads; reused after every stream synchronisation
  size_t arena_off = 0;
  std::unique_ptr<dab::HostPool> pool; // host threads of the per-recording control loops (created by the first decoder run)
  dab::HostPool & host_pool()
  {
    if (!pool)
    {
      const char * ev = getenv("DABSTAR_HOST_THREADS"); // total threads incl. the caller (1 = serial)
      const char * sp = getenv("DABSTAR_HOST_SPIN_US"); // how long an idle worker polls before it sleeps (hostpool.h)
      pool.reset(new dab::HostPool(ev ? std::max(0, atoi(ev) - 1) : dab::HostPool::default_workers(), sp ? std::max(0, atoi(sp)) : 1000));
    }
    return *pool;
  }

  int fail(int code, const char * fmt, ...)
  {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    err = buf;
    return code;
  }
  int cuda_fail(cudaError_t e, const char * what) { return fail(DABSTAR_E_CUDA, "%s: %s", what, cudaGetErrorString(e)); }
};

struct dabstar_tii
{
  dabstar_ctx * ctx = nullptr;
  int n = 0;
  int collisions = 0, sub_id_coll = 0;
  DevBuf null_sum, decoded, tables, results;
  DevBuf staging;
};

#define CK(call)                                                     \
  do {                                                               \
    cudaError_t e_ = (call);                                         \
    if (e_ != cudaSuccess) return ctx->cuda_fail(e_, #call);         \
  } while (0)

// cudaStreamSynchronize of the context's stream; every staged upload has been consumed afterwards
int sync_stream(dabstar_ctx * ctx);
// Asynchronous small host->device copy on the context's stream (see k_upload). `src` may be reused on return.
int upload(dabstar_ctx * ctx, void * dst, const void * src, size_t bytes);
// The same in two halves: upload_begin hands out the staging area (the caller fills it, e.g. from several threads),
// upload_commit queues the copy kernel.
int upload_begin(dabstar_ctx * ctx, size_t bytes, unsigned char ** stage);
int upload_commit(dabstar_ctx * ctx, void * dst, const unsigned char * stage, size_t bytes);
#define UP(dst, src, bytes) do { if (int r_ = upload(ctx, (dst), (src), (bytes))) return r_; } while (0)
#define SYNC() do { if (int r_ = sync_stream(ctx)) return r_; } while (0)

// The super-frames Mp4Processor attempts in every stream of p.streams, decoded on the device (dabplus_kernels.cu): scan the
// Fire code of every window, then alternate walk and decode until a walk lists no window without an outcome (one small
// read-back per round), then compact the attempted windows in stream order and copy them to p.h_out. Runs on `s`.
int run_dabplus(dabstar_ctx * ctx, cudaStream_t s, DabplusPass & p);
inline dabstar_superframe superframe_public(const dab::SuperFrameRec & r)
{
  dabstar_superframe o;
  o.first_frame = r.first_frame; o.ok = r.ok; o.rs_errors = r.rs_errors; o.rs_corrections = r.rs_corrections; o.fc_corrected = r.fc_corrected;
  o.dac_rate = r.dac_rate; o.sbr_flag = r.sbr_flag; o.aac_channel_mode = r.aac_channel_mode; o.ps_flag = r.ps_flag; o.mpeg_surround = r.mpeg_surround;
  o.num_aus = r.num_aus;
  for (int i = 0; i < 7; i++) o.au_start[i] = r.au_start[i];
  for (int i = 0; i < 6; i++) o.au_state[i] = r.au_state[i];
  return o;
}

// The audio-frame slots of every stream of p.streams, on the device (mp2_kernels.cu): classify every logical frame, walk each
// stream (one read-back of the per-stream counts), then compact the records and OK frames in stream order and copy them to
// p.h_out. Runs on `s`.
int run_mp2(dabstar_ctx * ctx, cudaStream_t s, Mp2Pass & p);
inline dabstar_mp2_frame mp2_public(const dab::Mp2Rec & r)
{
  dabstar_mp2_frame o;
  o.first_frame = r.first_frame; o.n_frames = r.n_frames; o.status = r.status; o.header = r.header; o.crc_stored = r.crc_stored; o.crc_computed = r.crc_computed;
  return o;
}

// The data groups of every stream of p.streams, on the device (packet_kernels.cu): parse every logical frame's packets once per
// sub-channel, walk each stream (one read-back of the per-stream counters), then compact the records and group bytes in stream
// order and copy them to p.h_out. Runs on `s`.
int run_packet(dabstar_ctx * ctx, cudaStream_t s, PacketPass & p);
// The FEC frames of every stream of p.streams, on the device (pfec_kernels.cu): copy the span of all streams' bytes to p.d_copy
// (one cudaMemcpyAsync), locate the FEC-packet runs of every slot, list each stream's runs (one read-back of the per-stream counts), then
// correct the rows of every complete frame in the copies and copy the records to p.h_rec. The packet pass then reads the copies
// with p.mask (PacketSub::fec). Runs on `s`.
int run_packet_fec(dabstar_ctx * ctx, cudaStream_t s, PfecPass & p);
inline dabstar_fec_frame fec_frame_public(const dab::PfecRec & r)
{
  static_assert(sizeof(dab::PfecRec) == sizeof(dabstar_fec_frame), "PfecRec mirrors dabstar_fec_frame");
  dabstar_fec_frame o;
  memcpy(&o, &r, sizeof o);
  return o;
}
inline dabstar_data_group data_group_public(const dab::DgRec & r)
{
  static_assert(sizeof(dab::DgRec) == sizeof(dabstar_data_group), "DgRec mirrors dabstar_data_group");
  dabstar_data_group o;
  memcpy(&o, &r, sizeof o);
  return o;
}
// the counters of a stream; the groups by status are counted from its n records
inline dabstar_packet_stats packet_stats_public(const dab::PacketCount & c, const dab::DgRec * rec, long long n)
{
  dabstar_packet_stats o{};
  o.packets = c.packets; o.crc_errors = c.crc_errors; o.bad_length = c.bad_length; o.cut = c.cut; o.padding = c.padding; o.command = c.command;
  o.other_address = c.other_address; o.continuity_breaks = c.continuity_breaks; o.abandoned = c.abandoned; o.dropped = c.dropped;
  for (long long i = 0; i < n; i++)
    if (rec[i].status >= 0 && rec[i].status < 5) o.groups[rec[i].status]++;
  return o;
}

int get_profile(dabstar_ctx * ctx, int short_form, int bit_rate, int prot_level);
int sync_profiles(dabstar_ctx * ctx);
int reserve_viterbi_ws(dabstar_ctx * ctx, int n_jobs, int max_steps);
int run_viterbi_jobs(dabstar_ctx * ctx, const std::vector<dab::VitJob> & jobs, int max_steps, const int16_t * d_soft, uint8_t * d_bits,
                     uint8_t * d_crc, int * d_ber, DevBuf & jobbuf);
// full: constructor state of OfdmDecoder; otherwise its reset()
int ofdm_state_init(dabstar_ctx * ctx, dab::OfdmStateDev * dev, bool full, int count = 1);
// The figures OfdmDecoder hands to signal_show_lcd_data, from the sums of a state or of one frame.
void quality_from_sums(const dab::FrameQual & q, float sigma_sq_freq_corr, float out[6]);
int quality_from_state(dabstar_ctx * ctx, const dab::OfdmStateDev * dev, float sigma_sq_freq_corr, float out[6]);
