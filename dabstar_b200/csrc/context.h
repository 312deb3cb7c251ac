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
