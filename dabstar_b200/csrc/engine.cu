// engine.cu — context, stage taps and the whole-path decoder behind include/dabstar_b200.h.
//
// The decoder restates DabProcessor's control flow (main/dab_processor.cpp:110-442) as a host-side state machine
// per recording that drives BATCHED kernels: all recordings advance in lock step, and inside a recording the
// frame-to-frame dependencies (frame position from the PRS peak, AFC from the cyclic-prefix phase, coarse AFC
// gated by the FIC success counter) are handled by speculation: a window of frames is laid out assuming the PRS
// peak stays at T_g and the FIC keeps decoding, every kernel runs over the whole window, and the per-frame PRS
// peaks / FIB CRCs are verified afterwards. A window that fails verification is replayed from a state snapshot
// with the length that verified. Acquisition (first frames, or after a sync loss) runs with windows of one frame.
#include "../../include/dabstar_b200.h"
#include "kernels.h"
#include "tables.h"
#include "hostpool.h"
#include "fft2048.cuh"

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

using namespace dab;

// ------------------------------------------------------------------------------------------------ helpers
namespace
{
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
} // namespace

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

// Small host->device transfers (descriptors, job lists) go through a pinned, device-mapped arena and a copy KERNEL
// instead of cudaMemcpyAsync: the H2D copy engine is a FIFO shared by all streams, and while a recording upload is
// queued on it (dabstar_decoder_run with host input) a 6 KB descriptor copy would wait behind hundreds of megabytes.
__global__ void k_upload(unsigned char * __restrict__ dst, const unsigned char * __restrict__ src, size_t bytes)
{
  const size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  if ((((size_t)dst | (size_t)src) & 15) == 0)
  {
    const size_t n16 = bytes >> 4;
    for (size_t i = i0; i < n16; i += stride) reinterpret_cast<uint4 *>(dst)[i] = reinterpret_cast<const uint4 *>(src)[i];
    for (size_t i = (n16 << 4) + i0; i < bytes; i += stride) dst[i] = src[i];
  }
  else for (size_t i = i0; i < bytes; i += stride) dst[i] = src[i];
}

__global__ void k_ofdm_state_init(OfdmStateDev * __restrict__ st, int count, int full)
{
  // full: constructor state (mMeanValue = 1); otherwise reset(), which keeps mMeanValue (ofdm_decoder.cpp:90-101)
  const int per = (int)(sizeof(OfdmStateDev) / sizeof(float));
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)count * per; i += (size_t)gridDim.x * blockDim.x)
  {
    float * f = reinterpret_cast<float *>(st) + i;
    const bool is_mean_value = (i % per) == offsetof(OfdmStateDev, mean_value) / sizeof(float);
    const bool is_pow_carry = (i % per) == offsetof(OfdmStateDev, pow_carry) / sizeof(float);
    if (is_mean_value) { if (full) *f = 1.0f; }
    else *f = is_pow_carry ? 1.0f : 0.0f; // mMeanPowerOvrAll = 1 (ofdm_decoder.h:99, ofdm_decoder.cpp:98)
  }
}

struct dabstar_ctx
{
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::string err;
  unsigned long long launches = 0;
  DeviceTables tab{};
  std::vector<int16_t> h_bin_signed;
  std::vector<float2> h_prs;
  std::vector<VitProfile> profiles; // [0] = FIC
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

#define CK(call)                                                     \
  do {                                                               \
    cudaError_t e_ = (call);                                         \
    if (e_ != cudaSuccess) return ctx->cuda_fail(e_, #call);         \
  } while (0)

namespace
{
// cudaStreamSynchronize of the context's stream; every staged upload has been consumed afterwards
int sync_stream(dabstar_ctx * ctx)
{
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->arena_off = 0;
  return 0;
}

// Asynchronous small host->device copy on the context's stream (see k_upload). `src` may be reused on return.
int upload(dabstar_ctx * ctx, void * dst, const void * src, size_t bytes)
{
  if (bytes == 0) return 0;
  const size_t need = (bytes + 255) & ~(size_t)255;
  if (ctx->arena.cap < need || ctx->arena_off + need > ctx->arena.cap)
  {
    if (int r = sync_stream(ctx)) return r;
    if (ctx->arena.cap < need) CK(ctx->arena.reserve(std::max<size_t>(need, (size_t)8 << 20)));
  }
  unsigned char * stage = ctx->arena.as<unsigned char>() + ctx->arena_off;
  memcpy(stage, src, bytes);
  ctx->arena_off += need;
  const int grid = (int)std::min<size_t>(64, (bytes / 16 + 255) / 256 + 1);
  k_upload<<<grid, 256, 0, ctx->stream>>>(static_cast<unsigned char *>(dst), stage, bytes);
  ctx->launches++;
  CK(cudaGetLastError());
  return 0;
}
// The same in two halves: upload_begin hands out the staging area (the caller fills it, e.g. from several threads),
// upload_commit queues the copy kernel.
int upload_begin(dabstar_ctx * ctx, size_t bytes, unsigned char ** stage)
{
  const size_t need = (bytes + 255) & ~(size_t)255;
  if (ctx->arena.cap < need || ctx->arena_off + need > ctx->arena.cap)
  {
    if (int r = sync_stream(ctx)) return r;
    if (ctx->arena.cap < need) CK(ctx->arena.reserve(std::max<size_t>(need, (size_t)8 << 20)));
  }
  *stage = ctx->arena.as<unsigned char>() + ctx->arena_off;
  ctx->arena_off += need;
  return 0;
}
int upload_commit(dabstar_ctx * ctx, void * dst, const unsigned char * stage, size_t bytes)
{
  const int grid = (int)std::min<size_t>(64, (bytes / 16 + 255) / 256 + 1);
  k_upload<<<grid, 256, 0, ctx->stream>>>(static_cast<unsigned char *>(dst), stage, bytes);
  ctx->launches++;
  CK(cudaGetLastError());
  return 0;
}
#define UP(dst, src, bytes) do { if (int r_ = upload(ctx, (dst), (src), (bytes))) return r_; } while (0)
#define SYNC() do { if (int r_ = sync_stream(ctx)) return r_; } while (0)

// Registers a profile: appends its step table (viterbi.cuh: vit_step_entry_make) and returns its index.
int push_profile(dabstar_ctx * ctx, VitProfile p)
{
  p.tab_off = (int)ctx->step_tab.size();
  const int steps = p.n_bits + 6;
  int kept = 0;
  for (int t = 0; t < steps; t++)
  {
    unsigned mask = 0;
    for (int g = 0; g < 4; g++) if (vit_src_index(p, 4 * t + g) >= 0) mask |= 1u << g;
    ctx->step_tab.push_back(vit_step_entry_make(kept, mask));
    kept += __builtin_popcount(mask);
  }
  ctx->profiles.push_back(p);
  ctx->profiles_dirty = true;
  return (int)ctx->profiles.size() - 1;
}

int get_profile(dabstar_ctx * ctx, int short_form, int bit_rate, int prot_level)
{
  const long long key = ((long long)(short_form ? 1 : 0) << 40) | ((long long)bit_rate << 8) | (long long)(prot_level & 0xff);
  auto it = ctx->profile_index.find(key);
  if (it != ctx->profile_index.end()) return it->second;
  VitProfile p;
  if (!make_msc_profile(short_form, bit_rate, prot_level, p)) return -1;
  const int idx = push_profile(ctx, p);
  ctx->profile_index[key] = idx;
  return idx;
}

int get_identity_profile(dabstar_ctx * ctx, int n_bits)
{
  const long long key = (2LL << 40) | (long long)n_bits;
  auto it = ctx->profile_index.find(key);
  if (it != ctx->profile_index.end()) return it->second;
  const int idx = push_profile(ctx, make_identity_profile(n_bits));
  ctx->profile_index[key] = idx;
  return idx;
}

int sync_profiles(dabstar_ctx * ctx)
{
  if (!ctx->profiles_dirty) return 0;
  CK(ctx->d_profiles.reserve(sizeof(VitProfile) * std::max<size_t>(ctx->profiles.size(), 64)));
  CK(cudaMemcpyAsync(ctx->d_profiles.p, ctx->profiles.data(), sizeof(VitProfile) * ctx->profiles.size(), cudaMemcpyHostToDevice, ctx->stream));
  CK(ctx->d_step_tab.reserve(sizeof(uint32_t) * std::max<size_t>(ctx->step_tab.size(), 4096)));
  CK(cudaMemcpyAsync(ctx->d_step_tab.p, ctx->step_tab.data(), sizeof(uint32_t) * ctx->step_tab.size(), cudaMemcpyHostToDevice, ctx->stream));
  SYNC();
  ctx->profiles_dirty = false;
  return 0;
}

// Brings `bytes` at `src` (host or device per `mem`) into device memory; returns the device pointer.
int stage_in(dabstar_ctx * ctx, DevBuf & buf, const void * src, size_t bytes, int mem, const void ** out)
{
  if (mem == DABSTAR_MEM_DEVICE) { *out = src; return 0; }
  CK(buf.reserve(bytes));
  CK(cudaMemcpyAsync(buf.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  *out = buf.p;
  return 0;
}
int stage_out_begin(dabstar_ctx * ctx, DevBuf & buf, void * dst, size_t bytes, int mem, void ** out)
{
  if (mem == DABSTAR_MEM_DEVICE) { *out = dst; return 0; }
  CK(buf.reserve(bytes));
  *out = buf.p;
  return 0;
}
int stage_out_end(dabstar_ctx * ctx, const void * dev, void * dst, size_t bytes, int mem)
{
  if (mem == DABSTAR_MEM_HOST) CK(cudaMemcpyAsync(dst, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
} // namespace

// ------------------------------------------------------------------------------------------------ context
extern "C" int dabstar_abi_version(void) { return DABSTAR_ABI_VERSION; }

extern "C" int dabstar_create(dabstar_ctx ** out, int device, void * stream)
{
  if (!out) return DABSTAR_E_INVALID;
  *out = nullptr;
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0 || device < 0 || device >= n_dev) return DABSTAR_E_CUDA; // no CPU fallback
  std::unique_ptr<dabstar_ctx> ctx(new dabstar_ctx);
  ctx->device = device;
  if (cudaSetDevice(device) != cudaSuccess) return DABSTAR_E_CUDA;
  if (stream) ctx->stream = (cudaStream_t)stream;
  else
  {
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) return DABSTAR_E_CUDA;
    ctx->own_stream = true;
  }
  // tables
  ctx->h_bin_signed.resize(K_CARR);
  host_freq_interleaver(ctx->h_bin_signed.data());
  ctx->h_prs.resize(T_U);
  host_phase_table(ctx->h_prs.data());
  std::vector<float2> w(T_U);
  host_w2048(w.data());
  std::vector<int16_t> bin_idx(K_CARR), rel(K_CARR);
  for (int k = 0; k < K_CARR; k++)
  {
    const int b = ctx->h_bin_signed[k];
    bin_idx[k] = (int16_t)(b < 0 ? b + T_U : b);
    rel[k] = (int16_t)(b < 0 ? b + K_CARR / 2 : b + K_CARR / 2 - 1); // ofdm_decoder.cpp:169-180
  }
  // energy dispersal: as long as the longest logical frame make_msc_profile accepts (24 x 1024 bits; the reference builds
  // 24 x bitRate entries per Backend, backend.cpp:72-83) plus slack for the kernels' 8-byte loads
  std::vector<uint8_t> prbs(PRBS_LEN);
  host_prbs(prbs.data(), PRBS_LEN);
  bool ok = true;
  ok = ok && cudaMalloc(&ctx->tab.w2048, sizeof(float2) * T_U) == cudaSuccess;
  ok = ok && cudaMalloc(&ctx->tab.prs, sizeof(float2) * T_U) == cudaSuccess;
  ok = ok && cudaMalloc(&ctx->tab.ref_arg_conj, sizeof(float2) * T_U) == cudaSuccess;
  ok = ok && cudaMalloc(&ctx->tab.bin_of_k, sizeof(int16_t) * K_CARR) == cudaSuccess;
  ok = ok && cudaMalloc(&ctx->tab.rel_of_k, sizeof(int16_t) * K_CARR) == cudaSuccess;
  ok = ok && cudaMalloc(&ctx->tab.prbs, PRBS_LEN) == cudaSuccess;
  std::vector<uint16_t> slot_w(16 * FFT_THREADS), slot_r(K_CARR);
  host_fft_epilogue_layout(bin_idx.data(), slot_w.data(), slot_r.data());
  ok = ok && cudaMalloc(&ctx->tab.fft_slot_w, sizeof(uint16_t) * slot_w.size()) == cudaSuccess;
  ok = ok && cudaMalloc(&ctx->tab.fft_slot_r, sizeof(uint16_t) * slot_r.size()) == cudaSuccess;
  ok = ok && cudaMemcpy(ctx->tab.fft_slot_w, slot_w.data(), sizeof(uint16_t) * slot_w.size(), cudaMemcpyHostToDevice) == cudaSuccess;
  ok = ok && cudaMemcpy(ctx->tab.fft_slot_r, slot_r.data(), sizeof(uint16_t) * slot_r.size(), cudaMemcpyHostToDevice) == cudaSuccess;
  ok = ok && cudaMemcpy(ctx->tab.w2048, w.data(), sizeof(float2) * T_U, cudaMemcpyHostToDevice) == cudaSuccess;
  ok = ok && cudaMemcpy(ctx->tab.prs, ctx->h_prs.data(), sizeof(float2) * T_U, cudaMemcpyHostToDevice) == cudaSuccess;
  ok = ok && cudaMemcpy(ctx->tab.bin_of_k, bin_idx.data(), sizeof(int16_t) * K_CARR, cudaMemcpyHostToDevice) == cudaSuccess;
  ok = ok && cudaMemcpy(ctx->tab.rel_of_k, rel.data(), sizeof(int16_t) * K_CARR, cudaMemcpyHostToDevice) == cudaSuccess;
  ok = ok && cudaMemcpy(ctx->tab.prbs, prbs.data(), PRBS_LEN, cudaMemcpyHostToDevice) == cudaSuccess;
  ok = ok && launch_init_ref_arg(ctx->stream, ctx->tab, &ctx->launches) == cudaSuccess;
  ok = ok && cudaStreamSynchronize(ctx->stream) == cudaSuccess;
  if (!ok) { dabstar_destroy(ctx.release()); return DABSTAR_E_CUDA; }
  push_profile(ctx.get(), make_fic_profile());
  *out = ctx.release();
  return DABSTAR_OK;
}

extern "C" void dabstar_destroy(dabstar_ctx * ctx)
{
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaFree(ctx->tab.w2048); cudaFree(ctx->tab.prs); cudaFree(ctx->tab.ref_arg_conj);
  cudaFree(ctx->tab.bin_of_k); cudaFree(ctx->tab.rel_of_k); cudaFree(ctx->tab.prbs); cudaFree(ctx->tab.fft_slot_w); cudaFree(ctx->tab.fft_slot_r);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

extern "C" const char * dabstar_last_error(const dabstar_ctx * ctx) { return ctx ? ctx->err.c_str() : "null context"; }
extern "C" uint64_t dabstar_kernel_launches(const dabstar_ctx * ctx) { return ctx ? ctx->launches : 0; }

// ------------------------------------------------------------------------------------------------ tables
extern "C" int dabstar_freq_interleaver(dabstar_ctx * ctx, int16_t out[1536])
{
  if (!ctx || !out) return DABSTAR_E_INVALID;
  memcpy(out, ctx->h_bin_signed.data(), sizeof(int16_t) * K_CARR);
  return 0;
}
extern "C" int dabstar_phase_table(dabstar_ctx * ctx, float out[4096])
{
  if (!ctx || !out) return DABSTAR_E_INVALID;
  memcpy(out, ctx->h_prs.data(), sizeof(float2) * T_U);
  return 0;
}
extern "C" int dabstar_protection_addresses(dabstar_ctx * ctx, int short_form, int bit_rate, int prot_level, int32_t * addr, int cap)
{
  if (!ctx || !addr) return DABSTAR_E_INVALID;
  VitProfile p;
  if (!make_msc_profile(short_form, bit_rate, prot_level, p)) return ctx->fail(DABSTAR_E_INVALID, "unknown protection profile %d/%d/%d", short_form, bit_rate, prot_level);
  return profile_addresses(p, addr, cap);
}

// ------------------------------------------------------------------------------------------------ ingest (I1)
extern "C" int dabstar_sample_format_bytes(const dabstar_sample_format * fmt)
{
  if (!fmt || fmt->iq_order < 0 || fmt->iq_order > 3) return 0;
  int b;
  switch (fmt->container)
  {
  case DABSTAR_CONTAINER_INT8: case DABSTAR_CONTAINER_UINT8: case DABSTAR_CONTAINER_UINT8_PCM: b = 1; break;
  case DABSTAR_CONTAINER_INT16: b = 2; break;
  case DABSTAR_CONTAINER_INT24: b = 3; break;
  case DABSTAR_CONTAINER_INT32: case DABSTAR_CONTAINER_FLOAT32: case DABSTAR_CONTAINER_INT32_PCM: b = 4; break;
  default: return 0;
  }
  return fmt->iq_order <= DABSTAR_ORDER_QI ? 2 * b : b;
}

extern "C" int dabstar_ingest_convert(dabstar_ctx * ctx, const void * src, const dabstar_sample_format * fmt, int64_t n_samples, float * dst, int mem)
{
  if (!ctx || !src || !fmt || !dst || n_samples < 0) return DABSTAR_E_INVALID;
  const int elem = dabstar_sample_format_bytes(fmt);
  if (elem == 0) return ctx->fail(DABSTAR_E_INVALID, "unknown sample format %d / order %d", fmt->container, fmt->iq_order);
  if (n_samples == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  const int width = fmt->container == DABSTAR_CONTAINER_INT16 ? 16 : (fmt->container == DABSTAR_CONTAINER_INT24 ? 24 : 32);
  const int bits = fmt->bits_per_channel > 0 ? fmt->bits_per_channel : width;
  if (bits < 1 || bits > 32) return ctx->fail(DABSTAR_E_INVALID, "bits_per_channel %d", fmt->bits_per_channel);
  // f32 scaler = f32(shift(nrBits)), shift(a) = 2^(a-1) in i32 (xml_reader.cpp:43-51): 32 bits wrap to -2^31, so int32
  // files come out negated exactly as the reference reads them; x / (+-2^k) == x * (+-2^-k) exactly
  const float inv_scaler = 1.0f / (float)(int32_t)(1u << (bits - 1));
  const float * d_lut = nullptr;
  if (fmt->container <= DABSTAR_CONTAINER_UINT8 || fmt->container == DABSTAR_CONTAINER_UINT8_PCM)
  {
    float lut[256];
    for (int i = 0; i < 256; i++)
    {
      if (fmt->container == DABSTAR_CONTAINER_UINT8_PCM) lut[i] = (float)(i - 128) / 128.0f;                 // libsndfile pcm.c uc2f: (v - 128) / 128
      else if (fmt->container == DABSTAR_CONTAINER_UINT8) lut[i] = ((float)i - 127.38f) / 128.0f;            // mapTable, xml_reader.cpp:93-96
      else if (fmt->iq_order == DABSTAR_ORDER_IQ) lut[i] = (float)(int8_t)i / 127.0f;                        // xml_reader.cpp:266
      else lut[i] = (float)((double)(int8_t)i / 127.0);                                                      // xml_reader.cpp:411,560,690: double division
    }
    CK(ctx->scratch[5].reserve(sizeof(lut)));
    UP(ctx->scratch[5].p, lut, sizeof(lut));
    d_lut = ctx->scratch[5].as<float>();
  }
  const void * dsrc; void * ddst;
  if (int r = stage_in(ctx, ctx->scratch[0], src, (size_t)n_samples * elem, mem, &dsrc)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], dst, sizeof(float2) * (size_t)n_samples, mem, &ddst)) return r;
  CK(launch_ingest_convert(ctx->stream, dsrc, fmt->container, fmt->msb_first ? 1 : 0, fmt->iq_order, inv_scaler, d_lut, n_samples, (float2 *)ddst, &ctx->launches));
  if (int r = stage_out_end(ctx, ddst, dst, sizeof(float2) * (size_t)n_samples, mem)) return r;
  ctx->arena_off = 0; // the stream is idle: staged uploads have been consumed
  return 0;
}

// ------------------------------------------------------------------------------------------------ TII detector (next row f4)
struct dabstar_tii
{
  dabstar_ctx * ctx = nullptr;
  int n = 0;
  int collisions = 0, sub_id_coll = 0;
  DevBuf null_sum, decoded, tables, results;
  DevBuf staging;
};

extern "C" int dabstar_tii_create(dabstar_ctx * ctx, int n_detectors, dabstar_tii ** out)
{
  if (!ctx || !out || n_detectors <= 0) return DABSTAR_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  std::unique_ptr<dabstar_tii> t(new dabstar_tii);
  t->ctx = ctx;
  t->n = n_detectors;
  CK(t->null_sum.reserve(sizeof(float2) * (size_t)n_detectors * T_U));
  CK(t->decoded.reserve(sizeof(float2) * (size_t)n_detectors * 768));
  CK(t->tables.reserve(70 + 768 + 16));
  // cMainIdPatternTable (tii_detector.cpp:19-90): the 70 bytes with four bits set, ascending (EN 300 401 table 42);
  // cPhaseCorrTable (:92-125): quadrant(PRS[k]) - quadrant(PRS[k + 1]) mod 4 for the carrier pair k, k + 1
  uint8_t tab[70 + 768];
  int np = 0;
  for (int b = 0; b < 256; b++) if (__builtin_popcount((unsigned)b) == 4) tab[np++] = (uint8_t)b;
  auto quadrant = [&](int f) { const float2 v = ctx->h_prs[f]; return fabsf(v.x) > fabsf(v.y) ? (v.x > 0 ? 0 : 2) : (v.y > 0 ? 1 : 3); };
  for (int i = 0; i < 768; i++)
  {
    const int k = -K_CARR / 2 + 2 * i, f = k < 0 ? k + T_U : k + 1;
    tab[70 + i] = (uint8_t)((quadrant(f) - quadrant(f + 1)) & 3);
  }
  CK(cudaMemcpyAsync(t->tables.p, tab, sizeof(tab), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(t->null_sum.p, 0, sizeof(float2) * (size_t)n_detectors * T_U, ctx->stream));
  CK(cudaMemsetAsync(t->decoded.p, 0, sizeof(float2) * (size_t)n_detectors * 768, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *out = t.release();
  return 0;
}
extern "C" void dabstar_tii_destroy(dabstar_tii * t)
{
  if (!t) return;
  if (t->ctx) cudaSetDevice(t->ctx->device);
  delete t;
}
extern "C" int dabstar_tii_reset(dabstar_tii * t)
{
  if (!t) return DABSTAR_E_INVALID;
  dabstar_ctx * ctx = t->ctx;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemsetAsync(t->null_sum.p, 0, sizeof(float2) * (size_t)t->n * T_U, ctx->stream));
  CK(cudaMemsetAsync(t->decoded.p, 0, sizeof(float2) * (size_t)t->n * 768, ctx->stream));
  return 0;
}
extern "C" int dabstar_tii_set_collisions(dabstar_tii * t, int on, int sub_id)
{
  if (!t || sub_id < 0 || sub_id > 23) return DABSTAR_E_INVALID;
  t->collisions = on ? 1 : 0;
  t->sub_id_coll = sub_id;
  return 0;
}
extern "C" int dabstar_tii_add(dabstar_tii * t, const float * fft, int n_symbols, int mem)
{
  if (!t || !fft || n_symbols < 0) return DABSTAR_E_INVALID;
  if (n_symbols == 0) return 0;
  dabstar_ctx * ctx = t->ctx;
  CK(cudaSetDevice(ctx->device));
  const void * dfft;
  if (int r = stage_in(ctx, t->staging, fft, sizeof(float2) * (size_t)t->n * n_symbols * T_U, mem, &dfft)) return r;
  CK(launch_tii_add(ctx->stream, (const float2 *)dfft, t->n, n_symbols, t->null_sum.as<float2>(), &ctx->launches));
  if (mem == DABSTAR_MEM_HOST) CK(cudaStreamSynchronize(ctx->stream)); // the caller may reuse its buffer
  return 0;
}
extern "C" int dabstar_tii_process(dabstar_tii * t, int threshold_db, dabstar_tii_result * out, int cap, int32_t * counts)
{
  if (!t || !out || !counts || cap <= 0) return DABSTAR_E_INVALID;
  dabstar_ctx * ctx = t->ctx;
  CK(cudaSetDevice(ctx->device));
  static_assert(sizeof(TiiResultDev) == sizeof(dabstar_tii_result), "result layout");
  CK(t->results.reserve(sizeof(TiiResultDev) * (size_t)t->n * cap + sizeof(int) * (size_t)t->n));
  TiiResultDev * d_res = t->results.as<TiiResultDev>();
  int * d_cnt = reinterpret_cast<int *>(d_res + (size_t)t->n * cap);
  const float factor = powf(10.0f, (float)(int16_t)threshold_db / 10.0f); // std::pow(10.0f, (f32)iThreshold_db / 10.0f), tii_detector.cpp:193
  const uint8_t * tab = t->tables.as<uint8_t>();
  CK(launch_tii_process(ctx->stream, t->n, t->null_sum.as<float2>(), t->decoded.as<float2>(), tab, tab + 70, factor, t->collisions, t->sub_id_coll, d_res, cap, d_cnt,
                        &ctx->launches));
  CK(cudaMemcpyAsync(out, d_res, sizeof(TiiResultDev) * (size_t)t->n * cap, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(counts, d_cnt, sizeof(int) * (size_t)t->n, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  // std::sort by strength, descending (tii_detector.cpp:236); the comb threads append in no particular order
  for (int d = 0; d < t->n; d++)
  {
    dabstar_tii_result * r = out + (size_t)d * cap;
    const int n = std::min(counts[d], cap);
    std::sort(r, r + n, [](const dabstar_tii_result & a, const dabstar_tii_result & b) {
      return a.strength != b.strength ? a.strength > b.strength : (a.sub_id != b.sub_id ? a.sub_id < b.sub_id : a.main_id < b.main_id);
    });
  }
  return 0;
}
extern "C" int dabstar_tii_decoded(dabstar_tii * t, int detector, float * out)
{
  if (!t || !out || detector < 0 || detector >= t->n) return DABSTAR_E_INVALID;
  dabstar_ctx * ctx = t->ctx;
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(out, t->decoded.as<float2>() + (size_t)detector * 768, sizeof(float2) * 768, cudaMemcpyDeviceToHost));
  return 0;
}

// ---- SampleReader's DC / IQ-imbalance correction (sample_reader.cpp:216-243; set_dc_and_iq_correction, sample_reader.h:66)
extern "C" int dabstar_dc_iq_correct(dabstar_ctx * ctx, const float * in, int64_t n_samples, int do_iq, dabstar_dciq_state * state, float * out, int mem)
{
  if (!ctx || !in || !out || n_samples < 0) return DABSTAR_E_INVALID;
  if (n_samples == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  dabstar_dciq_state fresh{ 0.0f, 0.0f, 1.0f, 1.0f, 0.0f }; // sample_reader.h:102-106
  dabstar_dciq_state * st = state ? state : &fresh;
  double sv[5] = { st->mean_i, st->mean_q, st->mean_ii, st->mean_iq, st->mean_qq };
  const double alpha = (double)(1.0f / (float)FS / 1.00f); // constexpr f32 ALPHA = 1.0f / INPUT_RATE / 1.00f
  const void * din; void * dout;
  const size_t bytes = sizeof(float2) * (size_t)n_samples;
  if (int r = stage_in(ctx, ctx->scratch[0], in, bytes, mem, &din)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], out, bytes, mem, &dout)) return r;
  CK(ctx->scratch[2].reserve(dciq_workspace_bytes(n_samples)));
  CK(launch_dc_iq_correct(ctx->stream, (const float2 *)din, n_samples, do_iq != 0, alpha, sv, ctx->scratch[2].p, (float2 *)dout, &ctx->launches));
  if (int r = stage_out_end(ctx, dout, out, bytes, mem)) return r;
  st->mean_i = (float)sv[0]; st->mean_q = (float)sv[1]; st->mean_ii = (float)sv[2]; st->mean_iq = (float)sv[3]; st->mean_qq = (float)sv[4];
  return 0;
}

// ---- sample-rate conversion of the file readers (xml_reader.cpp:70-76,212-231; wav_reader.cpp:66-83,196-211)
static void resample_tables(int sample_rate, int reader, short base[2048], float frac[2048], int * block_in, int * shift)
{
  if (reader == DABSTAR_READER_WAV)
  {
    // mConvBufferSize = rate / 1000; tables in float (wav_reader.cpp:66-79)
    *block_in = (int)(int16_t)(sample_rate / 1000);
    *shift = 0;
    const float in_val = (float)sample_rate / 1000.0f;
    for (int i = 0; i < 2048; i++)
    {
      base[i] = (short)floorf((float)i * (in_val / 2048.0f));
      frac[i] = (float)i * (in_val / 2048.0f) - (float)base[i];
    }
  }
  else
  {
    // convBufferSize = rate / 1000; integer part in double, fraction in float (xml_reader.cpp:70-76)
    *block_in = sample_rate / 1000;
    *shift = 1;
    const float in_val = (float)(sample_rate / 1000);
    for (int i = 0; i < 2048; i++)
    {
      base[i] = (short)floor(i * (in_val / 2048.0));
      frac[i] = i * (in_val / 2048.0f) - base[i];
    }
  }
}

extern "C" int64_t dabstar_resample_count(int64_t n_in, int sample_rate, int reader)
{
  if (n_in < 0 || sample_rate < 1000 || sample_rate > 32000000 || (reader != DABSTAR_READER_XML && reader != DABSTAR_READER_WAV)) return DABSTAR_E_INVALID;
  if (sample_rate == FS) return n_in;
  const int64_t n = sample_rate / 1000;
  // whole 1 ms blocks only: the WAV reader needs N + 1 samples for its first block and N for every further one
  const int64_t blocks = reader == DABSTAR_READER_WAV ? (n_in >= 1 ? (n_in - 1) / n : 0) : n_in / n;
  return blocks * 2048;
}

extern "C" int64_t dabstar_resample_linear(dabstar_ctx * ctx, const float * in, int64_t n_in, int sample_rate, int reader, float * out, int64_t out_cap, int mem)
{
  if (!ctx || !in || !out) return DABSTAR_E_INVALID;
  const int64_t n_out = dabstar_resample_count(n_in, sample_rate, reader);
  if (n_out < 0) return ctx->fail(DABSTAR_E_INVALID, "resample: rate %d / reader %d", sample_rate, reader);
  if (n_out > out_cap) return ctx->fail(DABSTAR_E_INVALID, "resample: %lld output samples, room for %lld", (long long)n_out, (long long)out_cap);
  if (n_out == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  if (sample_rate == FS)
  {
    CK(cudaMemcpyAsync(out, in, sizeof(float2) * (size_t)n_in, mem == DABSTAR_MEM_HOST ? cudaMemcpyHostToHost : cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return n_out;
  }
  short base[2048];
  float frac[2048];
  int block_in = 0, shift = 0;
  resample_tables(sample_rate, reader, base, frac, &block_in, &shift);
  CK(ctx->scratch[5].reserve(sizeof(base) + sizeof(frac)));
  float * d_frac = ctx->scratch[5].as<float>();
  short * d_base = reinterpret_cast<short *>(d_frac + 2048);
  CK(cudaMemcpyAsync(d_frac, frac, sizeof(frac), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_base, base, sizeof(base), cudaMemcpyHostToDevice, ctx->stream));
  const void * din; void * dout;
  if (int r = stage_in(ctx, ctx->scratch[0], in, sizeof(float2) * (size_t)n_in, mem, &din)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], out, sizeof(float2) * (size_t)n_out, mem, &dout)) return r;
  CK(launch_resample_linear(ctx->stream, (const float2 *)din, n_in, block_in, shift, d_base, d_frac, n_out, (float2 *)dout, &ctx->launches));
  if (int r = stage_out_end(ctx, dout, out, sizeof(float2) * (size_t)n_out, mem)) return r; // (synchronises: base / frac are consumed)
  return n_out;
}

// ------------------------------------------------------------------------------------------------ DAB+ outer code (next row f2)
extern "C" int dabstar_dabplus_decode(dabstar_ctx * ctx, const uint8_t * frame_bits, int bit_rate, int n_frames, dabstar_superframe * out, int cap,
                                      uint8_t * payload, int mem)
{
  if (!ctx || (!frame_bits && n_frames > 0) || n_frames < 0 || cap < 0 || (cap > 0 && !out)) return DABSTAR_E_INVALID;
  if (bit_rate < 8 || bit_rate > 192 || bit_rate % 8) return ctx->fail(DABSTAR_E_INVALID, "DAB+ bit rate %d", bit_rate);
  const int n_windows = n_frames - 4;
  if (n_windows <= 0) return 0;
  CK(cudaSetDevice(ctx->device));
  if (!ctx->d_gf.p)
  {
    std::vector<uint8_t> gf;
    std::vector<uint16_t> syn;
    dabplus_host_tables(gf, syn);
    CK(ctx->d_gf.reserve(gf.size()));
    CK(ctx->d_fc_syn.reserve(sizeof(uint16_t) * syn.size()));
    CK(cudaMemcpyAsync(ctx->d_gf.p, gf.data(), gf.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_fc_syn.p, syn.data(), sizeof(uint16_t) * syn.size(), cudaMemcpyHostToDevice, ctx->stream));
    SYNC();
  }
  const int rs_dims = bit_rate / 8, sf_bytes = 110 * rs_dims;
  const size_t n_bits = (size_t)n_frames * 24 * bit_rate;
  const void * dbits;
  if (int r = stage_in(ctx, ctx->scratch[0], frame_bits, n_bits, mem, &dbits)) return r;
  CK(ctx->scratch[1].reserve(n_bits / 8));                                   // packed frames
  CK(ctx->scratch[2].reserve((size_t)n_windows * sf_bytes));                 // decoded super-frame of every window
  CK(ctx->scratch[3].reserve((size_t)n_windows * rs_dims));                  // Reed-Solomon return codes
  CK(ctx->scratch[4].reserve(sizeof(SuperFrameRec) * (size_t)n_windows));
  CK(launch_pack_bits(ctx->stream, (const uint8_t *)dbits, ctx->scratch[1].as<uint8_t>(), (long long)(n_bits / 8), &ctx->launches));
  CK(launch_dabplus(ctx->stream, ctx->scratch[1].as<uint8_t>(), bit_rate, n_frames, ctx->d_gf.p, ctx->d_fc_syn.as<uint16_t>(), ctx->scratch[2].as<uint8_t>(),
                    ctx->scratch[3].as<int8_t>(), ctx->scratch[4].as<SuperFrameRec>(), &ctx->launches));
  std::vector<SuperFrameRec> rec((size_t)n_windows);
  CK(cudaMemcpyAsync(rec.data(), ctx->scratch[4].p, sizeof(SuperFrameRec) * rec.size(), cudaMemcpyDeviceToHost, ctx->stream));
  SYNC();
  // Mp4Processor::add_to_frame (mp4processor.cpp:95-180): which windows the processor attempts, given every window's outcome
  int in_buf = 0, sync = 0, n_out = 0;
  for (int f = 0; f < n_frames; f++)
  {
    if (++in_buf < 5) continue;
    const int w = f - 4;
    if (sync == 0)
    {
      if (rec[w].pre_ok) sync = 4;
      else { in_buf = 4; continue; }
    }
    in_buf = 0;
    if (rec[w].ok) sync = 4;
    else if (--sync == 0) in_buf = 4;
    if (n_out < cap)
    {
      const SuperFrameRec & r = rec[w];
      dabstar_superframe & o = out[n_out];
      o.first_frame = r.first_frame; o.ok = r.ok; o.rs_errors = r.rs_errors; o.rs_corrections = r.rs_corrections; o.fc_corrected = r.fc_corrected;
      o.dac_rate = r.dac_rate; o.sbr_flag = r.sbr_flag; o.aac_channel_mode = r.aac_channel_mode; o.ps_flag = r.ps_flag; o.mpeg_surround = r.mpeg_surround;
      o.num_aus = r.num_aus;
      for (int i = 0; i < 7; i++) o.au_start[i] = r.au_start[i];
      for (int i = 0; i < 6; i++) o.au_state[i] = r.au_state[i];
      if (payload)
        CK(cudaMemcpyAsync(payload + (size_t)n_out * sf_bytes, ctx->scratch[2].as<uint8_t>() + (size_t)w * sf_bytes, (size_t)sf_bytes,
                           mem == DABSTAR_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, ctx->stream));
    }
    n_out++;
  }
  SYNC();
  return n_out;
}

// ------------------------------------------------------------------------------------------------ stage taps
extern "C" int dabstar_fft2048(dabstar_ctx * ctx, const float * in, float * out, int n, int sign, int mem)
{
  if (!ctx || !in || !out || n < 0) return DABSTAR_E_INVALID;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  const size_t bytes = sizeof(float2) * T_U * (size_t)n;
  const void * din; void * dout;
  if (int r = stage_in(ctx, ctx->scratch[0], in, bytes, mem, &din)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], out, bytes, mem, &dout)) return r;
  CK(launch_fft_batch(ctx->stream, ctx->tab, (const float2 *)din, (float2 *)dout, n, sign, &ctx->launches));
  return stage_out_end(ctx, dout, out, bytes, mem);
}

// Workspace of the thread-per-code-word Viterbi: what one launch needs, capped (the launcher then works in chunks).
static int reserve_viterbi_ws(dabstar_ctx * ctx, int n_jobs, int max_steps)
{
  // 6 GiB of the 180 GB: about 125 000 of the longest MSC code words (3078 steps x 16 B) per launch, i.e. four warps per scheduler
  // (the kernel's register limit); a 1.5 GiB cap left a launch at 1.7 warps per scheduler (ncu: 33 % of the stall samples on loads)
  const size_t cap = (size_t)6 << 30;
  CK(ctx->vit_ws.reserve(std::min(viterbi_ws_bytes(n_jobs, max_steps), cap)));
  return 0;
}

static int run_viterbi_jobs(dabstar_ctx * ctx, const std::vector<VitJob> & jobs, int max_steps, const int16_t * d_soft, uint8_t * d_bits,
                            uint8_t * d_crc, int * d_ber, DevBuf & jobbuf)
{
  if (jobs.empty()) return 0;
  if (int r = sync_profiles(ctx)) return r;
  CK(jobbuf.reserve(sizeof(VitJob) * jobs.size()));
  UP(jobbuf.p, jobs.data(), sizeof(VitJob) * jobs.size());
  if (int r = reserve_viterbi_ws(ctx, (int)jobs.size(), max_steps)) return r;
  CK(launch_viterbi(ctx->stream, jobbuf.as<VitJob>(), nullptr, (int)jobs.size(), ctx->d_profiles.as<VitProfile>(), max_steps, d_soft, d_bits,
                    ctx->tab.prbs, d_crc, d_ber, ctx->d_step_tab.as<unsigned>(), ctx->vit_ws.p, ctx->vit_ws.cap, &ctx->launches));
  return 0;
}

extern "C" int dabstar_viterbi(dabstar_ctx * ctx, const int16_t * soft, const int64_t * soft_off, const int32_t * frame_bits, int n,
                               uint8_t * bits, const int64_t * bits_off, int mem)
{
  if (!ctx || !soft || !soft_off || !frame_bits || !bits || !bits_off || n < 0) return DABSTAR_E_INVALID;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  size_t soft_len = 0, bits_len = 0;
  int max_steps = 0;
  std::vector<VitJob> jobs((size_t)n);
  for (int i = 0; i < n; i++)
  {
    if (frame_bits[i] <= 0 || frame_bits[i] > 16384) return ctx->fail(DABSTAR_E_INVALID, "frame_bits[%d] = %d", i, frame_bits[i]);
    if (soft_off[i] < 0 || bits_off[i] < 0) return ctx->fail(DABSTAR_E_INVALID, "negative offset for code word %d", i);
    VitJob & j = jobs[i];
    memset(&j, 0, sizeof(j));
    j.src = soft_off[i];
    j.out = bits_off[i];
    j.profile = get_identity_profile(ctx, frame_bits[i]);
    j.src_mode = VIT_SRC_LINEAR;
    soft_len = std::max(soft_len, (size_t)soft_off[i] + 4 * (size_t)(frame_bits[i] + 6));
    bits_len = std::max(bits_len, (size_t)bits_off[i] + (size_t)frame_bits[i]);
    max_steps = std::max(max_steps, frame_bits[i] + 6);
  }
  const void * dsoft; void * dbits;
  if (int r = stage_in(ctx, ctx->scratch[0], soft, soft_len * sizeof(int16_t), mem, &dsoft)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], bits, bits_len, mem, &dbits)) return r;
  if (int r = run_viterbi_jobs(ctx, jobs, max_steps, (const int16_t *)dsoft, (uint8_t *)dbits, nullptr, nullptr, ctx->scratch[2])) return r;
  return stage_out_end(ctx, dbits, bits, bits_len, mem);
}

extern "C" int dabstar_protection_deconvolve(dabstar_ctx * ctx, int short_form, int bit_rate, int prot_level, int size_cu,
                                             const int16_t * soft, int n, uint8_t * bits, int mem)
{
  if (!ctx || !soft || !bits || n < 0 || size_cu <= 0) return DABSTAR_E_INVALID;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  const int prof = get_profile(ctx, short_form, bit_rate, prot_level);
  if (prof < 0) return ctx->fail(DABSTAR_E_INVALID, "unknown protection profile %d/%d/%d", short_form, bit_rate, prot_level);
  const VitProfile & p = ctx->profiles[prof];
  if (p.n_kept > size_cu * 64) return ctx->fail(DABSTAR_E_INVALID, "size_cu %d too small for profile (%d soft bits)", size_cu, p.n_kept);
  const void * dsoft; void * dbits;
  const size_t in_bytes = sizeof(int16_t) * (size_t)n * size_cu * 64, out_bytes = (size_t)n * p.n_bits;
  if (int r = stage_in(ctx, ctx->scratch[0], soft, in_bytes, mem, &dsoft)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], bits, out_bytes, mem, &dbits)) return r;
  // the job list is written on the device (one job per logical frame at a constant stride)
  if (int r = sync_profiles(ctx)) return r;
  CK(ctx->scratch[2].reserve(sizeof(VitJob) * (size_t)n));
  CK(launch_linear_jobs(ctx->stream, ctx->scratch[2].as<VitJob>(), n, (long long)size_cu * 64, p.n_bits, prof, &ctx->launches));
  if (int r = reserve_viterbi_ws(ctx, n, p.n_bits + 6)) return r;
  CK(launch_viterbi(ctx->stream, ctx->scratch[2].as<VitJob>(), nullptr, n, ctx->d_profiles.as<VitProfile>(), p.n_bits + 6, (const int16_t *)dsoft, (uint8_t *)dbits,
                    ctx->tab.prbs, nullptr, nullptr, ctx->d_step_tab.as<unsigned>(), ctx->vit_ws.p, ctx->vit_ws.cap, &ctx->launches));
  return stage_out_end(ctx, dbits, bits, out_bytes, mem);
}

static void make_fic_jobs(std::vector<VitJob> & jobs, long long soft_base, long long out_base, int aux_base, int n_fic)
{
  for (int b = 0; b < n_fic; b++)
  {
    VitJob j;
    memset(&j, 0, sizeof(j));
    j.src = soft_base + (long long)b * FIC_IN;
    j.out = out_base + (long long)b * FIC_OUT;
    j.profile = 0;
    j.src_mode = VIT_SRC_LINEAR;
    j.flags = VIT_FLAG_PRBS | VIT_FLAG_FIC;
    j.aux = aux_base + b;
    jobs.push_back(j);
  }
}

extern "C" int dabstar_fic_decode(dabstar_ctx * ctx, const int16_t * soft, int64_t frame_stride, int n, uint8_t * fib_bits,
                                  uint8_t * crc_ok, int32_t * ber, int mem)
{
  if (!ctx || !soft || !fib_bits || !crc_ok || !ber || n < 0 || frame_stride < FIC_SOFT) return DABSTAR_E_INVALID;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  std::vector<VitJob> jobs;
  jobs.reserve((size_t)4 * n);
  for (int f = 0; f < n; f++) make_fic_jobs(jobs, (long long)f * frame_stride, (long long)f * 4 * FIC_OUT, 4 * f, 4);
  const void * dsoft; void * dbits; void * dcrc; void * dber;
  const size_t in_bytes = sizeof(int16_t) * ((size_t)(n - 1) * frame_stride + FIC_SOFT);
  if (int r = stage_in(ctx, ctx->scratch[0], soft, in_bytes, mem, &dsoft)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], fib_bits, (size_t)n * 3072, mem, &dbits)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[3], crc_ok, (size_t)n * 12, mem, &dcrc)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[4], ber, sizeof(int32_t) * (size_t)n * 8, mem, &dber)) return r;
  if (int r = run_viterbi_jobs(ctx, jobs, FIC_OUT + 6, (const int16_t *)dsoft, (uint8_t *)dbits, (uint8_t *)dcrc, (int *)dber, ctx->scratch[2])) return r;
  if (mem == DABSTAR_MEM_HOST)
  {
    CK(cudaMemcpyAsync(crc_ok, dcrc, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ber, dber, sizeof(int32_t) * (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  }
  return stage_out_end(ctx, dbits, fib_bits, (size_t)n * 3072, mem);
}

// Jobs of one Backend over CIFs [g_begin, g_end) of a recording whose frame slot 0 starts at int16 index `rec_base`.
// g_start = first CIF the Backend saw. Emission starts with its 17th CIF (backend/backend.cpp:146-150).
static void make_backend_jobs(std::vector<VitJob> & jobs, int prof, const VitProfile & p, long long rec_base, int g_start, int g_begin, int g_end,
                              int start_cu, long long out_base)
{
  long long out = out_base;
  for (int g = std::max(g_begin, g_start + 16); g < g_end; g++)
  {
    VitJob j;
    memset(&j, 0, sizeof(j));
    j.src = rec_base;
    j.out = out;
    j.profile = prof;
    j.src_mode = VIT_SRC_TIME_DEINTERLEAVE;
    j.flags = VIT_FLAG_PRBS;
    j.cif_first = g - 16;
    const int lo = std::max(0, g_start - (g - 16)); // rows m with g - 16 + m >= g_start hold CIFs the Backend has seen
    j.row_mask = lo >= 16 ? 0 : ((0xFFFF << lo) & 0xFFFF);
    j.frag_off = start_cu * 64;
    jobs.push_back(j);
    out += p.n_bits;
  }
}

extern "C" int dabstar_backend_process(dabstar_ctx * ctx, const dabstar_subch * sc, const int16_t * cifs, int n_cifs, uint8_t * bits, int mem)
{
  if (!ctx || !sc || !cifs || !bits || n_cifs < 0) return DABSTAR_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  const int prof = get_profile(ctx, sc->short_form, sc->bit_rate, sc->prot_level);
  if (prof < 0) return ctx->fail(DABSTAR_E_INVALID, "unknown protection profile %d/%d/%d", sc->short_form, sc->bit_rate, sc->prot_level);
  const VitProfile p = ctx->profiles[prof];
  if (sc->start_cu < 0 || sc->size_cu <= 0 || sc->start_cu + sc->size_cu > 864 || p.n_kept > sc->size_cu * 64)
    return ctx->fail(DABSTAR_E_INVALID, "sub-channel geometry %d+%d does not fit", sc->start_cu, sc->size_cu);
  const int n_out = std::max(0, n_cifs - 16);
  if (n_out == 0) return 0;
  // The tap takes plain CIFs; the kernel addresses CIFs inside frame slots, so lay them out as slots (FIC part unused).
  const int n_slots = (n_cifs + 3) / 4;
  CK(ctx->scratch[0].reserve(sizeof(int16_t) * (size_t)n_slots * FRAME_SOFT));
  int16_t * dsoft = ctx->scratch[0].as<int16_t>();
  for (int g = 0; g < n_cifs; g++)
    CK(cudaMemcpyAsync(dsoft + cif_offset(g), cifs + (size_t)g * CIF_BITS, sizeof(int16_t) * CIF_BITS,
                       mem == DABSTAR_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, ctx->stream));
  std::vector<VitJob> jobs;
  make_backend_jobs(jobs, prof, p, 0, 0, 0, n_cifs, sc->start_cu, 0);
  void * dbits;
  const size_t out_bytes = (size_t)n_out * p.n_bits;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], bits, out_bytes, mem, &dbits)) return r;
  if (int r = run_viterbi_jobs(ctx, jobs, p.n_bits + 6, dsoft, (uint8_t *)dbits, nullptr, nullptr, ctx->scratch[2])) return r;
  if (int r = stage_out_end(ctx, dbits, bits, out_bytes, mem)) return r;
  return n_out;
}

struct dabstar_ofdm_state
{
  OfdmStateDev * dev = nullptr;
};

static int ofdm_state_init(dabstar_ctx * ctx, OfdmStateDev * dev, bool full, int count = 1)
{
  k_ofdm_state_init<<<std::min(count * 8, 1024), 256, 0, ctx->stream>>>(dev, count, full ? 1 : 0);
  ctx->launches++;
  CK(cudaGetLastError());
  return 0;
}

extern "C" int dabstar_ofdm_state_create(dabstar_ctx * ctx, dabstar_ofdm_state ** out)
{
  if (!ctx || !out) return DABSTAR_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  std::unique_ptr<dabstar_ofdm_state> st(new dabstar_ofdm_state);
  CK(cudaMalloc(&st->dev, sizeof(OfdmStateDev)));
  if (int r = ofdm_state_init(ctx, st->dev, true)) { cudaFree(st->dev); return r; }
  *out = st.release();
  return 0;
}
extern "C" void dabstar_ofdm_state_destroy(dabstar_ctx * ctx, dabstar_ofdm_state * st)
{
  if (!st) return;
  if (ctx) cudaSetDevice(ctx->device);
  cudaFree(st->dev);
  delete st;
}
extern "C" int dabstar_ofdm_state_reset(dabstar_ctx * ctx, dabstar_ofdm_state * st)
{
  if (!ctx || !st) return DABSTAR_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  return ofdm_state_init(ctx, st->dev, false);
}
// The figures OfdmDecoder hands to signal_show_lcd_data (ofdm_decoder.cpp:326-345, _compute_noise_Power :357-371):
// out = { MER dB, SNR dB, mMeanValue, mMeanPowerOvrAll, noise power, sqrt(mMeanSigmaSqFreqCorr) }, from the sums of a state
// (quality_from_state, or k_frame_quality per frame in the same order and precision).
static void quality_from_sums(const FrameQual & q, float sigma_sq_freq_corr, float out[6])
{
  float sum_noise = q.sum_null_pow, sd = q.sum_stddev;
  if (sum_noise == 0.0f) sum_noise = (1.0f / 32767.0f) * (1.0f / 32767.0f) * (float)K_CARR;
  const float noise = sum_noise / (float)K_CARR;
  float snr = (q.mean_pow_all - noise) / noise;
  if (snr <= 0.0f) snr = 0.1f;
  sd /= (float)K_CARR;
  const float pi_4 = 0.78539816339744830962f;
  out[0] = 10.0f * log10f(pi_4 * pi_4 / sd);
  out[1] = 10.0f * log10f(snr);
  out[2] = q.mean_value;
  out[3] = q.mean_pow_all;
  out[4] = noise;
  out[5] = sqrtf(sigma_sq_freq_corr);
}
// ... from a recording's state
static int quality_from_state(dabstar_ctx * ctx, const OfdmStateDev * dev, float sigma_sq_freq_corr, float out[6])
{
  CK(cudaStreamSynchronize(ctx->stream));
  std::unique_ptr<OfdmStateDev> h(new OfdmStateDev);
  CK(cudaMemcpy(h.get(), dev, sizeof(OfdmStateDev), cudaMemcpyDeviceToHost));
  // mMeanPowerOvrAll = A^G y0 + b sum_k (1-b)^(1535-k) c_k (kernels.h, OfdmStateDev)
  double acc = 0.0, w = 1.0;
  for (int k = K_CARR - 1; k >= 0; k--) { acc += w * (double)h->pow_acc[k]; w *= 1.0 - POW_ALL_BETA; }
  const float mean_pow_all = (float)((double)h->pow_carry + POW_ALL_BETA * acc);
  float sum_noise = 0.0f, sd = 0.0f;
  for (int k = 0; k < K_CARR; k++) { sum_noise += h->null_pow[k]; sd += h->stddev[k]; }
  quality_from_sums(FrameQual{ sd, sum_noise, mean_pow_all, h->mean_value }, sigma_sq_freq_corr, out);
  return 0;
}

extern "C" int dabstar_ofdm_state_get(dabstar_ctx * ctx, dabstar_ofdm_state * st, int which, float * out)
{
  if (!ctx || !st || !out || which < 0 || which > 5) return DABSTAR_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  OfdmStateDev * d = st->dev;
  if (which == 5)
  {
    float q[6];
    if (int r = quality_from_state(ctx, d, 0.0f, q)) return r;
    out[0] = q[2]; out[1] = q[3];
    return 0;
  }
  const float * src[5] = { d->integ, d->stddev, d->mean_pow, d->mean_sigma, d->null_pow };
  CK(cudaMemcpy(out, src[which], sizeof(float) * K_CARR, cudaMemcpyDeviceToHost));
  return 0;
}
extern "C" int dabstar_ofdm_state_quality(dabstar_ctx * ctx, dabstar_ofdm_state * st, float out[6])
{
  if (!ctx || !st || !out) return DABSTAR_E_INVALID;
  CK(cudaSetDevice(ctx->device));
  return quality_from_state(ctx, st->dev, 0.0f, out);
}

static int ofdm_decode_frames(dabstar_ctx * ctx, dabstar_ofdm_state * st, const float * fft, int n_frames, const float * clock_err,
                              const uint8_t * null_is_tii, int soft_bit_type, int16_t * soft, int mem, float * quality)
{
  if (!ctx || !st || !fft || !soft || n_frames < 0 || soft_bit_type < 0 || soft_bit_type > 2) return DABSTAR_E_INVALID;
  if (n_frames == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  const size_t in_bytes = sizeof(float2) * (size_t)n_frames * X_ROWS * T_U, out_bytes = sizeof(int16_t) * (size_t)n_frames * FRAME_SOFT;
  const void * dfft; void * dsoft;
  if (int r = stage_in(ctx, ctx->scratch[0], fft, in_bytes, mem, &dfft)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], soft, out_bytes, mem, &dsoft)) return r;
  CK(ctx->scratch[2].reserve(sizeof(float2) * (size_t)n_frames * X_ROWS * K_CARR));
  CK(launch_reorder_frames(ctx->stream, ctx->tab, (const float2 *)dfft, n_frames, ctx->scratch[2].as<float2>(), &ctx->launches));
  std::vector<FrameDesc> fd((size_t)n_frames);
  std::vector<uint8_t> tii((size_t)n_frames, 0);
  for (int f = 0; f < n_frames; f++)
  {
    memset(&fd[f], 0, sizeof(FrameDesc));
    fd[f].slot = f;
    fd[f].xslot = f;
    fd[f].clock_err = clock_err ? clock_err[f] : 0.0f;
    fd[f].n_syms = 75;
    if (null_is_tii) tii[f] = null_is_tii[f];
  }
  DemapWork wk{ 0, n_frames, 0, 0, 0, 0 };
  // with quality: aux also holds the per-frame sums behind the descriptors (16-byte aligned), the snapshots go to scratch[4]
  const size_t fq_off = (sizeof(FrameDesc) * fd.size() + sizeof(DemapWork) + tii.size() + 15) & ~(size_t)15;
  CK(ctx->scratch[3].reserve(fq_off + (quality ? sizeof(FrameQual) * fd.size() : 0) + 64));
  FrameQualSnap * dsnap = nullptr;
  if (quality)
  {
    CK(ctx->scratch[4].reserve(sizeof(FrameQualSnap) * fd.size()));
    dsnap = ctx->scratch[4].as<FrameQualSnap>();
  }
  char * aux = ctx->scratch[3].as<char>();
  FrameDesc * dfd = reinterpret_cast<FrameDesc *>(aux);
  DemapWork * dwk = reinterpret_cast<DemapWork *>(aux + sizeof(FrameDesc) * fd.size());
  uint8_t * dtii = reinterpret_cast<uint8_t *>(dwk + 1);
  UP(dfd, fd.data(), sizeof(FrameDesc) * fd.size());
  UP(dwk, &wk, sizeof(wk));
  UP(dtii, tii.data(), tii.size());
  // X rows of slot f live at f*77 rows; soft slot f at f*FRAME_SOFT: both match the tap's layout.
  CK(ctx->demap_ring.reserve(demap_ring_bytes(1)));
  CK(launch_demap(ctx->stream, ctx->tab, dwk, 1, dfd, dtii, ctx->scratch[2].as<float2>(), st->dev, soft_bit_type, (int16_t *)dsoft,
                  ctx->demap_ring.as<unsigned long long>(), dsnap, &ctx->launches));
  if (quality)
  {
    FrameQual * dfq = reinterpret_cast<FrameQual *>(aux + fq_off);
    CK(launch_frame_quality(ctx->stream, dfd, n_frames, dsnap, dfq, &ctx->launches));
    std::vector<FrameQual> fq((size_t)n_frames);
    CK(cudaMemcpyAsync(fq.data(), dfq, sizeof(FrameQual) * fq.size(), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int f = 0; f < n_frames; f++) quality_from_sums(fq[(size_t)f], 0.0f, quality + 6 * (size_t)f);
  }
  return stage_out_end(ctx, dsoft, soft, out_bytes, mem);
}
extern "C" int dabstar_ofdm_decode_frames(dabstar_ctx * ctx, dabstar_ofdm_state * st, const float * fft, int n_frames, const float * clock_err,
                                          const uint8_t * null_is_tii, int soft_bit_type, int16_t * soft, int mem)
{
  return ofdm_decode_frames(ctx, st, fft, n_frames, clock_err, null_is_tii, soft_bit_type, soft, mem, nullptr);
}
extern "C" int dabstar_ofdm_decode_frames_quality(dabstar_ctx * ctx, dabstar_ofdm_state * st, const float * fft, int n_frames, const float * clock_err,
                                                  const uint8_t * null_is_tii, int soft_bit_type, int16_t * soft, int mem, float * quality)
{
  if (!quality) return DABSTAR_E_INVALID;
  return ofdm_decode_frames(ctx, st, fft, n_frames, clock_err, null_is_tii, soft_bit_type, soft, mem, quality);
}

extern "C" int dabstar_prs_correlate(dabstar_ctx * ctx, const float * samples, int n, float threshold, int strongest_peak, int32_t * start_index, int mem)
{
  if (!ctx || !samples || !start_index || n < 0) return DABSTAR_E_INVALID;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  const void * din; void * dout;
  if (int r = stage_in(ctx, ctx->scratch[0], samples, sizeof(float2) * T_U * (size_t)n, mem, &din)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], start_index, sizeof(int32_t) * (size_t)n, mem, &dout)) return r;
  CK(launch_prs_corr_raw(ctx->stream, ctx->tab, (const float2 *)din, n, threshold, strongest_peak, (int *)dout, &ctx->launches));
  return stage_out_end(ctx, dout, start_index, sizeof(int32_t) * (size_t)n, mem);
}

extern "C" int dabstar_estimate_carrier_offset(dabstar_ctx * ctx, const float * fft, int n, int32_t * offset_hz, int mem)
{
  if (!ctx || !fft || !offset_hz || n < 0) return DABSTAR_E_INVALID;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  const void * din; void * dout;
  if (int r = stage_in(ctx, ctx->scratch[0], fft, sizeof(float2) * T_U * (size_t)n, mem, &din)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], offset_hz, sizeof(int32_t) * (size_t)n, mem, &dout)) return r;
  CK(launch_coarse_afc_raw(ctx->stream, ctx->tab, (const float2 *)din, n, (int *)dout, &ctx->launches));
  return stage_out_end(ctx, dout, offset_hz, sizeof(int32_t) * (size_t)n, mem);
}

// Stage tap of the cyclic-prefix correlation (main/dab_processor.cpp:317-333,366): samples = n frames x (75 x T_s) complex floats, the
// data symbols 1..75 of each frame WITH their cyclic prefixes, as DabProcessor reads them; out[f] = sum over the 75 symbols and
// the 504 prefix samples of x[i + T_u] conj(x[i]) (re, im): the value whose argument becomes the fine frequency correction.
extern "C" int dabstar_cp_correlate(dabstar_ctx * ctx, const float * samples, int n, float * out, int mem)
{
  if (!ctx || !samples || !out || n < 0) return DABSTAR_E_INVALID;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  const long long per = 75LL * T_S;
  const void * din; void * dout;
  if (int r = stage_in(ctx, ctx->scratch[0], samples, sizeof(float2) * (size_t)per * n, mem, &din)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], out, sizeof(float2) * (size_t)n, mem, &dout)) return r;
  std::vector<FrameDesc> fd((size_t)n);
  for (int f = 0; f < n; f++)
  {
    memset(&fd[f], 0, sizeof(FrameDesc));
    fd[f].sym0 = (long long)f * per - T_U; // the kernel's symbol 1 starts T_u after sym0
    fd[f].n_syms = 75;
  }
  const RecInput rin{ din, per * n };
  CK(ctx->scratch[3].reserve(sizeof(FrameDesc) * fd.size() + sizeof(RecInput) + 64));
  FrameDesc * dfd = ctx->scratch[3].as<FrameDesc>();
  RecInput * drin = reinterpret_cast<RecInput *>(dfd + fd.size());
  UP(dfd, fd.data(), sizeof(FrameDesc) * fd.size());
  UP(drin, &rin, sizeof(rin));
  CK(launch_cp_corr(ctx->stream, dfd, n, drin, FMT_CF32, (float2 *)dout, &ctx->launches));
  return stage_out_end(ctx, dout, out, sizeof(float2) * (size_t)n, mem);
}

// Stage tap of k_fft_frames (and k_fft_null) over caller-made frame descriptors: the recordings lie end to end in one buffer, so
// their base addresses take every alignment a caller's device buffer can have. Every argument is checked before anything is
// queued: an xslot out of range would be a store outside X.
extern "C" int dabstar_fft_frames(dabstar_ctx * ctx, const void * samples, int fmt, const int64_t * rec_samples, int n_recs,
                                  const dabstar_fft_frame * frames, int n_frames, int n_xslots, int max_ctas_per_sm, float * X,
                                  float * null_fft, int mem)
{
  if (!ctx || !samples || !X || n_recs < 0 || n_frames < 0 || n_xslots < 0 || max_ctas_per_sm < 0) return DABSTAR_E_INVALID;
  if ((n_recs > 0 && !rec_samples) || (n_frames > 0 && !frames)) return DABSTAR_E_INVALID;
  if (fmt != FMT_CF32 && fmt != FMT_U8 && fmt != FMT_I16) return ctx->fail(DABSTAR_E_INVALID, "unknown sample format %d", fmt);
  const size_t elem = fmt == FMT_CF32 ? sizeof(float2) : (fmt == FMT_I16 ? 2 * sizeof(int16_t) : 2 * sizeof(uint8_t));
  long long total = 0;
  for (int r = 0; r < n_recs; r++)
  {
    if (rec_samples[r] < 0) return ctx->fail(DABSTAR_E_INVALID, "recording %d: %lld samples", r, (long long)rec_samples[r]);
    total += rec_samples[r];
  }
  std::vector<FrameDesc> fd((size_t)n_frames);
  for (int f = 0; f < n_frames; f++)
  {
    const dabstar_fft_frame & s = frames[f];
    if (s.rec < 0 || s.rec >= n_recs) return ctx->fail(DABSTAR_E_INVALID, "frame %d: recording %d of %d", f, s.rec, n_recs);
    if (s.xslot < 0 || s.xslot >= n_xslots) return ctx->fail(DABSTAR_E_INVALID, "frame %d: X slot %d of %d", f, s.xslot, n_xslots);
    if (s.n_syms < 0 || s.n_syms > 75) return ctx->fail(DABSTAR_E_INVALID, "frame %d: n_syms %d", f, s.n_syms);
    for (int hz : { s.f_sym0, s.f_data, s.f_null })
      if (hz <= -FS || hz >= FS) return ctx->fail(DABSTAR_E_INVALID, "frame %d: %d Hz", f, hz); // (keeps the kernel's 32-bit phase products in range)
    memset(&fd[f], 0, sizeof(FrameDesc));
    fd[f].sym0 = s.sym0;
    fd[f].eval = s.eval;
    fd[f].rec = s.rec;
    fd[f].slot = f;
    fd[f].xslot = s.xslot;
    fd[f].f_sym0 = s.f_sym0; fd[f].ph_eval = s.ph_eval;
    fd[f].f_data = s.f_data; fd[f].ph_data = s.ph_data;
    fd[f].f_null = s.f_null; fd[f].ph_null = s.ph_null;
    fd[f].n_syms = s.n_syms;
  }
  CK(cudaSetDevice(ctx->device));
  const size_t x_bytes = sizeof(float2) * (size_t)n_xslots * X_ROWS * K_CARR, null_bytes = sizeof(float2) * (size_t)n_frames * T_U;
  const void * din = samples; void * dX; void * dnull = nullptr;
  if (total > 0)
    if (int r = stage_in(ctx, ctx->scratch[0], samples, elem * (size_t)total, mem, &din)) return r;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], X, x_bytes, mem, &dX)) return r;
  if (null_fft && n_frames > 0)
    if (int r = stage_out_begin(ctx, ctx->scratch[4], null_fft, null_bytes, mem, &dnull)) return r;
  std::vector<RecInput> rin((size_t)n_recs);
  long long off = 0;
  for (int r = 0; r < n_recs; off += rec_samples[r], r++) rin[r] = RecInput{ static_cast<const unsigned char *>(din) + elem * (size_t)off, rec_samples[r] };
  CK(cudaMemsetAsync(dX, 0xFF, x_bytes, ctx->stream));
  if (n_frames > 0)
  {
    CK(ctx->scratch[3].reserve(sizeof(FrameDesc) * fd.size() + sizeof(RecInput) * rin.size() + 64));
    FrameDesc * dfd = ctx->scratch[3].as<FrameDesc>();
    RecInput * drin = reinterpret_cast<RecInput *>(dfd + fd.size());
    UP(dfd, fd.data(), sizeof(FrameDesc) * fd.size());
    UP(drin, rin.data(), sizeof(RecInput) * rin.size());
    CK(launch_fft_frames(ctx->stream, ctx->tab, dfd, n_frames, drin, fmt, (float2 *)dX, max_ctas_per_sm, &ctx->launches));
    if (dnull)
    {
      CK(launch_fft_null(ctx->stream, ctx->tab, dfd, n_frames, drin, fmt, (float2 *)dnull, &ctx->launches));
      if (mem == DABSTAR_MEM_HOST) CK(cudaMemcpyAsync(null_fft, dnull, null_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
  }
  return stage_out_end(ctx, dX, X, x_bytes, mem);
}

// ------------------------------------------------------------------------------------------------ whole path
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

struct Recording
{
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
  std::vector<MscOut> msc;
  bool eti_on = false;       // EtiGenerator running from the first frame of the run (DabProcessor::start_eti_generator)
  int eti_cif_hi = 0, eti_cif_lo = 0; // IFibDecoder::get_cif_count(hi, lo) as the generator samples it at symbol 4
  std::vector<uint8_t> eti;  // ETI-NI frames of the last run, 6144 bytes each
  // TII (dab_processor.cpp:273-300): needs auto_cfg, because which null symbols carry TII follows from the CIF counter
  struct TiiCfg { bool on = false; int frames_to_count = 5, threshold_db = 8, collisions = 0, sub_id = 0; } tii;
  struct TiiEvent { int frame; std::vector<dabstar_tii_result> res; int total; };
  std::vector<TiiEvent> tii_events;  // one per process_tii_data call of the last run
  std::vector<FrameDesc> descs;      // descriptors of the accepted frames (the TII pass transforms their null symbols again)
  std::vector<int> sync_frames;      // n_slots at every successful time sync (mTiiDetector.reset(), dab_processor.cpp:150-152)
  bool auto_cfg = false;     // sub-channels and CIF counter from the recording's own FIG 0/0 and 0/1
  bool tii_nulls = false;    // auto_cfg level 2: null symbols whose CIF counter has (count & 7) >= 4 do not update the null power
  std::vector<uint8_t> tii_flags; // ... per frame, as known from the previous pass over this recording (see dabstar_decoder_run)
  std::vector<int> cif_hi_f, cif_lo_f; // auto_cfg: CIF counter as the FIB decoder holds it after each frame's FIC (-1: none yet)
  dabstar_ensemble_info ens{};
  long long cnt_good_fibs = 0, cnt_sync_ok = 0, cnt_sync_fail = 0, cnt_windows = 0, cnt_cut = 0, cnt_heavy = 0, cnt_warmup = 0;
  // window scratch
  int w_first_desc = 0, w_frames = 0;
  bool w_careful = false;
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
    long long stream_pos = 0, abs_frames = 0, lead = 0;
    int rec_state = 0, osc_phase = 0, fic_ratio = 0, first_after_sync = 1, known_start = -2, spec_ok = 0, careful_spec = 1, last_start = -1, ofdm_reset = 1;
    float f_sync = 0, f_bb = 0, clock_err = 0, phase_cp = 0;
    int hist = 0;
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
  std::vector<int16_t> h_soft_one;
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

static inline int mod_fs_host(long long x)
{
  long long r = x % FS;
  return (int)(r < 0 ? r + FS : r);
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
  r.msc.clear();
  for (int i = 0; i < n; i++)
  {
    MscOut m;
    m.sc = sc[i];
    m.profile = get_profile(ctx, sc[i].short_form, sc[i].bit_rate, sc[i].prot_level);
    if (m.profile < 0) return ctx->fail(DABSTAR_E_INVALID, "unknown protection profile %d/%d/%d", sc[i].short_form, sc[i].bit_rate, sc[i].prot_level);
    const VitProfile & p = ctx->profiles[m.profile];
    if (sc[i].start_cu < 0 || sc[i].size_cu <= 0 || sc[i].start_cu + sc[i].size_cu > 864 || p.n_kept > sc[i].size_cu * 64 || sc[i].start_frame < 0)
      return ctx->fail(DABSTAR_E_INVALID, "sub-channel %d geometry does not fit", sc[i].sub_ch_id);
    r.msc.push_back(m);
  }
  return 0;
}

extern "C" int dabstar_decoder_set_auto_config(dabstar_decoder * dec, int recording, int enable)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  dec->recs[recording].auto_cfg = enable != 0;
  dec->recs[recording].tii_nulls = enable == 2;
  return 0;
}
extern "C" int dabstar_decoder_subchannels(const dabstar_decoder * dec, int recording, dabstar_subch * out, int cap)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size() || (!out && cap > 0)) return DABSTAR_E_INVALID;
  const std::vector<MscOut> & m = dec->recs[recording].msc;
  for (int i = 0; i < (int)m.size() && i < cap; i++) out[i] = m[i].sc;
  return (int)m.size();
}
extern "C" int dabstar_decoder_ensemble(const dabstar_decoder * dec, int recording, dabstar_ensemble_info * out)
{
  if (!dec || !out || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  *out = dec->recs[recording].ens;
  return 0;
}
extern "C" int dabstar_decoder_enable_eti(dabstar_decoder * dec, int recording, int enable, int cif_count_hi, int cif_count_lo)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  if (enable && (cif_count_hi < 0 || cif_count_lo < 0)) return dec->ctx->fail(DABSTAR_E_INVALID, "negative CIF count"); // the generator waits for a valid count (eti_generator.cpp:158-162)
  Recording & r = dec->recs[recording];
  r.eti_on = enable != 0;
  r.eti_cif_hi = cif_count_hi;
  r.eti_cif_lo = cif_count_lo;
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

static int decoder_run_pass(dabstar_decoder * dec, const void * const * iq, const int64_t * n_samples, int mem)
{
  if (!dec || !iq || !n_samples) return DABSTAR_E_INVALID;
  dabstar_ctx * ctx = dec->ctx;
  CK(cudaSetDevice(ctx->device));
  const int n_rec = (int)dec->recs.size();
  const int fmt = dec->cfg.input_format;
  const size_t bps = fmt == FMT_U8 ? 2 : (fmt == FMT_I16 ? 4 : 8);
  cudaStream_t st = ctx->stream;
  dec->spans.clear();
  dec->heavy_spans.clear();
  dec->fft_demap_spans.clear();
  dec->heavy_ms = dec->fft_demap_ms = 0;
  dec->ev_used = 0;
  for (int i = 0; i < 10; i++) { dec->stage_ms[i] = 0; dec->stage_launches[i] = 0; }
  CK(cudaEventRecord(dec->ev0, st));
  ctx->host_pool().prewake(); // the first region of the run is less than a wake-up away

  static const bool trace = getenv("DABSTAR_TRACE") != nullptr; // per-round progress on stderr (debug aid)
  const auto t_run0 = std::chrono::steady_clock::now();
  auto tr = [&](const char * what) {
    if (trace) fprintf(stderr, "[dabstar]   %-28s t=%.3f ms\n", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_run0).count());
  };
  // ---- inputs
  // Host input is uploaded in time-ordered chunks on the copy stream; the decode stream waits for the chunk a kernel
  // reads (need_upto), and windows are sized to what has arrived, so the PCIe transfer overlaps the decode.
  std::vector<RecInput> rin((size_t)n_rec);
  const bool host_in = mem == DABSTAR_MEM_HOST;
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
  // the decode stream must not read samples at or beyond `upto` before their chunk has landed
  auto need_upto = [&](long long upto) -> cudaError_t {
    if (!host_in) return cudaSuccess;
    int c = (int)std::min<long long>(dec->n_chunks - 1, std::max<long long>(0, (upto - 1) / dec->chunk_samples));
    if (c <= dec->chunks_waited) return cudaSuccess;
    dec->chunks_waited = c;
    return cudaStreamWaitEvent(st, dec->chunk_ev[c], 0);
  };
  // samples known to be resident (polled, never blocks)
  auto resident_upto = [&]() -> long long {
    if (!host_in) return (long long)1 << 62;
    while (dec->chunks_done < dec->n_chunks && cudaEventQuery(dec->chunk_ev[dec->chunks_done]) == cudaSuccess) dec->chunks_done++;
    (void)cudaGetLastError(); // cudaErrorNotReady from the poll is not an error
    if (dec->chunks_done >= dec->n_chunks) return (long long)1 << 62;
    return (long long)dec->chunks_done * dec->chunk_samples;
  };
  CK(dec->d_recs.reserve(sizeof(RecInput) * (size_t)n_rec));
  UP(dec->d_recs.p, rin.data(), sizeof(RecInput) * (size_t)n_rec);
  const RecInput * d_rin = dec->d_recs.as<RecInput>();

  // ---- per-recording reset (DabProcessor::run prologue, dab_processor.cpp:110-142), or continuation of a stream
  dec->total_slots = 0;
  for (int r = 0; r < n_rec; r++)
  {
    Recording & R = dec->recs[r];
    std::vector<MscOut> keep = std::move(R.msc);
    const bool eti_on = R.eti_on, auto_cfg = R.auto_cfg;
    const int eti_hi = R.eti_cif_hi, eti_lo = R.eti_cif_lo;
    const Recording::TiiCfg tii_cfg = R.tii;
    const bool tii_nulls = R.tii_nulls;
    std::vector<uint8_t> tii_flags = std::move(R.tii_flags);
    R = Recording();
    R.tii = tii_cfg;
    R.tii_nulls = tii_nulls;
    R.tii_flags = std::move(tii_flags);
    R.auto_cfg = auto_cfg;
    if (auto_cfg) keep.clear(); // rediscovered from this run's FIC
    R.msc = std::move(keep);
    R.eti_on = eti_on;
    R.eti_cif_hi = eti_hi;
    R.eti_cif_lo = eti_lo;
    for (auto & m : R.msc) { m.out_off = 0; m.out_len = 0; }
    R.d_iq = rin[r].iq;
    R.n = rin[r].n;
    const dabstar_decoder::Resume & rs = dec->resume[r];
    if (rs.on)
    {
      if (eti_on || auto_cfg || tii_cfg.on) return ctx->fail(DABSTAR_E_UNSUPPORTED, "stream continuation with ETI / self-configuration / TII is not supported");
      if (rs.lead > R.n) return ctx->fail(DABSTAR_E_INVALID, "recording %d: %lld lead samples, %lld samples given", r, rs.lead, R.n);
      R.hist = rs.hist;
      R.abs_frames = rs.abs_frames;
      R.abs_pos0 = rs.stream_pos - rs.lead;
      R.pos = rs.lead;
      R.osc_phase = rs.osc_phase; R.f_sync = rs.f_sync; R.f_bb = rs.f_bb; R.clock_err = rs.clock_err; R.phase_cp = rs.phase_cp; R.fic_ratio = rs.fic_ratio;
      R.first_after_sync = rs.first_after_sync != 0; R.known_start = rs.known_start; R.spec_ok = rs.spec_ok != 0; R.careful_spec = rs.careful_spec != 0;
      R.last_start = rs.last_start; R.ofdm_reset = rs.ofdm_reset != 0;
      R.state = rs.rec_state == 1 ? RecState::WAIT_SYNC : RecState::EVAL;
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

  tr("setup done");
  const float thr0 = dec->cfg.sync_threshold;
  // X budget: bound the frames of one round so the window spectrum buffer stays below ~12 GB
  const long long x_frame_bytes = (long long)sizeof(float2) * X_ROWS * K_CARR;
  const long long max_round_frames = std::max<long long>(n_rec, (12LL << 30) / x_frame_bytes);

  std::vector<FrameCtl> ctl;
  std::vector<CtlSnapshot> snaps((size_t)n_rec);
  std::vector<int> win_recs;

  while (true)
  {
    // ================= time sync for recordings without frame lock
    {
      std::vector<DipWork> dw;
      std::vector<int> who;
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
        who.push_back(r);
      }
      if (!dw.empty())
      {
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
        for (size_t i = 0; i < who.size(); i++)
        {
          Recording & R = dec->recs[who[i]];
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
      }
    }

    // ================= lay out this round's windows
    ctl.clear();
    win_recs.clear();
    long long budget = max_round_frames;
    bool any_wait = false;
    for (int r = 0; r < n_rec; r++)
    {
      Recording & R = dec->recs[r];
      if (R.state == RecState::WAIT_SYNC) { any_wait = true; continue; }
      if (R.state != RecState::EVAL) continue;
      if (R.pos + T_U > R.n) { R.state = RecState::DONE; R.held = dec->streaming; R.held_state = 0; continue; } // the eval read hits the end of the data
      R.w_careful = (R.fic_ratio * 10 < 30) || (R.known_start == -2 && !R.spec_ok);
      R.w_first_desc = (int)ctl.size();
      R.w_frames = 0;
      snaps[r] = take(R);
      win_recs.push_back(r);
    }
    if (win_recs.empty()) { if (any_wait) continue; break; }
    tr("  windows opened");

    // ---- step A: measure the PRS peak of the first frame where it is not known and not speculated
    {
      std::vector<FrameDesc> fd;
      std::vector<uint8_t> first;
      std::vector<int> who;
      for (int r : win_recs)
      {
        Recording & R = dec->recs[r];
        if (!(R.w_careful && R.known_start == -2)) continue;
        FrameDesc d;
        memset(&d, 0, sizeof(d));
        d.rec = r; d.eval = R.pos; d.f_sym0 = (int)roundf(R.f_bb); d.ph_eval = R.osc_phase;
        fd.push_back(d);
        first.push_back(R.first_after_sync ? 1 : 0);
        who.push_back(r);
      }
      if (!fd.empty())
      {
        CK(dec->d_desc.reserve(sizeof(FrameDesc) * fd.size() + fd.size() + 64));
        CK(dec->d_start.reserve(sizeof(int) * fd.size()));
        uint8_t * dfirst = dec->d_desc.as<uint8_t>() + sizeof(FrameDesc) * fd.size();
        UP(dec->d_desc.p, fd.data(), sizeof(FrameDesc) * fd.size());
        UP(dfirst, first.data(), first.size());
        {
          long long upto = 0;
          for (auto & d : fd) upto = std::max(upto, (long long)d.eval + T_U);
          CK(need_upto(upto));
        }
        dec->span_begin(ST_PRS);
        CK(launch_prs_corr(st, ctx->tab, dec->d_desc.as<FrameDesc>(), (int)fd.size(), d_rin, fmt, thr0, 2.0f * thr0, dfirst,
                           dec->cfg.strongest_peak, dec->d_start.as<int>(), &ctx->launches));
        dec->span_end();
        CK(dec->h_start.reserve(sizeof(int) * fd.size()));
        const int * si = dec->h_start.as<int>();
        CK(cudaMemcpyAsync(dec->h_start.p, dec->d_start.p, sizeof(int) * fd.size(), cudaMemcpyDeviceToHost, st));
        SYNC();
        for (size_t i = 0; i < who.size(); i++)
        {
          Recording & R = dec->recs[who[i]];
          if (si[i] < 0)
          {
            // no peak: the 2048 samples are consumed and the time sync starts over (dab_processor.cpp:397-401)
            R.osc_phase = mod_fs_host((long long)R.osc_phase - (long long)roundf(R.f_bb) * T_U);
            R.pos += T_U;
            R.state = RecState::WAIT_SYNC;
          }
          else R.known_start = si[i];
        }
        win_recs.erase(std::remove_if(win_recs.begin(), win_recs.end(), [&](int r) { return dec->recs[r].state != RecState::EVAL; }), win_recs.end());
        if (win_recs.empty()) continue;
      }
    }

    // ---- frame layout. A window is grown in passes: lay out the frames that follow the verified ones assuming the PRS
    //      peak stays at T_g, run the cheap kernels on them (CP correlation, PRS correlation; coarse AFC for a careful
    //      frame), resolve the scalar AFC / clock recurrences on the host, and keep the frames up to the first one whose
    //      measured peak differs from the layout. That frame's peak is now known, so the next pass continues from it.
    //      The expensive kernels run once per round, over verified frames only.
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
    std::vector<Plan> plans;
    for (int r : win_recs)
    {
      Recording & R = dec->recs[r];
      int want = R.force_window > 0 ? R.force_window : ((R.w_careful && !R.careful_spec) ? 1 : dec->cfg.max_window);
      want = (int)std::min<long long>(want, std::max<long long>(1, budget / std::max<size_t>(1, win_recs.size())));
      want = std::min(want, R.slot_cap - R.n_slots);
      plans.push_back({ r, want, {}, true, R.known_start, 0, 0, 0, 75 });
      plans.back().fr.reserve((size_t)std::max(want, 1));
    }
    const long long resident = resident_upto();
    bool first_pass = true;
    dab::HostPool & pool = ctx->host_pool();
    tr("  plans made");
    while (true)
    {
      // tail layout of the open plans: positions first (a few integer operations per frame), then the descriptors of all
      // plans filled in by the pool
      long long window_end = 0;
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
      // (plan, first frame, end frame) pieces of at most 1024 frames: one long recording is a single plan, the pool works on pieces
      std::vector<std::array<int, 3>> pieces;
      for (size_t pi = 0; pi < plans.size(); pi++)
        if (plans[pi].open)
          for (int j0 = 0; j0 < plans[pi].t_frames; j0 += 1024) pieces.push_back({ (int)pi, j0, std::min(plans[pi].t_frames, j0 + 1024) });
      pool.parallel_for((int)pieces.size(), [&](int k) {
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
      const int n_tail = (int)ctl.size();
      if (n_tail == 0) break;
      if (trace) fprintf(stderr, "[dabstar]     pass: %d tail frames\n", n_tail);
      tr("  tail laid out");
      CK(need_upto(window_end));
      // descriptors go from the control records straight into the pinned staging area, a share per pool thread
      auto upload_descs = [&](int n) -> int {
        unsigned char * stage = nullptr;
        if (int r_ = upload_begin(ctx, sizeof(FrameDesc) * (size_t)n, &stage)) return r_;
        FrameDesc * o = reinterpret_cast<FrameDesc *>(stage);
        const int parts = std::max(1, std::min(n / 512, 16));
        pool.parallel_for(parts, [&](int k) {
          for (int i = (int)((long long)n * k / parts); i < (int)((long long)n * (k + 1) / parts); i++) o[i] = ctl[(size_t)i].desc;
        });
        return upload_commit(ctx, dec->d_desc.p, stage, sizeof(FrameDesc) * (size_t)n);
      };
      CK(dec->d_desc.reserve(sizeof(FrameDesc) * (size_t)n_tail + (size_t)n_tail + 64));
      if (int r_ = upload_descs(n_tail)) return r_;
      FrameDesc * d_fd = dec->d_desc.as<FrameDesc>();

      // CP correlation on raw samples (all tail frames) and coarse AFC (first frame of a careful window)
      CK(dec->d_cp.reserve(sizeof(float2) * (size_t)n_tail));
      dec->span_begin(ST_CP);
      CK(launch_cp_corr(st, d_fd, n_tail, d_rin, fmt, dec->d_cp.as<float2>(), &ctx->launches));
      dec->span_end();
      CK(dec->h_cp.reserve(sizeof(float2) * (size_t)n_tail));
      const float2 * cp = dec->h_cp.as<float2>();
      CK(cudaMemcpyAsync(dec->h_cp.p, dec->d_cp.p, sizeof(float2) * (size_t)n_tail, cudaMemcpyDeviceToHost, st));
      std::vector<int> coarse((size_t)n_tail, 0);
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

      // scalar recurrences (dab_processor.cpp:205-251), with the control state after every frame
      std::vector<CtlSnapshot> after((size_t)n_tail), before_tail(plans.size());
      std::vector<uint8_t> first_flags((size_t)n_tail, 0);
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
      auto recur_plan = [&](size_t pi) {
        Plan & pl = plans[pi];
        if (!pl.open) return;
        Recording & R = dec->recs[pl.rec];
        before_tail[pi] = take(R);
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
          ctl_finish_frame(R, cp[i], ran_coarse, coarse[i], fc, spec_f[pi], spec_ph[(size_t)i]);
          fc.desc.rec = pl.rec;
          fc.desc.slot = slot;
          fc.desc.xslot = i;
          ctl[i] = fc;
          after[i] = take(R);
        }
      };
      pool.parallel_for((int)plans.size(), [&](int pi) { recur_plan((size_t)pi); });
      if (int r_ = upload_descs(n_tail)) return r_;
      tr("  recurrences done");

      // PRS peak of every tail frame
      uint8_t * d_first = dec->d_desc.as<uint8_t>() + sizeof(FrameDesc) * (size_t)n_tail;
      UP(d_first, first_flags.data(), (size_t)n_tail);
      CK(dec->d_start.reserve(sizeof(int) * (size_t)n_tail));
      dec->span_begin(ST_PRS);
      CK(launch_prs_corr(st, ctx->tab, d_fd, n_tail, d_rin, fmt, thr0, 2.0f * thr0, d_first, dec->cfg.strongest_peak, dec->d_start.as<int>(), &ctx->launches));
      dec->span_end();
      CK(dec->h_start.reserve(sizeof(int) * (size_t)n_tail));
      const int * start = dec->h_start.as<int>();
      CK(cudaMemcpyAsync(dec->h_start.p, dec->d_start.p, sizeof(int) * (size_t)n_tail, cudaMemcpyDeviceToHost, st));
      SYNC();
      tr("  prs synced");

      std::atomic<int> n_open{ 0 };
      pool.parallel_for((int)plans.size(), [&](int pi_) {
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
      const bool any_open = n_open.load() > 0;
      first_pass = false;
      tr("layout pass done");
      if (!any_open) break;
    }

    // ---- this round's verified frames
    int n_round = 0;
    {
      std::vector<Plan> kept;
      for (auto & pl : plans)
      {
        Recording & R = dec->recs[pl.rec];
        if (pl.fr.empty())
        {
          if (pl.event == 1)
          {
            // no peak: the 2048 samples are consumed and the time sync starts over (dab_processor.cpp:397-401)
            R.cnt_windows++;
            R.osc_phase = mod_fs_host((long long)R.osc_phase - (long long)roundf(R.f_bb) * T_U);
            R.pos += T_U;
            R.state = RecState::WAIT_SYNC;
          }
          else { R.state = RecState::DONE; R.held = dec->streaming; R.held_state = 0; } // nothing left to read
          continue;
        }
        R.w_first_desc = n_round;
        R.w_frames = (int)pl.fr.size();
        n_round += (int)pl.fr.size();
        budget -= (long long)pl.fr.size();
        kept.push_back(std::move(pl));
      }
      plans.swap(kept);
    }
    if (plans.empty()) continue;
    dec->cnt_rounds++;
    const int n_desc = n_round;
    ctl.resize((size_t)n_desc);
    CK(dec->d_desc.reserve(sizeof(FrameDesc) * (size_t)n_desc + 64));
    unsigned char * desc_stage = nullptr;
    if (int r_ = upload_begin(ctx, sizeof(FrameDesc) * (size_t)n_desc, &desc_stage)) return r_;
    {
      std::vector<std::array<int, 3>> pieces;
      for (size_t pi = 0; pi < plans.size(); pi++)
        for (int j0 = 0; j0 < (int)plans[pi].fr.size(); j0 += 1024) pieces.push_back({ (int)pi, j0, std::min((int)plans[pi].fr.size(), j0 + 1024) });
      pool.parallel_for((int)pieces.size(), [&](int k) {
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
    }
    if (trace)
      fprintf(stderr, "[dabstar] round %lld t=%.3f ms: %zu recordings, %d frames, chunks resident %d/%d waited %d\n", dec->cnt_rounds,
              std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_run0).count(), plans.size(), n_desc, dec->chunks_done, dec->n_chunks,
              dec->chunks_waited);
    if (int r_ = upload_commit(ctx, dec->d_desc.p, desc_stage, sizeof(FrameDesc) * (size_t)n_desc)) return r_;
    FrameDesc * d_fd = dec->d_desc.as<FrameDesc>();

    cudaEvent_t wake_ev = nullptr; // end of the round's last demapper launch
    // ---- heavy pass: FFT (+ingest, derotation, de-interleave) -> demap -> FIC, one launch of each over the whole window
    CK(dec->d_X.reserve((size_t)x_frame_bytes * (size_t)n_desc));
    FrameQualSnap * d_qsnap = nullptr;
    if (dec->frame_quality)
    {
      CK(dec->d_qsnap.reserve(sizeof(FrameQualSnap) * (size_t)n_desc));
      d_qsnap = dec->d_qsnap.as<FrameQualSnap>();
    }
    if (int e = sync_profiles(ctx)) return e;
    if (int e = reserve_viterbi_ws(ctx, 4 * n_desc, FIC_OUT + 6)) return e;
    {
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
          if (R.tii_flags.empty()) continue;
          if (tii.empty()) tii.assign((size_t)n_desc, 0);
          for (int j = 0; j < (int)pl.fr.size(); j++)
          {
            const size_t f = (size_t)R.n_slots + (size_t)j;
            if (f < R.tii_flags.size()) tii[(size_t)R.w_first_desc + (size_t)j] = R.tii_flags[f];
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
    }

    tr("heavy pass enqueued");
    // ---- read back the FIB CRC flags
    // (one copy of the slot range this round touched: a copy per recording costs more in launch overhead than the bytes saved)
    std::vector<uint8_t> crc((size_t)n_desc * 12);
    {
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
      if (wake_ev) { CK(cudaEventSynchronize(wake_ev)); pool.prewake(); }
      SYNC();
      for (auto & pl : plans)
      {
        Recording & R = dec->recs[pl.rec];
        memcpy(crc.data() + (size_t)R.w_first_desc * 12, dec->h_crc.as<uint8_t>() + (size_t)(ctl[R.w_first_desc].desc.slot - s_lo) * 12, pl.fr.size() * 12);
      }
    }

    tr("heavy pass done");
    // ---- accept: the FIC success ratio must not have fallen below 30 % at a frame start (that frame needs the coarse AFC)
    // (the OFDM state of a rolled-back recording is still in its current buffer: nothing to restore on the device)
    pool.parallel_for((int)plans.size(), [&](int pi) {
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
        if (pl.event == 1 && R.state == RecState::EVAL)
        {
          // the frame after this window has no PRS peak (dab_processor.cpp:397-401)
          R.osc_phase = mod_fs_host((long long)R.osc_phase - (long long)roundf(R.f_bb) * T_U);
          R.pos += T_U;
          R.state = RecState::WAIT_SYNC;
        }
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

  // ================= self-configuration: sub-channels and CIF counter from the recording's own FIC (FIG 0/0, 0/1)
  // FibDecoder::process_FIB sees the CRC-good FIBs in stream order; a Backend is taken to exist from the frame after the one
  // whose FIC first described its sub-channel (in the reference that moment is a GUI action), EtiGenerator samples the
  // sub-channel list and the CIF counter at symbol 4 of every frame, i.e. after that frame's own FIC.
  {
    bool any = false;
    for (int r = 0; r < n_rec; r++) any = any || (dec->recs[r].auto_cfg && dec->recs[r].n_slots > 0);
    if (any)
    {
      CK(dec->h_fib.reserve((size_t)dec->total_slots * 3072));
      for (int r = 0; r < n_rec; r++)
      {
        Recording & R = dec->recs[r];
        const int fs = std::min(R.slot_cap, R.n_slots + (R.partial_syms > 3 ? 1 : 0));
        if (R.auto_cfg && fs > 0)
          CK(cudaMemcpyAsync(dec->h_fib.as<uint8_t>() + (size_t)R.slot_base * 3072, dec->d_fib.as<uint8_t>() + (size_t)R.slot_base * 3072, (size_t)fs * 3072, cudaMemcpyDeviceToHost, st));
      }
      SYNC();
      for (int r = 0; r < n_rec; r++)
      {
        Recording & R = dec->recs[r];
        if (!R.auto_cfg || R.n_slots == 0) continue;
        dabstar_fib_parser * fp = nullptr;
        if (dabstar_fib_parser_create(&fp) != 0) return ctx->fail(DABSTAR_E_NOMEM, "fib parser");
        R.msc.clear();
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
          if (e.restarts > 0 && e.n_subch < known) { R.msc.clear(); known = 0; } // the parser dropped its database
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
            R.msc.push_back(m);
          }
          known = e.n_subch;
          R.ens = e;
        }
        for (int f = n_f; f <= R.n_slots; f++) { R.cif_hi_f[f] = f > 0 ? R.cif_hi_f[f - 1] : -1; R.cif_lo_f[f] = f > 0 ? R.cif_lo_f[f - 1] : -1; }
        dabstar_fib_parser_destroy(fp);
      }
      if (int e = sync_profiles(ctx)) return e;
    }
  }

  // ================= TII (dab_processor.cpp:273-300) for self-configured recordings: the null symbol after frame f carries TII
  // when the CIF counter the FIB decoder holds after that frame's FIC has (count & 7) >= 4. Those null symbols are
  // transformed again (the demapper's spectrum buffer is per window), accumulated tiiFramesToCount at a time and searched;
  // a time re-synchronisation resets the detector and the counter (dab_processor.cpp:150-152).
  {
    struct Seg { int rec; std::vector<int> frames; bool reset_before; };
    std::map<int, std::vector<Seg>> per_rec;
    for (int r = 0; r < n_rec; r++)
    {
      Recording & R = dec->recs[r];
      R.tii_events.clear();
      if (!R.tii.on || !R.auto_cfg || R.n_slots == 0) continue;
      const int need = std::max(1, R.tii.frames_to_count);
      std::vector<int> acc;
      bool reset_pending = false;
      size_t si = 0;
      for (int f = 0; f < R.n_slots; f++)
      {
        while (si < R.sync_frames.size() && R.sync_frames[si] <= f) { acc.clear(); reset_pending = true; si++; }
        if (f >= (int)R.cif_hi_f.size() || R.cif_hi_f[f] < 0) continue; // get_cif_count() is still 0: not a TII null symbol
        if ((((R.cif_hi_f[f] * 250 + R.cif_lo_f[f]) & 7) >= 4))
        {
          acc.push_back(f);
          if ((int)acc.size() >= need) { per_rec[r].push_back({ r, acc, reset_pending }); acc.clear(); reset_pending = false; }
        }
      }
    }
    if (!per_rec.empty())
    {
      // recordings with more events first: event e then concerns the first n_e detectors
      std::vector<int> order;
      for (auto & kv : per_rec) order.push_back(kv.first);
      std::sort(order.begin(), order.end(), [&](int a, int b) { return per_rec[a].size() != per_rec[b].size() ? per_rec[a].size() > per_rec[b].size() : a < b; });
      dabstar_tii * det = nullptr;
      if (int e = dabstar_tii_create(ctx, (int)order.size(), &det)) return e;
      std::unique_ptr<dabstar_tii, void (*)(dabstar_tii *)> guard(det, dabstar_tii_destroy);
      const int need = std::max(1, dec->recs[order[0]].tii.frames_to_count), cap = 128;
      for (int r : order)
        if (std::max(1, dec->recs[r].tii.frames_to_count) != need || dec->recs[r].tii.threshold_db != dec->recs[order[0]].tii.threshold_db ||
            dec->recs[r].tii.collisions != dec->recs[order[0]].tii.collisions || dec->recs[r].tii.sub_id != dec->recs[order[0]].tii.sub_id)
          return ctx->fail(DABSTAR_E_INVALID, "TII settings must be the same for every recording of a decoder");
      dabstar_tii_set_collisions(det, dec->recs[order[0]].tii.collisions, dec->recs[order[0]].tii.sub_id);
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
        if (e == 0) e = dabstar_tii_process(det, dec->recs[order[0]].tii.threshold_db, res.data(), cap, cnt.data());
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
    }
  }

  // ================= MSC: all logical frames of all sub-channels in one batch per profile size
  if (!dec->cfg.scan_mode)
  {
    // One job per sub-channel and CIF (several hundred thousand for a full ensemble), grouped by code-word length (one launch
    // per length: shared-memory footprint). The host only lists one range per Backend; the jobs are written on the device.
    // The decoded bits are laid out group by group (code-word length), so that a group's payload can be packed and copied
    // to the host while the next group is decoded; nothing on the host waits between the groups.
    struct Group { std::vector<BackendJobRange> ranges; std::vector<MscOut *> outs; int n_jobs = 0; long long bits = 0, bit_base = 0; int job_base = 0; };
    std::map<int, Group> groups;
    for (int r = 0; r < n_rec; r++)
    {
      Recording & R = dec->recs[r];
      const int n_cifs = 4 * R.n_slots + std::max(0, (R.partial_syms - 3) / 18);
      for (size_t c = 0; c < R.msc.size(); c++)
      {
        MscOut & m = R.msc[c];
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
    if (out_total > 0)
    {
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
      {
        cudaEvent_t ev = dec->ev_get();
        CK(cudaEventRecord(ev, dec->copy_stream));
        CK(cudaStreamWaitEvent(st, ev, 0)); // the run's final synchronisation of `st` covers the copies
      }
      tr("msc enqueued");
    }
  }
  // ================= ETI: every sub-channel of every CIF through EtiGenerator's own de-interleaver (eti_generator.cpp:90-204)
  // The generator's ring holds 16 whole CIFs and, unlike Backend, emits with its 17th CIF but loses the 16th from the
  // history while `Minor` is still -1 (the CIF is stored, index_Out does not advance, the next CIF overwrites it). Seen
  // from ETI frame n (n = 0 is CIF 16 of the run) de-interleaver row m therefore reads entry n - 1 + m of the CIF sequence
  // 0..14, 16, 17, ...; entry -1 (row 0 of frame 0) is the slot about to be overwritten, which still holds CIF 15.
  struct EtiRef { int rec; long long bit_off; int n_out; };
  std::vector<EtiRef> eti_refs;
  {
    std::map<int, std::vector<VitJob>> by_steps;
    long long bits_total = 0;
    for (int r = 0; r < n_rec; r++)
    {
      Recording & R = dec->recs[r];
      R.eti.clear();
      if (!R.eti_on || R.msc.empty()) continue;
      const int n_cifs = 4 * R.n_slots + std::max(0, (R.partial_syms - 3) / 18);
      const int n_out = std::max(0, n_cifs - 16);
      if (n_out == 0) continue;
      eti_refs.push_back({ r, bits_total, n_out });
      for (int n = 0; n < n_out; n++)
        for (MscOut & m : R.msc)
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
    if (bits_total > 0)
    {
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
    }
  }
  tr("rounds done");
  // FIB bits of all accepted frames
  // The decoded FIBs leave the device packed 8 bits per byte (32 bytes per FIB, the reference's FIC dump format,
  // fic_decoder.cpp:291-308): 3.8 MB instead of 30.6 MB per 10 000 frames; dabstar_decoder_fib_bits unpacks on request.
  if (dec->total_slots > 0)
  {
    const long long n_bytes = (long long)dec->total_slots * 384;
    CK(dec->d_fibp.reserve((size_t)n_bytes));
    CK(dec->h_fibp.reserve((size_t)n_bytes));
    CK(launch_pack_bits(st, dec->d_fib.as<uint8_t>(), dec->d_fibp.as<uint8_t>(), n_bytes, &ctx->launches));
    CK(cudaMemcpyAsync(dec->h_fibp.p, dec->d_fibp.p, (size_t)n_bytes, cudaMemcpyDeviceToHost, st));
  }
  std::vector<uint8_t> eti_packed;
  if (!eti_refs.empty())
  {
    const EtiRef & last = eti_refs.back();
    long long bits_total = last.bit_off;
    for (int n = 0; n < last.n_out; n++)
      for (const MscOut & m : dec->recs[last.rec].msc) if (m.first_seen <= 4 + (n >> 2)) bits_total += 24LL * m.sc.bit_rate;
    eti_packed.resize((size_t)(bits_total / 8));
    CK(cudaMemcpyAsync(eti_packed.data(), dec->d_etipacked.p, eti_packed.size(), cudaMemcpyDeviceToHost, st));
  }
  CK(cudaEventRecord(dec->ev1, st));
  SYNC();
  if (trace) fprintf(stderr, "[dabstar] run done t=%.3f ms\n", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_run0).count());
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
      for (const MscOut & m : R.msc) if (m.first_seen <= fr) { streams.push_back(MscOut()); streams.back().sc = m.sc; need += 4 + 3 * (size_t)m.sc.bit_rate; }
      if (streams.size() > 64 || need > 6144) return ctx->fail(DABSTAR_E_INVALID, "ETI frame overflow: %zu streams, %zu bytes", streams.size(), need);
      const bool own = R.auto_cfg && fr < (int)R.cif_hi_f.size() && R.cif_hi_f[fr] >= 0;
      int o = eti_header(f, own ? R.cif_hi_f[fr] : R.eti_cif_hi, own ? R.cif_lo_f[fr] : R.eti_cif_lo, n & 3, streams);
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
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, dec->ev0, dec->ev1));
  dec->last_ms = ms;
  for (auto & sp : dec->spans)
  {
    float t = 0;
    if (cudaEventElapsedTime(&t, sp.a, sp.b) == cudaSuccess) dec->stage_ms[sp.stage] += t;
  }
  for (auto & hs : dec->heavy_spans)
  {
    float t = 0;
    if (cudaEventElapsedTime(&t, hs.first, hs.second) == cudaSuccess) dec->heavy_ms += t;
  }
  for (auto & hs : dec->fft_demap_spans)
  {
    float t = 0;
    if (cudaEventElapsedTime(&t, hs.first, hs.second) == cudaSuccess) dec->fft_demap_ms += t;
  }
  return 0;
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
  for (auto & R : dec->recs) R.tii_flags.clear();
  int rc = decoder_run_pass(dec, iq, n_samples, mem);
  double total_ms = dec->last_ms;
  for (int pass = 1; rc == 0 && pass <= 3; pass++)
  {
    bool again = false;
    for (auto & R : dec->recs)
    {
      if (!R.auto_cfg || !R.tii_nulls || R.n_slots == 0) continue;
      std::vector<uint8_t> flags((size_t)R.n_slots, 0);
      for (int f = 0; f < R.n_slots; f++)
        if (f < (int)R.cif_hi_f.size() && R.cif_hi_f[f] >= 0) flags[f] = (((R.cif_hi_f[f] * 250 + R.cif_lo_f[f]) & 7) >= 4) ? 1 : 0;
      bool any = false;
      for (uint8_t v : flags) any = any || v;
      std::vector<uint8_t> used = R.tii_flags;
      used.resize(flags.size(), 0);
      if (any && used != flags) again = true;
      R.tii_flags = std::move(flags);
    }
    if (!again) break;
    // the recordings are resident on the device after the first pass
    std::vector<const void *> dptr(dec->recs.size());
    for (size_t r = 0; r < dec->recs.size(); r++) dptr[r] = dec->recs[r].d_iq;
    rc = decoder_run_pass(dec, dptr.data(), n_samples, DABSTAR_MEM_DEVICE);
    total_ms += dec->last_ms;
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
  for (const auto & m : dec->recs[recording].msc) if (m.sc.sub_ch_id == sub_ch_id) return &m;
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
  // mMeanSigmaSqFreqCorr (ofdm_decoder.cpp:296-300): at symbol 1 of every frame, from the cyclic-prefix phase the
  // previous frame left behind (dab_processor.cpp:236-240,342); not touched by OfdmDecoder::reset()
  const Recording & R = dec->recs[recording];
  float sigma = 0.0f, phase = 0.0f;
  for (const auto & fi : R.frames)
  {
    const float fc = phase / TWO_PI_F * 1000.0f;
    sigma += 0.2f * (fc * fc - sigma);
    phase = fi.phase_cp;
  }
  return quality_from_state(ctx, dec->d_states.as<OfdmStateDev>() + recording + (size_t)R.state_cur * dec->recs.size(), sigma, out);
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
  // the mMeanSigmaSqFreqCorr replay of dabstar_decoder_quality, one frame at a time
  float sigma = 0.0f, phase = 0.0f;
  for (int f = 0; f < n; f++)
  {
    const float fc = phase / TWO_PI_F * 1000.0f;
    sigma += 0.2f * (fc * fc - sigma);
    phase = R.frames[(size_t)f].phase_cp;
    quality_from_sums(fq[(size_t)f], sigma, out + 6 * (size_t)f);
  }
  return R.n_slots;
}
extern "C" int dabstar_decoder_enable_tii(dabstar_decoder * dec, int recording, int enable, int frames_to_count, int threshold_db, int collisions, int sub_id)
{
  if (!dec || recording < 0 || recording >= (int)dec->recs.size()) return DABSTAR_E_INVALID;
  if (enable && (frames_to_count < 1 || sub_id < 0 || sub_id > 23)) return dec->ctx->fail(DABSTAR_E_INVALID, "TII: frames_to_count %d, sub id %d", frames_to_count, sub_id);
  Recording & R = dec->recs[recording];
  R.tii.on = enable != 0;
  if (enable) { R.tii.frames_to_count = frames_to_count; R.tii.threshold_db = threshold_db; R.tii.collisions = collisions ? 1 : 0; R.tii.sub_id = sub_id; }
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

namespace
{
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
} // namespace

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
  StateBlobHdr h;
  memset(&h, 0, sizeof(h));
  h.magic = STATE_MAGIC; h.version = 1; h.bytes = need;
  h.stream_pos = R.abs_pos0 + R.pos;
  h.abs_frames = R.abs_frames + R.n_slots;
  h.rec_state = R.held_state;
  h.osc_phase = R.osc_phase; h.fic_ratio = R.fic_ratio; h.first_after_sync = R.first_after_sync ? 1 : 0; h.known_start = R.known_start;
  h.spec_ok = R.spec_ok ? 1 : 0; h.careful_spec = R.careful_spec ? 1 : 0; h.last_start = R.last_start; h.ofdm_reset = R.ofdm_reset ? 1 : 0;
  h.f_sync = R.f_sync; h.f_bb = R.f_bb; h.clock_err = R.clock_err; h.phase_cp = R.phase_cp;
  h.hist = hist_frames_after(R);
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
  rs.stream_pos = h.stream_pos; rs.abs_frames = h.abs_frames; rs.lead = lead_samples;
  rs.rec_state = h.rec_state; rs.osc_phase = h.osc_phase; rs.fic_ratio = h.fic_ratio; rs.first_after_sync = h.first_after_sync; rs.known_start = h.known_start;
  rs.spec_ok = h.spec_ok; rs.careful_spec = h.careful_spec; rs.last_start = h.last_start; rs.ofdm_reset = h.ofdm_reset;
  rs.f_sync = h.f_sync; rs.f_bb = h.f_bb; rs.clock_err = h.clock_err; rs.phase_cp = h.phase_cp;
  rs.hist = h.hist;
  const unsigned char * in = static_cast<const unsigned char *>(blob) + sizeof(h);
  rs.ofdm.assign(in, in + sizeof(OfdmStateDev));
  rs.soft.resize((size_t)h.hist * FRAME_SOFT);
  if (h.hist > 0) memcpy(rs.soft.data(), in + sizeof(OfdmStateDev), sizeof(int16_t) * rs.soft.size());
  return 0;
}
