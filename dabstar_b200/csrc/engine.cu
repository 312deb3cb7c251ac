// engine.cu — the context, its staging helpers and the stage taps behind include/dabstar_b200.h (the whole-path decoder is
// decoder.cu).
#include "context.h"
#include "tables.h"
#include "fft2048.cuh"

using namespace dab;

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

int sync_stream(dabstar_ctx * ctx)
{
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->arena_off = 0;
  return 0;
}

int upload(dabstar_ctx * ctx, void * dst, const void * src, size_t bytes)
{
  if (bytes == 0) return 0;
  unsigned char * stage = nullptr;
  if (int r = upload_begin(ctx, bytes, &stage)) return r;
  memcpy(stage, src, bytes);
  return upload_commit(ctx, dst, stage, bytes);
}
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
// Registers a profile: appends its step table (viterbi.cuh: vit_step_entry_make) and returns its index.
static int push_profile(dabstar_ctx * ctx, VitProfile p)
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

static int get_identity_profile(dabstar_ctx * ctx, int n_bits)
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
static int stage_in(dabstar_ctx * ctx, DevBuf & buf, const void * src, size_t bytes, int mem, const void ** out)
{
  if (mem == DABSTAR_MEM_DEVICE) { *out = src; return 0; }
  CK(buf.reserve(bytes));
  CK(cudaMemcpyAsync(buf.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  *out = buf.p;
  return 0;
}
static int stage_out_begin(dabstar_ctx * ctx, DevBuf & buf, void * dst, size_t bytes, int mem, void ** out)
{
  if (mem == DABSTAR_MEM_DEVICE) { *out = dst; return 0; }
  CK(buf.reserve(bytes));
  *out = buf.p;
  return 0;
}
static int stage_out_end(dabstar_ctx * ctx, const void * dev, void * dst, size_t bytes, int mem)
{
  if (mem == DABSTAR_MEM_HOST) CK(cudaMemcpyAsync(dst, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
// Frame descriptors and the recordings they index, uploaded back to back into scratch[3]; returns the device copies.
static int upload_frames(dabstar_ctx * ctx, const std::vector<FrameDesc> & fd, const std::vector<RecInput> & rin, FrameDesc ** dfd, RecInput ** drin)
{
  CK(ctx->scratch[3].reserve(sizeof(FrameDesc) * fd.size() + sizeof(RecInput) * rin.size() + 64));
  *dfd = ctx->scratch[3].as<FrameDesc>();
  *drin = reinterpret_cast<RecInput *>(*dfd + fd.size());
  UP(*dfd, fd.data(), sizeof(FrameDesc) * fd.size());
  UP(*drin, rin.data(), sizeof(RecInput) * rin.size());
  return 0;
}

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
// Grows a device buffer of which the first `used` bytes are live, keeping them.
static int reserve_keep(dabstar_ctx * ctx, cudaStream_t s, DevBuf & b, size_t used, size_t bytes)
{
  if (bytes <= b.cap) return 0;
  DevBuf n;
  CK(n.reserve(std::max(bytes, 2 * b.cap)));
  if (used) CK(cudaMemcpyAsync(n.p, b.p, used, cudaMemcpyDeviceToDevice, s));
  CK(cudaStreamSynchronize(s)); // the old buffer is freed below
  std::swap(b.p, n.p);
  std::swap(b.cap, n.cap);
  return 0;
}

int run_dabplus(dabstar_ctx * ctx, cudaStream_t s, DabplusPass & p)
{
  if (!ctx->d_gf.p)
  {
    std::vector<uint8_t> gf;
    std::vector<uint16_t> syn;
    dabplus_host_tables(gf, syn);
    CK(ctx->d_gf.reserve(gf.size()));
    CK(ctx->d_fc_syn.reserve(sizeof(uint16_t) * syn.size()));
    CK(cudaMemcpy(ctx->d_gf.p, gf.data(), gf.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->d_fc_syn.p, syn.data(), sizeof(uint16_t) * syn.size(), cudaMemcpyHostToDevice));
  }
  if (!p.ev0) { CK(cudaEventCreate(&p.ev0)); CK(cudaEventCreate(&p.ev1)); }
  const int ns = (int)p.streams.size();
  long long n_win = 0, est_entries = 0, est_bytes = 0;
  for (DabplusStream & st : p.streams)
  {
    const long long nw = std::max(0, st.n_frames - 4), sf = 110LL * (st.bit_rate / 8);
    st.win0 = n_win;
    st.att0 = n_win;
    n_win += nw;
    est_entries += st.n_frames / 5 + (nw > 0 ? 2 : 0); // a clean stream, plus room for a few extra attempts
    est_bytes += (st.n_frames / 5 + (nw > 0 ? 2 : 0)) * sf;
  }
  p.n_out.assign((size_t)ns, 0);
  p.scanned = n_win;
  p.decoded = 0;
  p.rounds = 0;
  p.ms = 0;
  p.rec = nullptr;
  p.payload = nullptr;
  if (n_win == 0) return 0;
  CK(cudaEventRecord(p.ev0, s));
  CK(p.d_streams.reserve(sizeof(DabplusStream) * (size_t)ns));
  CK(p.d_state.reserve((size_t)n_win));
  CK(p.d_slot.reserve(sizeof(int) * (size_t)n_win));
  CK(p.d_list.reserve(sizeof(DabplusEntry) * (size_t)n_win)); // every window is listed at most once
  CK(p.d_att.reserve(sizeof(int) * (size_t)n_win));
  const size_t meta_bytes = sizeof(DabplusMeta) + sizeof(int) * (size_t)ns;
  CK(p.d_meta.reserve(meta_bytes));
  CK(p.h_meta.reserve(meta_bytes));
  CK(p.d_rec.reserve(sizeof(SuperFrameRec) * (size_t)est_entries));
  CK(p.d_pay.reserve((size_t)est_bytes));
  DabplusStream * d_st = p.d_streams.as<DabplusStream>();
  DabplusMeta * d_meta = p.d_meta.as<DabplusMeta>();
  int * d_att_n = reinterpret_cast<int *>(d_meta + 1);
  CK(cudaMemcpyAsync(d_st, p.streams.data(), sizeof(DabplusStream) * (size_t)ns, cudaMemcpyHostToDevice, s));
  CK(cudaMemsetAsync(d_meta, 0, sizeof(DabplusMeta), s));
  CK(launch_dabplus_scan(s, d_st, ns, n_win, ctx->d_gf.p, p.d_state.as<uint8_t>(), &ctx->launches));
  DabplusMeta done{ 0, 0 };
  const DabplusMeta * h_meta = p.h_meta.as<DabplusMeta>();
  while (true)
  {
    CK(launch_dabplus_walk(s, d_st, ns, p.d_state.as<uint8_t>(), p.d_att.as<int>(), d_meta, d_att_n, p.d_list.as<DabplusEntry>(), p.d_slot.as<int>(), &ctx->launches));
    CK(cudaMemcpyAsync(p.h_meta.p, d_meta, meta_bytes, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    p.rounds++;
    const DabplusMeta now = *h_meta;
    const int n_new = (int)(now.entries - done.entries);
    if (n_new == 0) break;
    if (int r = reserve_keep(ctx, s, p.d_rec, sizeof(SuperFrameRec) * done.entries, sizeof(SuperFrameRec) * now.entries)) return r;
    if (int r = reserve_keep(ctx, s, p.d_pay, (size_t)done.bytes, (size_t)now.bytes)) return r;
    CK(p.d_ler.reserve((size_t)n_new * DABPLUS_MAX_RS_DIMS));
    CK(launch_dabplus_decode(s, d_st, p.d_list.as<DabplusEntry>() + done.entries, n_new, ctx->d_gf.p, ctx->d_fc_syn.as<uint16_t>(), p.d_pay.as<uint8_t>(),
                             p.d_ler.as<int8_t>(), p.d_rec.as<SuperFrameRec>() + done.entries, p.d_state.as<uint8_t>(), &ctx->launches));
    p.decoded += n_new;
    done = now;
  }
  // the last walk's attempts are final: compact them in stream order
  const int * att_n = reinterpret_cast<const int *>(h_meta + 1);
  long long n_rec = 0, n_bytes = 0;
  for (int i = 0; i < ns; i++)
  {
    DabplusStream & st = p.streams[(size_t)i];
    p.n_out[(size_t)i] = att_n[i];
    st.out_rec0 = n_rec;
    st.out_pay0 = n_bytes;
    n_rec += att_n[i];
    n_bytes += (long long)att_n[i] * 110 * (st.bit_rate / 8);
  }
  const size_t rec_bytes = sizeof(SuperFrameRec) * (size_t)n_rec, out_bytes = rec_bytes + (size_t)n_bytes;
  if (n_rec > 0)
  {
    CK(p.d_out.reserve(out_bytes));
    CK(p.h_out.reserve(out_bytes));
    CK(cudaMemcpyAsync(d_st, p.streams.data(), sizeof(DabplusStream) * (size_t)ns, cudaMemcpyHostToDevice, s));
    CK(launch_dabplus_compact(s, d_st, ns, n_rec, p.d_att.as<int>(), p.d_slot.as<int>(), p.d_list.as<DabplusEntry>(), p.d_rec.as<SuperFrameRec>(), p.d_pay.as<uint8_t>(),
                              p.d_out.as<SuperFrameRec>(), p.d_out.as<uint8_t>() + rec_bytes, &ctx->launches));
    CK(cudaMemcpyAsync(p.h_out.p, p.d_out.p, out_bytes, cudaMemcpyDeviceToHost, s));
    p.rec = p.h_out.as<SuperFrameRec>();
    p.payload = p.h_out.as<uint8_t>() + rec_bytes;
  }
  CK(cudaEventRecord(p.ev1, s));
  CK(cudaStreamSynchronize(s));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, p.ev0, p.ev1));
  p.ms = ms;
  return 0;
}

extern "C" int dabstar_dabplus_decode(dabstar_ctx * ctx, const uint8_t * frame_bits, int bit_rate, int n_frames, dabstar_superframe * out, int cap,
                                      uint8_t * payload, int mem)
{
  if (!ctx || (!frame_bits && n_frames > 0) || n_frames < 0 || cap < 0 || (cap > 0 && !out)) return DABSTAR_E_INVALID;
  if (bit_rate < 8 || bit_rate > 192 || bit_rate % 8) return ctx->fail(DABSTAR_E_INVALID, "DAB+ bit rate %d", bit_rate);
  if (n_frames < 5) return 0;
  CK(cudaSetDevice(ctx->device));
  const size_t n_bits = (size_t)n_frames * 24 * bit_rate;
  const void * dbits;
  if (int r = stage_in(ctx, ctx->scratch[0], frame_bits, n_bits, mem, &dbits)) return r;
  CK(ctx->scratch[1].reserve(n_bits / 8)); // packed frames
  CK(launch_pack_bits(ctx->stream, (const uint8_t *)dbits, ctx->scratch[1].as<uint8_t>(), (long long)(n_bits / 8), &ctx->launches));
  DabplusPass & p = ctx->dabplus;
  p.streams.assign(1, DabplusStream{ ctx->scratch[1].as<uint8_t>(), bit_rate, n_frames, 0, 0, 0, 0 });
  if (int r = run_dabplus(ctx, ctx->stream, p)) return r;
  ctx->arena_off = 0;
  const int n_out = p.n_out[0], sf_bytes = 110 * (bit_rate / 8), n_copy = std::min(n_out, cap);
  for (int i = 0; i < n_copy; i++) out[i] = superframe_public(p.rec[i]);
  if (payload && n_copy > 0)
  {
    if (mem == DABSTAR_MEM_HOST) memcpy(payload, p.payload, (size_t)n_copy * sf_bytes);
    else CK(cudaMemcpy(payload, p.payload, (size_t)n_copy * sf_bytes, cudaMemcpyHostToDevice));
  }
  return n_out;
}

// ------------------------------------------------------------------------------------------------ MPEG layer II audio frames
int run_mp2(dabstar_ctx * ctx, cudaStream_t s, Mp2Pass & p)
{
  if (!p.ev0) { CK(cudaEventCreate(&p.ev0)); CK(cudaEventCreate(&p.ev1)); }
  const int ns = (int)p.streams.size();
  long long n_slots = 0;
  for (Mp2Stream & st : p.streams)
  {
    st.slot0 = n_slots;
    n_slots += st.n_frames;
  }
  p.n_out.assign((size_t)ns, Mp2Count{ 0, 0 });
  p.slots = n_slots;
  p.ms = 0;
  p.rec = nullptr;
  p.payload = nullptr;
  if (n_slots == 0) return 0;
  CK(cudaEventRecord(p.ev0, s));
  CK(p.d_streams.reserve(sizeof(Mp2Stream) * (size_t)ns));
  CK(p.d_cls.reserve((size_t)n_slots));
  CK(p.d_crc.reserve(sizeof(int2) * (size_t)n_slots));
  CK(p.d_hdr.reserve(sizeof(uint32_t) * (size_t)n_slots));
  CK(p.d_stage.reserve(sizeof(Mp2Rec) * (size_t)n_slots)); // a stream has at most one record per logical frame
  CK(p.d_stage_off.reserve(sizeof(long long) * (size_t)n_slots));
  CK(p.d_cnt.reserve(sizeof(Mp2Count) * (size_t)ns));
  CK(p.h_cnt.reserve(sizeof(Mp2Count) * (size_t)ns));
  Mp2Stream * d_st = p.d_streams.as<Mp2Stream>();
  CK(cudaMemcpyAsync(d_st, p.streams.data(), sizeof(Mp2Stream) * (size_t)ns, cudaMemcpyHostToDevice, s));
  CK(launch_mp2_scan(s, d_st, ns, n_slots, p.d_cls.as<uint8_t>(), p.d_crc.as<int2>(), p.d_hdr.as<uint32_t>(), &ctx->launches));
  CK(launch_mp2_walk(s, d_st, ns, p.d_cls.as<uint8_t>(), p.d_crc.as<int2>(), p.d_hdr.as<uint32_t>(), p.d_stage.as<Mp2Rec>(), p.d_stage_off.as<long long>(),
                     p.d_cnt.as<Mp2Count>(), &ctx->launches));
  CK(cudaMemcpyAsync(p.h_cnt.p, p.d_cnt.p, sizeof(Mp2Count) * (size_t)ns, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  const Mp2Count * cnt = p.h_cnt.as<Mp2Count>();
  long long n_rec = 0, n_bytes = 0;
  for (int i = 0; i < ns; i++)
  {
    Mp2Stream & st = p.streams[(size_t)i];
    p.n_out[(size_t)i] = cnt[i];
    st.out_rec0 = n_rec;
    st.out_pay0 = n_bytes;
    n_rec += cnt[i].recs;
    n_bytes += cnt[i].bytes;
  }
  const size_t rec_bytes = sizeof(Mp2Rec) * (size_t)n_rec, out_bytes = rec_bytes + (size_t)n_bytes;
  CK(p.d_out.reserve(out_bytes));
  CK(p.h_out.reserve(out_bytes));
  CK(cudaMemcpyAsync(d_st, p.streams.data(), sizeof(Mp2Stream) * (size_t)ns, cudaMemcpyHostToDevice, s));
  CK(launch_mp2_compact(s, d_st, ns, n_rec, p.d_stage.as<Mp2Rec>(), p.d_stage_off.as<long long>(), p.d_out.as<Mp2Rec>(), p.d_out.as<uint8_t>() + rec_bytes, &ctx->launches));
  CK(cudaMemcpyAsync(p.h_out.p, p.d_out.p, out_bytes, cudaMemcpyDeviceToHost, s));
  p.rec = p.h_out.as<Mp2Rec>();
  p.payload = p.h_out.as<uint8_t>() + rec_bytes;
  CK(cudaEventRecord(p.ev1, s));
  CK(cudaStreamSynchronize(s));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, p.ev0, p.ev1));
  p.ms = ms;
  return 0;
}

extern "C" int dabstar_mp2_frames(dabstar_ctx * ctx, const uint8_t * frame_bits, int bit_rate, int n_frames, dabstar_mp2_frame * out, int cap,
                                  uint8_t * payload, int mem)
{
  if (!ctx || (!frame_bits && n_frames > 0) || n_frames < 0 || cap < 0 || (cap > 0 && !out)) return DABSTAR_E_INVALID;
  if (!mp2_rate_ok(bit_rate)) return ctx->fail(DABSTAR_E_INVALID, "MP2: %d kbit/s is not a layer II bit rate", bit_rate);
  if (n_frames == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  const size_t n_bits = (size_t)n_frames * 24 * bit_rate;
  const void * dbits;
  if (int r = stage_in(ctx, ctx->scratch[0], frame_bits, n_bits, mem, &dbits)) return r;
  CK(ctx->scratch[1].reserve(n_bits / 8)); // packed frames
  CK(launch_pack_bits(ctx->stream, (const uint8_t *)dbits, ctx->scratch[1].as<uint8_t>(), (long long)(n_bits / 8), &ctx->launches));
  Mp2Pass & p = ctx->mp2;
  p.streams.assign(1, Mp2Stream{ ctx->scratch[1].as<uint8_t>(), bit_rate, n_frames, 0, 0, 0 });
  if (int r = run_mp2(ctx, ctx->stream, p)) return r;
  ctx->arena_off = 0;
  const int n_out = (int)p.n_out[0].recs, n_copy = std::min(n_out, cap);
  size_t bytes = 0;
  for (int i = 0; i < n_copy; i++)
  {
    out[i] = mp2_public(p.rec[i]);
    if (p.rec[i].status == MP2_OK) bytes += (size_t)p.rec[i].n_frames * 3 * bit_rate;
  }
  if (payload && bytes > 0)
  {
    if (mem == DABSTAR_MEM_HOST) memcpy(payload, p.payload, bytes);
    else CK(cudaMemcpy(payload, p.payload, bytes, cudaMemcpyHostToDevice));
  }
  return n_out;
}

// ------------------------------------------------------------------------------------------------ packet-mode data groups
int run_packet(dabstar_ctx * ctx, cudaStream_t s, PacketPass & p)
{
  if (!p.ev0) { CK(cudaEventCreate(&p.ev0)); CK(cudaEventCreate(&p.ev1)); }
  const int nsub = (int)p.subs.size(), ns = (int)p.streams.size();
  long long n_frames = 0, n_slots = 0, n_stage = 0;
  for (PacketSub & sb : p.subs)
  {
    sb.frame0 = n_frames;
    sb.slot0 = n_slots;
    n_frames += sb.n_frames;
    n_slots += (long long)sb.n_frames * (sb.bit_rate / 8);
  }
  for (PacketStream & st : p.streams)
  {
    const PacketSub & sb = p.subs[(size_t)st.sub];
    st.stage0 = n_stage;
    n_stage += (long long)sb.n_frames * (sb.bit_rate / 8); // a stream has at most one group per packet slot
  }
  p.n_out.assign((size_t)ns, PacketCount{});
  p.slots = n_slots;
  p.ms = 0;
  p.rec = nullptr;
  p.payload = nullptr;
  if (n_slots == 0 || ns == 0) return 0;
  CK(cudaEventRecord(p.ev0, s));
  CK(p.d_subs.reserve(sizeof(PacketSub) * (size_t)nsub));
  CK(p.d_streams.reserve(sizeof(PacketStream) * (size_t)ns));
  CK(p.d_slots.reserve(sizeof(PacketSlot) * (size_t)n_slots));
  CK(p.d_stage.reserve(sizeof(PacketStage) * (size_t)n_stage));
  CK(p.d_cnt.reserve(sizeof(PacketCount) * (size_t)ns));
  CK(p.h_cnt.reserve(sizeof(PacketCount) * (size_t)ns));
  PacketSub * d_sub = p.d_subs.as<PacketSub>();
  PacketStream * d_st = p.d_streams.as<PacketStream>();
  CK(cudaMemcpyAsync(d_sub, p.subs.data(), sizeof(PacketSub) * (size_t)nsub, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_st, p.streams.data(), sizeof(PacketStream) * (size_t)ns, cudaMemcpyHostToDevice, s));
  CK(launch_packet_scan(s, d_sub, nsub, n_frames, p.d_slots.as<PacketSlot>(), &ctx->launches));
  CK(launch_packet_walk(s, d_sub, d_st, ns, p.d_slots.as<PacketSlot>(), p.d_stage.as<PacketStage>(), p.d_cnt.as<PacketCount>(), &ctx->launches));
  CK(cudaMemcpyAsync(p.h_cnt.p, p.d_cnt.p, sizeof(PacketCount) * (size_t)ns, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  const PacketCount * cnt = p.h_cnt.as<PacketCount>();
  long long n_rec = 0, n_bytes = 0;
  for (int i = 0; i < ns; i++)
  {
    PacketStream & st = p.streams[(size_t)i];
    p.n_out[(size_t)i] = cnt[i];
    st.out_rec0 = n_rec;
    st.out_pay0 = n_bytes;
    n_rec += cnt[i].groups;
    n_bytes += cnt[i].bytes;
  }
  const size_t rec_bytes = sizeof(DgRec) * (size_t)n_rec, out_bytes = rec_bytes + (size_t)n_bytes;
  CK(p.d_out.reserve(out_bytes));
  CK(p.h_out.reserve(out_bytes));
  CK(cudaMemcpyAsync(d_st, p.streams.data(), sizeof(PacketStream) * (size_t)ns, cudaMemcpyHostToDevice, s));
  CK(launch_packet_compact(s, d_sub, d_st, ns, n_rec, p.d_slots.as<PacketSlot>(), p.d_stage.as<PacketStage>(), p.d_out.as<DgRec>(), p.d_out.as<uint8_t>() + rec_bytes,
                           &ctx->launches));
  if (out_bytes > 0) CK(cudaMemcpyAsync(p.h_out.p, p.d_out.p, out_bytes, cudaMemcpyDeviceToHost, s));
  p.rec = p.h_out.as<DgRec>();
  p.payload = p.h_out.as<uint8_t>() + rec_bytes;
  CK(cudaEventRecord(p.ev1, s));
  CK(cudaStreamSynchronize(s));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, p.ev0, p.ev1));
  p.ms = ms;
  return 0;
}

int run_packet_fec(dabstar_ctx * ctx, cudaStream_t s, PfecPass & p)
{
  if (!p.ev0) { CK(cudaEventCreate(&p.ev0)); CK(cudaEventCreate(&p.ev1)); }
  const int ns = (int)p.streams.size();
  long long n_slots = 0, n_stage = 0;
  for (PfecStream & st : p.streams)
  {
    st.slot0 = n_slots;
    st.stage0 = n_stage;
    const long long n = (long long)st.n_frames * (st.bit_rate / 8);
    n_slots += n;
    n_stage += n / 2 + 1; // two run starts are at least two slots apart
  }
  p.n_out.assign((size_t)ns, 0);
  p.slots = n_slots;
  p.ms = 0;
  p.rec = nullptr;
  p.mask = nullptr;
  if (n_slots == 0) return 0;
  CK(cudaEventRecord(p.ev0, s));
  if (p.tables.empty())
  {
    pfec_host_tables(p.tables);
    CK(p.d_tab.reserve(p.tables.size()));
    CK(cudaMemcpyAsync(p.d_tab.p, p.tables.data(), p.tables.size(), cudaMemcpyHostToDevice, s));
  }
  // one copy of the span of every stream's bytes (they lie in one allocation); the corrections go into it
  const uint8_t * lo = p.streams[0].src, * hi = lo;
  for (const PfecStream & st : p.streams)
  {
    lo = std::min(lo, st.src);
    hi = std::max(hi, st.src + (size_t)st.n_frames * 3 * st.bit_rate);
  }
  CK(p.d_streams.reserve(sizeof(PfecStream) * (size_t)ns));
  CK(p.d_copy.reserve((size_t)(hi - lo)));
  CK(p.d_code.reserve((size_t)n_slots));
  CK(p.d_start.reserve((size_t)n_slots));
  CK(p.d_mask.reserve((size_t)n_slots));
  CK(p.d_stage.reserve(sizeof(PfecStage) * (size_t)n_stage));
  CK(p.d_cnt.reserve(sizeof(int) * (size_t)ns));
  CK(p.h_cnt.reserve(sizeof(int) * (size_t)ns));
  CK(cudaMemcpyAsync(p.d_copy.p, lo, (size_t)(hi - lo), cudaMemcpyDeviceToDevice, s));
  for (PfecStream & st : p.streams) st.dst = p.d_copy.as<uint8_t>() + (st.src - lo);
  PfecStream * d_st = p.d_streams.as<PfecStream>();
  CK(cudaMemcpyAsync(d_st, p.streams.data(), sizeof(PfecStream) * (size_t)ns, cudaMemcpyHostToDevice, s));
  CK(cudaMemsetAsync(p.d_mask.p, 0, (size_t)n_slots, s));
  CK(launch_pfec_locate(s, d_st, ns, n_slots, p.d_code.as<uint8_t>(), p.d_start.as<uint8_t>(), &ctx->launches));
  CK(launch_pfec_list(s, d_st, ns, p.d_code.as<uint8_t>(), p.d_start.as<uint8_t>(), p.d_stage.as<PfecStage>(), p.d_cnt.as<int>(), p.d_mask.as<uint8_t>(),
                      &ctx->launches));
  CK(cudaMemcpyAsync(p.h_cnt.p, p.d_cnt.p, sizeof(int) * (size_t)ns, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  long long n_rec = 0;
  for (int i = 0; i < ns; i++)
  {
    p.n_out[(size_t)i] = p.h_cnt.as<int>()[i];
    p.streams[(size_t)i].out0 = n_rec;
    n_rec += p.n_out[(size_t)i];
  }
  CK(p.d_rec.reserve(sizeof(PfecRec) * (size_t)std::max(n_rec, 1LL)));
  CK(p.h_rec.reserve(sizeof(PfecRec) * (size_t)std::max(n_rec, 1LL)));
  CK(cudaMemcpyAsync(d_st, p.streams.data(), sizeof(PfecStream) * (size_t)ns, cudaMemcpyHostToDevice, s));
  CK(launch_pfec_correct(s, d_st, ns, n_rec, p.d_tab.p, p.d_stage.as<PfecStage>(), p.d_rec.as<PfecRec>(), &ctx->launches));
  if (n_rec > 0) CK(cudaMemcpyAsync(p.h_rec.p, p.d_rec.p, sizeof(PfecRec) * (size_t)n_rec, cudaMemcpyDeviceToHost, s));
  p.rec = p.h_rec.as<PfecRec>();
  p.mask = p.d_mask.as<uint8_t>();
  CK(cudaEventRecord(p.ev1, s));
  CK(cudaStreamSynchronize(s));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, p.ev0, p.ev1));
  p.ms = ms;
  return 0;
}

// The packed frames of a stage tap in ctx->scratch[1], and the FEC pass run on them when fec is set
static int packet_tap_in(dabstar_ctx * ctx, const uint8_t * frame_bits, int bit_rate, int n_frames, int mem, bool fec)
{
  CK(cudaSetDevice(ctx->device));
  const size_t n_bits = (size_t)n_frames * 24 * bit_rate;
  const void * dbits;
  if (int r = stage_in(ctx, ctx->scratch[0], frame_bits, n_bits, mem, &dbits)) return r;
  CK(ctx->scratch[1].reserve(n_bits / 8)); // packed frames
  CK(launch_pack_bits(ctx->stream, (const uint8_t *)dbits, ctx->scratch[1].as<uint8_t>(), (long long)(n_bits / 8), &ctx->launches));
  if (!fec) return 0;
  PfecPass & f = ctx->pfec;
  f.streams.assign(1, PfecStream{ ctx->scratch[1].as<uint8_t>(), nullptr, bit_rate, n_frames, 0, 0, 0 });
  return run_packet_fec(ctx, ctx->stream, f);
}

static int packet_groups_tap(dabstar_ctx * ctx, const uint8_t * frame_bits, int bit_rate, int n_frames, int address, int dg_flag, dabstar_data_group * out, int cap,
                             uint8_t * payload, int mem, bool fec)
{
  if (!ctx || (!frame_bits && n_frames > 0) || n_frames < 0 || cap < 0 || (cap > 0 && !out)) return DABSTAR_E_INVALID;
  if (bit_rate < 8 || bit_rate % 8) return ctx->fail(DABSTAR_E_INVALID, "packet mode: bit rate %d is not a multiple of 8", bit_rate);
  if (address < 1 || address > 1023) return ctx->fail(DABSTAR_E_INVALID, "packet mode: address %d is not 1..1023", address);
  if (n_frames == 0) return 0;
  if (int r = packet_tap_in(ctx, frame_bits, bit_rate, n_frames, mem, fec)) return r;
  PacketPass & p = ctx->packet;
  if (fec) p.subs.assign(1, PacketSub{ ctx->pfec.streams[0].dst, bit_rate, n_frames, 0, 0, ctx->pfec.mask });
  else p.subs.assign(1, PacketSub{ ctx->scratch[1].as<uint8_t>(), bit_rate, n_frames, 0, 0 });
  p.streams.assign(1, PacketStream{ 0, address, dg_flag ? 1 : 0, 0, 0, 0 });
  if (int r = run_packet(ctx, ctx->stream, p)) return r;
  ctx->arena_off = 0;
  const int n_out = (int)p.n_out[0].groups, n_copy = std::min(n_out, cap);
  size_t bytes = 0;
  for (int i = 0; i < n_copy; i++)
  {
    out[i] = data_group_public(p.rec[i]);
    bytes += (size_t)p.rec[i].length;
  }
  if (payload && bytes > 0)
  {
    if (mem == DABSTAR_MEM_HOST) memcpy(payload, p.payload, bytes);
    else CK(cudaMemcpy(payload, p.payload, bytes, cudaMemcpyHostToDevice));
  }
  return n_out;
}

extern "C" int dabstar_packet_groups(dabstar_ctx * ctx, const uint8_t * frame_bits, int bit_rate, int n_frames, int address, int dg_flag, dabstar_data_group * out,
                                     int cap, uint8_t * payload, int mem)
{
  return packet_groups_tap(ctx, frame_bits, bit_rate, n_frames, address, dg_flag, out, cap, payload, mem, false);
}

extern "C" int dabstar_packet_groups_fec(dabstar_ctx * ctx, const uint8_t * frame_bits, int bit_rate, int n_frames, int address, int dg_flag,
                                         dabstar_data_group * out, int cap, uint8_t * payload, dabstar_packet_stats * stats, dabstar_fec_frame * fec_out,
                                         int fec_cap, int * n_fec, int mem)
{
  if (!ctx || fec_cap < 0 || (fec_cap > 0 && !fec_out)) return DABSTAR_E_INVALID;
  const int n = packet_groups_tap(ctx, frame_bits, bit_rate, n_frames, address, dg_flag, out, cap, payload, mem, n_frames > 0);
  if (n < 0) return n;
  const bool ran = n_frames > 0;
  const int nf = ran ? ctx->pfec.n_out[0] : 0;
  for (int i = 0; i < nf && i < fec_cap; i++) fec_out[i] = fec_frame_public(ctx->pfec.rec[i]);
  if (n_fec) *n_fec = nf;
  if (stats)
  {
    const PacketPass & p = ctx->packet;
    *stats = ran && !p.n_out.empty() ? packet_stats_public(p.n_out[0], p.rec, p.n_out[0].groups) : dabstar_packet_stats{};
  }
  return n;
}

extern "C" int dabstar_packet_fec(dabstar_ctx * ctx, const uint8_t * frame_bits, int bit_rate, int n_frames, uint8_t * corrected_bits, dabstar_fec_frame * out,
                                  int cap, int mem)
{
  if (!ctx || (!frame_bits && n_frames > 0) || n_frames < 0 || cap < 0 || (cap > 0 && !out)) return DABSTAR_E_INVALID;
  if (bit_rate < 8 || bit_rate % 8) return ctx->fail(DABSTAR_E_INVALID, "packet mode: bit rate %d is not a multiple of 8", bit_rate);
  if (n_frames == 0) return 0;
  if (int r = packet_tap_in(ctx, frame_bits, bit_rate, n_frames, mem, true)) return r;
  ctx->arena_off = 0;
  const PfecPass & f = ctx->pfec;
  const int n_out = f.n_out[0];
  for (int i = 0; i < n_out && i < cap; i++) out[i] = fec_frame_public(f.rec[i]);
  if (corrected_bits)
  {
    const size_t n_bytes = (size_t)n_frames * 3 * bit_rate;
    std::vector<uint8_t> packed(n_bytes), bits(n_bytes * 8);
    CK(cudaMemcpyAsync(packed.data(), f.streams[0].dst, n_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < n_bytes; i++)
      for (int b = 0; b < 8; b++) bits[8 * i + b] = (uint8_t)((packed[i] >> (7 - b)) & 1u);
    if (mem == DABSTAR_MEM_HOST) memcpy(corrected_bits, bits.data(), bits.size());
    else CK(cudaMemcpy(corrected_bits, bits.data(), bits.size(), cudaMemcpyHostToDevice));
  }
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
int reserve_viterbi_ws(dabstar_ctx * ctx, int n_jobs, int max_steps)
{
  // 6 GiB of the 180 GB: about 125 000 of the longest MSC code words (3078 steps x 16 B) per launch, i.e. four warps per scheduler
  // (the kernel's register limit); a 1.5 GiB cap left a launch at 1.7 warps per scheduler (ncu: 33 % of the stall samples on loads)
  const size_t cap = (size_t)6 << 30;
  CK(ctx->vit_ws.reserve(std::min(viterbi_ws_bytes(n_jobs, max_steps), cap)));
  return 0;
}

int run_viterbi_jobs(dabstar_ctx * ctx, const std::vector<VitJob> & jobs, int max_steps, const int16_t * d_soft, uint8_t * d_bits,
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
  void * dbits;
  const size_t out_bytes = (size_t)n_out * p.n_bits;
  if (int r = stage_out_begin(ctx, ctx->scratch[1], bits, out_bytes, mem, &dbits)) return r;
  // the job list is written on the device, as the decoder's: one Backend that sees every CIF, emitting from its 17th
  if (int r = sync_profiles(ctx)) return r;
  const BackendJobRange range{ 0, 0, prof, p.n_bits, 0, 16, n_out, sc->start_cu * 64, 0, 0 };
  CK(ctx->scratch[2].reserve(sizeof(VitJob) * (size_t)n_out));
  CK(ctx->scratch[3].reserve(sizeof(range)));
  UP(ctx->scratch[3].p, &range, sizeof(range));
  CK(launch_expand_backend_jobs(ctx->stream, ctx->scratch[3].as<BackendJobRange>(), 1, ctx->scratch[2].as<VitJob>(), &ctx->launches));
  if (int r = reserve_viterbi_ws(ctx, n_out, p.n_bits + 6)) return r;
  CK(launch_viterbi(ctx->stream, ctx->scratch[2].as<VitJob>(), nullptr, n_out, ctx->d_profiles.as<VitProfile>(), p.n_bits + 6, dsoft, (uint8_t *)dbits,
                    ctx->tab.prbs, nullptr, nullptr, ctx->d_step_tab.as<unsigned>(), ctx->vit_ws.p, ctx->vit_ws.cap, &ctx->launches));
  if (int r = stage_out_end(ctx, dbits, bits, out_bytes, mem)) return r;
  return n_out;
}

struct dabstar_ofdm_state
{
  OfdmStateDev * dev = nullptr;
};

int ofdm_state_init(dabstar_ctx * ctx, OfdmStateDev * dev, bool full, int count)
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
void quality_from_sums(const FrameQual & q, float sigma_sq_freq_corr, float out[6])
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
int quality_from_state(dabstar_ctx * ctx, const OfdmStateDev * dev, float sigma_sq_freq_corr, float out[6])
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
  // window i = samples [2048 i, 2048 i + 2048) of recording 0; every other field is zero, so there is no oscillator
  // (f_sym0 = ph_eval = 0) and the decoder's kernel correlates the samples as given
  std::vector<FrameDesc> fd((size_t)n);
  for (int i = 0; i < n; i++) fd[i].eval = (long long)i * T_U;
  FrameDesc * dfd; RecInput * drin;
  if (int r = upload_frames(ctx, fd, { RecInput{ din, (long long)T_U * n } }, &dfd, &drin)) return r;
  CK(launch_prs_corr(ctx->stream, ctx->tab, dfd, n, drin, FMT_CF32, threshold, threshold, nullptr, strongest_peak, (int *)dout, &ctx->launches));
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
  FrameDesc * dfd; RecInput * drin;
  if (int r = upload_frames(ctx, fd, { RecInput{ din, per * n } }, &dfd, &drin)) return r;
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
    FrameDesc * dfd; RecInput * drin;
    if (int r = upload_frames(ctx, fd, rin, &dfd, &drin)) return r;
    CK(launch_fft_frames(ctx->stream, ctx->tab, dfd, n_frames, drin, fmt, (float2 *)dX, max_ctas_per_sm, &ctx->launches));
    if (dnull)
    {
      CK(launch_fft_null(ctx->stream, ctx->tab, dfd, n_frames, drin, fmt, (float2 *)dnull, &ctx->launches));
      if (mem == DABSTAR_MEM_HOST) CK(cudaMemcpyAsync(null_fft, dnull, null_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
  }
  return stage_out_end(ctx, dX, X, x_bytes, mem);
}
