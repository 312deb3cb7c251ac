// ofdm_kernels.cu — ingest, synchronisation, FFT and DQPSK demapping kernels for sm_100a.
//
// Reference rows (SURVEY.md section 8a): I1/I2 sample conversion and integer-Hz derotation
// (devices/filereaders/raw_files/raw_reader.cpp:66-70, ofdm/sample_reader.cpp:212-282), S1 TimeSyncer
// (ofdm/timesyncer.cpp:40-90), S2/S3 PhaseReference (ofdm/phasereference.cpp:87-280), F1 the FFTW plan
// (main/dab_processor.cpp:63), F2 cyclic-prefix correlation (main/dab_processor.cpp:317-333), D0-D3
// FreqInterleaver + OfdmDecoder (ofdm/ofdm_decoder.cpp:114-355).
#include "fft2048.cuh"
#include "kernels.h"
#include "devcache.h"

#include <algorithm>
#include <cstdlib>
#include <type_traits>

namespace dab
{
namespace
{
// ------------------------------------------------------------------------------------------------ ingest
// Raw IQ pair as stored in the recording. u8: (v - 127.38)/128 (raw_reader.cpp:66-70); i16: v/32768 (xml_reader.cpp:254-372).
// A u8 pair stays ONE 16-bit register value until it is converted (a uchar2 would be split into two byte registers
// right after the load); conversion = two I2F with byte / half-word selectors + one packed FFMA2:
// (v - 127.38) / 128 = fma(v, 2^-7, -127.38 * 2^-7) bit for bit (scaling by a power of two commutes with the rounding).
template <int FMT> struct Raw;
template <> struct Raw<FMT_U8> { typedef unsigned short type; typedef unsigned reg; };  // reg: how a loaded sample is held in registers
template <> struct Raw<FMT_I16> { typedef short2 type; typedef short2 reg; };
template <> struct Raw<FMT_CF32> { typedef float2 type; typedef float2 reg; };

__device__ __forceinline__ float2 to_cf(unsigned v)
{
  // byte -> float without the quarter-rate I2F: 0x4B0000bb is 2^23 + b exactly; subtracting 2^23 is exact
  const float2 m = make_float2(__uint_as_float(__byte_perm(v, 0x4B000000u, 0x7540)), __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7541)));
  const float2 f = __fadd2_rn(m, make_float2(-8388608.0f, -8388608.0f));
  return __ffma2_rn(f, make_float2(1.0f / 128.0f, 1.0f / 128.0f), make_float2(-127.38f / 128.0f, -127.38f / 128.0f));
}
__device__ __forceinline__ float2 to_cf(short2 v) { return __fmul2_rn(make_float2((float)v.x, (float)v.y), make_float2(1.0f / 32768.0f, 1.0f / 32768.0f)); }
__device__ __forceinline__ float2 to_cf(float2 v) { return v; }

template <int FMT> __device__ __forceinline__ float2 load_sample(const void * __restrict__ iq, long long i)
{
  return to_cf((typename Raw<FMT>::reg)reinterpret_cast<const typename Raw<FMT>::type *>(iq)[i]);
}

__device__ __forceinline__ unsigned smem_addr_u32(const void * p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(unsigned dst, const void * src) { asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ int mod_fs(long long x)
{
  int r = (int)(x % FS);
  return r < 0 ? r + FS : r;
}

// e^{j 2 pi idx / FS}, the reference's oscillator table entry (sample_reader.cpp:44-50), without the 16 MB table:
// exact integer reduction to a quadrant, float sincos of an angle in [0, pi/2) (|phase error| < 2e-7 rad), exact
// quadrant rotation.
__device__ __forceinline__ float2 osc(int idx)
{
  const int q = idx / (FS / 4), rem = idx - q * (FS / 4);
  float s, c;
  sincosf((float)rem * (PI_2_F / (float)(FS / 4)), &s, &c);
  switch (q)
  {
  case 0: return make_float2(c, s);
  case 1: return make_float2(-s, c);
  case 2: return make_float2(-c, -s);
  default: return make_float2(s, -c);
  }
}

// Fetches the 2048 raw samples starting at `start` in the FFT's register layout (r[n1] = x[128 n1 + tid]).
template <int FMT>
__device__ __forceinline__ void fetch_symbol(typename Raw<FMT>::reg (&r)[16], const void * __restrict__ iq, long long n_total, long long start, int tid)
{
  typedef typename Raw<FMT>::type T;
  const T * p = reinterpret_cast<const T *>(iq) + start + tid;
  if (start >= 0 && start + T_U <= n_total)
  {
#pragma unroll
    for (int n1 = 0; n1 < 16; n1++) r[n1] = p[128 * n1];
  }
  else
  {
#pragma unroll
    for (int n1 = 0; n1 < 16; n1++)
    {
      const long long i = start + 128 * n1 + tid;
      if (i >= 0 && i < n_total) r[n1] = p[128 * n1];
      else r[n1] = typename Raw<FMT>::reg(); // outside the recording; mix_symbol replaces it by a zero amplitude
    }
  }
}

// Converts the fetched samples and mixes them with the integer-Hz oscillator. `ph` is the oscillator phase BEFORE
// sample `start`. step[] is a 16-entry shared scratch (phasor of -f*128*n1). Samples outside the recording are zero.
template <int FMT>
__device__ __forceinline__ void mix_symbol(float2 (&v)[16], const typename Raw<FMT>::reg (&r)[16], long long n_total, long long start, int f, int ph,
                                           float2 * step, int tid)
{
  const bool inside = start >= 0 && start + T_U <= n_total;
#pragma unroll
  for (int n1 = 0; n1 < 16; n1++)
  {
    v[n1] = to_cf(r[n1]);
    if (!inside) { const long long i = start + 128 * n1 + tid; if (i < 0 || i >= n_total) v[n1] = make_float2(0.0f, 0.0f); }
  }
  if (f == 0 && ph == 0) return; // osc[0] = 1: the reference multiplies by exactly (1, 0)
  if (tid < 16) step[tid] = osc(mod_fs(-(long long)f * 128 * tid));
  __syncthreads();
  const float2 s0 = osc(mod_fs((long long)ph - (long long)f * (tid + 1)));
#pragma unroll
  for (int n1 = 0; n1 < 16; n1++) v[n1] = cmul(v[n1], n1 == 0 ? s0 : cmul(s0, step[n1]));
  __syncthreads();
}

template <int FMT>
__device__ __forceinline__ void load_symbol(float2 (&v)[16], const void * __restrict__ iq, long long n_total, long long start, int f, int ph,
                                            float2 * step, int tid)
{
  typename Raw<FMT>::reg r[16];
  fetch_symbol<FMT>(r, iq, n_total, start, tid);
  mix_symbol<FMT>(v, r, n_total, start, f, ph, step, tid);
}

// ------------------------------------------------------------------------------------------------ FFT of whole frames
// Work item = (frame, row): row 0 = symbol 0, rows 1..75 data symbols, row 76 the null symbol.
// Output: X[xslot][row][k] = spectrum at the bin of nominal carrier k (frequency de-interleaving fused into the store).
struct SymbolItem
{
  const void * iq;
  long long n_total, start;
  int f, ph;
  long long out; // float2 index of X row, -1: nothing to do
};

__device__ __forceinline__ SymbolItem symbol_item(const FrameDesc & fd, const RecInput & rin, int row)
{
  SymbolItem it;
  it.iq = rin.iq;
  it.n_total = rin.n;
  it.out = ((long long)fd.xslot * X_ROWS + row) * K_CARR;
  if (row == 0) { it.start = fd.sym0; it.f = fd.f_sym0; it.ph = mod_fs((long long)fd.ph_eval - (long long)it.f * (fd.sym0 - fd.eval)); }
  else if (row <= 75)
  {
    it.start = fd.sym0 + T_U + (long long)(row - 1) * T_S + T_G;
    it.f = fd.f_data;
    it.ph = mod_fs((long long)fd.ph_data - (long long)it.f * ((long long)(row - 1) * T_S + T_G));
    if (row > fd.n_syms) it.out = -1;
  }
  else
  {
    it.start = fd.sym0 + T_U + 75LL * T_S + T_G;
    it.f = fd.f_null;
    it.ph = mod_fs((long long)fd.ph_null - (long long)it.f * T_G);
    if (fd.n_syms < 75) it.out = -1;
  }
  return it;
}

// Raw samples reach the CTA through a double-buffered stage in shared memory filled by the TMA engine: ONE thread issues one
// bulk copy (cp.async.bulk, UBLKCP in SASS) of the 16-byte aligned superset of the next symbol's samples before the current
// symbol is transformed, completion is signalled on an mbarrier the consumers wait on (no per-thread LDGSTS, whose 16-byte
// shared-memory writes ran at 2.8x their ideal wavefronts, and no CTA barrier for the hand-over). Symbols within 8 samples of
// either end of a recording (where the aligned superset could leave the buffer) take the bounds-checked path.
template <int FMT> __host__ __device__ constexpr int fft_stage_bytes() { return T_U * (int)sizeof(typename Raw<FMT>::type) + 16; }

__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void * src, unsigned bytes, unsigned bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity)
{
  unsigned ok;
  do
  {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  } while (!ok);
}

template <int FMT>
__device__ __forceinline__ bool item_async(const SymbolItem & it) { return it.out >= 0 && it.start >= 8 && it.start + T_U + 8 <= it.n_total; }

// 32-bit (x mod FS) for |x| < 2^31
__device__ __forceinline__ int mod_fs32(int x)
{
  const int r = x % FS;
  return r < 0 ? r + FS : r;
}

// The 16 converted samples of a thread times the integer-Hz oscillator (sample_reader.cpp:276-281). f == 0 leaves ONE phasor
// for the whole symbol (the oscillator stands at `ph`); otherwise sample 128 n1 + tid takes osc[ph - f (128 n1 + tid + 1)] =
// s0(tid) * step[n1], step = phasors of -128 f n1 (shared, recomputed by the caller only when f changes).
template <int FMT>
__device__ __forceinline__ void convert_mix(float2 (&v)[16], const typename Raw<FMT>::reg (&r)[16], int f, int ph, const float2 * step, int tid)
{
#pragma unroll
  for (int n1 = 0; n1 < 16; n1++) v[n1] = to_cf(r[n1]);
  if (f == 0)
  {
    if (ph == 0) return; // osc[0] = 1: the reference multiplies by exactly (1, 0)
    const float2 c = step[0]; // osc(ph), filed by the caller when the phase changed (it stands still while f = 0)
#pragma unroll
    for (int n1 = 0; n1 < 16; n1++) v[n1] = cmul(v[n1], c);
    return;
  }
  const float2 s0 = osc(mod_fs32(ph - f * (tid + 1)));
#pragma unroll
  for (int n1 = 0; n1 < 16; n1++) v[n1] = cmul(v[n1], n1 == 0 ? s0 : cmul(s0, step[n1]));
}

template <int FMT>
__global__ void __launch_bounds__(FFT_THREADS, 5) k_fft_frames(const FrameDesc * __restrict__ frames, int n_items, const RecInput * __restrict__ recs,
                                                               const float2 * __restrict__ w2048, const uint16_t * __restrict__ slot_w,
                                                               const uint16_t * __restrict__ slot_r, float2 * __restrict__ X)
{
  typedef typename Raw<FMT>::type T;
  extern __shared__ __align__(16) unsigned char fft_stage[]; // 2 x fft_stage_bytes<FMT>()
  __shared__ __align__(16) float2 smem[FFT_SMEM_F2];
  __shared__ float2 tw2s[FFT_TW2_F2];
  __shared__ float2 step[16];
  __shared__ unsigned short pos[16 * FFT_THREADS]; // byte offset in `smem` of the staging slot of output i = 8 h + j2 of every thread
  __shared__ unsigned rpos[K_CARR / 2];            // byte offsets of the slots of carriers 2p (low half) and 2p + 1 (high half)
  __shared__ __align__(8) unsigned long long mbar[2];
  const int tid = threadIdx.x;
  FftTwiddles tw;
  fft_load_twiddles(tw, w2048, tw2s, tid);
  // Epilogue layout (tables.cu, host_fft_epilogue_layout): after stage 3 a thread holds the bins fft_out_index(tid, h, j2); each
  // goes straight to the staging slot of its nominal carrier (frequency de-interleaving, freq_interleaver.cpp), and a row of the
  // demapper's layout (carriers 2p, 2p + 1 as re, re, im, im) is two 8-byte reads per pair. The slots are chosen so that the
  // scatter stores AND the gather loads are free of bank conflicts; bins that carry no carrier (DC, guard band) go to slots
  // nobody reads.
#pragma unroll
  for (int i = 0; i < 16; i++) pos[i * FFT_THREADS + tid] = (unsigned short)(slot_w[i * FFT_THREADS + tid] * (int)sizeof(float2));
  for (int p = tid; p < K_CARR / 2; p += FFT_THREADS)
    rpos[p] = (unsigned)slot_r[2 * p] * (unsigned)sizeof(float2) | ((unsigned)slot_r[2 * p + 1] * (unsigned)sizeof(float2)) << 16;
  static_assert(2048 <= FFT_SMEM_F2, "the staging slots (16 per write group) must fit the transform buffer");
  const unsigned stage0 = smem_addr_u32(fft_stage);
  const unsigned bar0 = smem_addr_u32(mbar);
  constexpr int SB = fft_stage_bytes<FMT>();
  if (tid == 0)
  {
    mbar_init(bar0, 1);
    mbar_init(bar0 + 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  // A CTA walks a contiguous range of (frame, row) items: the frame descriptor is fetched once per 77 symbols and the items of
  // the data symbols follow from their predecessor (start + T_s, oscillator phase - f T_s) instead of 64-bit products and
  // remainders per symbol.
  const int per = n_items / (int)gridDim.x, rem = n_items - per * (int)gridDim.x;
  int item = (int)blockIdx.x * per + min((int)blockIdx.x, rem);
  const int item_end = item + per + ((int)blockIdx.x < rem ? 1 : 0);
  int buf = 0, fi = item / X_ROWS, row = item - fi * X_ROWS;
  unsigned phase_bits = 0; // bit b: parity the next wait on mbar[b] expects
  FrameDesc fd;
  RecInput rin;
  SymbolItem cur;
  cur.out = -1;
  int dph = 0;        // oscillator phase step of one data symbol: -f_data T_s mod FS
  int step_f = 0;     // integer Hz the shared step table holds (0: none)
  int step_ph = -1;   // f = 0: oscillator phase whose phasor step[0] holds (-1: none)
  auto issue = [&](const SymbolItem & it, int b) {
    if (tid == 0)
    {
      const unsigned long long a = (unsigned long long)(reinterpret_cast<const T *>(it.iq) + it.start);
      mbar_expect_tx(bar0 + 8u * (unsigned)b, (unsigned)SB);
      bulk_g2s(stage0 + (unsigned)(b * SB), reinterpret_cast<const void *>(a & ~15ull), (unsigned)SB, bar0 + 8u * (unsigned)b);
    }
  };
  if (item < item_end)
  {
    fd = frames[fi];
    rin = recs[fd.rec];
    cur = symbol_item(fd, rin, row);
    dph = mod_fs32(-(int)(((long long)fd.f_data * T_S) % FS));
    if (item_async<FMT>(cur)) issue(cur, 0);
  }
  while (item < item_end)
  {
    const int next = item + 1;
    SymbolItem nxt;
    nxt.out = -1;
    if (next < item_end)
    {
      if (++row == X_ROWS)
      {
        row = 0;
        fi++;
        fd = frames[fi];
        rin = recs[fd.rec];
        dph = mod_fs32(-(int)(((long long)fd.f_data * T_S) % FS));
      }
      if (row >= 2 && row <= 75)
      {
        // data symbol after a data symbol of the same frame
        nxt.iq = cur.iq;
        nxt.n_total = cur.n_total;
        nxt.start = cur.start + T_S;
        nxt.f = cur.f;
        nxt.ph = cur.ph + dph;
        if (nxt.ph >= FS) nxt.ph -= FS;
        nxt.out = row > fd.n_syms ? -1 : ((long long)fd.xslot * X_ROWS + row) * K_CARR;
      }
      else nxt = symbol_item(fd, rin, row);
      if (item_async<FMT>(nxt)) issue(nxt, buf ^ 1);
    }
    if (cur.out >= 0)
    {
      float2 v[16];
      if (cur.f != 0 ? cur.f != step_f : (cur.ph != 0 && cur.ph != step_ph))
      {
        // (all threads agree on cur.f / cur.ph: no divergence around the barriers)
        __syncthreads(); // nobody reads the previous table any more
        if (cur.f != 0)
        {
          if (tid < 16) step[tid] = osc(mod_fs32(-(int)(((long long)cur.f * 128 * tid) % FS)));
          step_f = cur.f;
          step_ph = -1;
        }
        else
        {
          if (tid == 0) step[0] = osc(cur.ph);
          step_ph = cur.ph;
          step_f = 0;
        }
        __syncthreads();
      }
      if (item_async<FMT>(cur))
      {
        mbar_wait(bar0 + 8u * (unsigned)buf, (phase_bits >> buf) & 1u); // the bulk copy of this symbol has landed (visible to every waiter)
        phase_bits ^= 1u << buf;
        const unsigned off = (unsigned)((unsigned long long)(reinterpret_cast<const T *>(cur.iq) + cur.start) & 15ull);
        const T * sp = reinterpret_cast<const T *>(fft_stage + buf * SB + off) + tid;
        typename Raw<FMT>::reg r[16];
#pragma unroll
        for (int n1 = 0; n1 < 16; n1++) r[n1] = sp[128 * n1];
        convert_mix<FMT>(v, r, cur.f, cur.ph, step, tid);
      }
      else
      {
        typename Raw<FMT>::reg r[16];
        fetch_symbol<FMT>(r, cur.iq, cur.n_total, cur.start, tid);
        convert_mix<FMT>(v, r, cur.f, cur.ph, step, tid);
        if (!(cur.start >= 0 && cur.start + T_U <= cur.n_total))
        {
#pragma unroll
          for (int n1 = 0; n1 < 16; n1++)
          {
            const long long i = cur.start + 128 * n1 + tid;
            if (i < 0 || i >= cur.n_total) v[n1] = make_float2(0.0f, 0.0f); // outside the recording: zero amplitude
          }
        }
      }
      fft_stage1(v, tw, smem, tid);
      __syncthreads();
      fft_stage2_read(v, smem, tid);
      __syncthreads();
      fft_stage2(v, tw, smem, tid);
      __syncthreads();
      fft_stage3(v, smem, tid);
      __syncthreads();
      unsigned char * sbase = reinterpret_cast<unsigned char *>(smem);
#pragma unroll
      for (int i = 0; i < 16; i++) *reinterpret_cast<float2 *>(sbase + pos[i * FFT_THREADS + tid]) = v[i];
      __syncthreads();
      float4 * out = reinterpret_cast<float4 *>(X + cur.out);
#pragma unroll
      for (int i = 0; i < K_CARR / 2 / FFT_THREADS; i++)
      {
        const int p = tid + FFT_THREADS * i;
        const unsigned rp = rpos[p];
        const float2 a = *reinterpret_cast<const float2 *>(sbase + (rp & 0xffffu)), b = *reinterpret_cast<const float2 *>(sbase + (rp >> 16));
        out[p] = make_float4(a.x, b.x, a.y, b.y);
      }
    }
    __syncthreads(); // smem and the stage buffer of this symbol are free again
    cur = nxt;
    item = next;
    buf ^= 1;
  }
}

// Natural-order batch transform (stage tap dabstar_fft2048). sign > 0: conj in, conj out.
__global__ void __launch_bounds__(FFT_THREADS, 4) k_fft_batch(const float2 * __restrict__ in, float2 * __restrict__ out, int n, int sign,
                                                              const float2 * __restrict__ w2048)
{
  __shared__ float2 smem[FFT_SMEM_F2];
  __shared__ float2 tw2s[FFT_TW2_F2];
  const int tid = threadIdx.x;
  FftTwiddles tw;
  fft_load_twiddles(tw, w2048, tw2s, tid);
  __syncthreads();
  for (int item = blockIdx.x; item < n; item += gridDim.x)
  {
    float2 v[16];
#pragma unroll
    for (int n1 = 0; n1 < 16; n1++)
    {
      v[n1] = in[(size_t)item * T_U + 128 * n1 + tid];
      if (sign > 0) v[n1].y = -v[n1].y;
    }
    fft2048_to_smem(v, tw, smem, tid);
    for (int i = tid; i < T_U; i += FFT_THREADS)
    {
      float2 r = smem[fft_nat(i)];
      if (sign > 0) r.y = -r.y;
      out[(size_t)item * T_U + i] = r;
    }
    __syncthreads();
  }
}

// FFT of the null symbol of every listed frame in fft order (the TII detector's input, dab_processor.cpp:275-276): the same
// samples, derotation and transform as row 76 of k_fft_frames, without the carrier selection.
template <int FMT>
__global__ void __launch_bounds__(FFT_THREADS, 4) k_fft_null(const FrameDesc * __restrict__ frames, int n_frames, const RecInput * __restrict__ recs,
                                                             const float2 * __restrict__ w2048, float2 * __restrict__ out)
{
  __shared__ float2 smem[FFT_SMEM_F2];
  __shared__ float2 step[16];
  __shared__ float2 tw2s[FFT_TW2_F2];
  const int tid = threadIdx.x;
  FftTwiddles tw;
  fft_load_twiddles(tw, w2048, tw2s, tid);
  __syncthreads();
  for (int fi = blockIdx.x; fi < n_frames; fi += gridDim.x)
  {
    const FrameDesc fd = frames[fi];
    const RecInput rin = recs[fd.rec];
    const SymbolItem it = symbol_item(fd, rin, X_ROWS - 1);
    float2 v[16];
    load_symbol<FMT>(v, it.iq, it.n_total, it.start, it.f, it.ph, step, tid);
    if (!(it.start >= 0 && it.start + T_U <= it.n_total))
    {
      // zero AFTER the oscillator, as k_fft_frames does: mixing a zero amplitude can give -0, and then a null symbol that lies
      // past the end of the recording transforms to a row with -0 where row 76 of X has +0
#pragma unroll
      for (int n1 = 0; n1 < 16; n1++)
      {
        const long long i = it.start + 128 * n1 + tid;
        if (i < 0 || i >= it.n_total) v[n1] = make_float2(0.0f, 0.0f);
      }
    }
    fft2048_to_smem(v, tw, smem, tid);
    for (int i = tid; i < T_U; i += FFT_THREADS) out[(size_t)fi * T_U + i] = smem[fft_nat(i)];
    __syncthreads();
  }
}

// Natural-order spectra [frame][77][2048] -> nominal-carrier order [frame][77][1536] in the demapper's pair layout
// (re 2p, re 2p+1, im 2p, im 2p+1) (stage tap for the demapper).
__global__ void k_reorder_frames(const float2 * __restrict__ fft_nat, int n_rows, const int16_t * __restrict__ bin_of_k, float2 * __restrict__ X)
{
  const int row = blockIdx.x;
  if (row >= n_rows) return;
  for (int p = threadIdx.x; p < K_CARR / 2; p += blockDim.x)
  {
    const float2 a = fft_nat[(size_t)row * T_U + bin_of_k[2 * p]], b = fft_nat[(size_t)row * T_U + bin_of_k[2 * p + 1]];
    reinterpret_cast<float4 *>(X + (size_t)row * K_CARR)[p] = make_float4(a.x, b.x, a.y, b.y); // the demapper's pair layout
  }
}

// ------------------------------------------------------------------------------------------------ block reductions
__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------------ PRS correlation (S2)
// samples already in registers (FFT layout). Returns the start index to thread 0's caller through *result.
__device__ void prs_correlate_cta(float2 (&v)[16], const FftTwiddles & tw, const float2 * __restrict__ prs, float threshold, int strongest,
                                  float2 * smem, float * red, int * result, int tid)
{
  fft2048_to_smem(v, tw, smem, tid);
  // |IFFT(X conj(P))| = |FFT(conj(X) P)|
#pragma unroll
  for (int n1 = 0; n1 < 16; n1++)
  {
    const int i = 128 * n1 + tid;
    const float2 x = smem[fft_nat(i)], p = prs[i];
    v[n1] = make_float2(x.x * p.x + x.y * p.y, x.x * p.y - x.y * p.x); // conj(x) * p
  }
  __syncthreads();
  fft2048_to_smem(v, tw, smem, tid);
  float * mag = reinterpret_cast<float *>(smem); // overwrite in place: mag[i] occupies the first half of smem[i]'s slot range
  float part = 0.0f;
  float m[16];
#pragma unroll
  for (int n1 = 0; n1 < 16; n1++)
  {
    const float2 c = smem[fft_nat(128 * n1 + tid)];
    m[n1] = sqrtf(c.x * c.x + c.y * c.y);
    part += m[n1];
  }
  __syncthreads();
#pragma unroll
  for (int n1 = 0; n1 < 16; n1++) mag[128 * n1 + tid] = m[n1];
  part = warp_sum(part);
  if ((tid & 31) == 0) red[tid >> 5] = part;
  if (tid == 0) *result = 0x7fffffff;
  __syncthreads();
  const float mean = (red[0] + red[1] + red[2] + red[3]) / (float)T_U;
  if (mean == 0.0f) { if (tid == 0) *result = -1; __syncthreads(); return; }
  constexpr int lo = T_G - 250, hi = T_G + 500;
  if (!strongest)
  {
    // first index whose level exceeds the threshold and is not topped within the next 9 samples
    // (phasereference.cpp:141-168); the reference's skip-ahead only affects later candidates.
    int best = 0x7fffffff;
    for (int i = lo + tid; i < hi; i += FFT_THREADS)
    {
      const float a = mag[i];
      if (!(a / mean > threshold)) continue;
      bool peak = true;
      for (int j = 1; j < 10 && i + j < hi; j++) if (mag[i + j] > a) { peak = false; break; }
      if (peak) { best = i; break; }
    }
    if (best != 0x7fffffff) atomicMin(result, best);
    __syncthreads();
    if (tid == 0 && *result == 0x7fffffff) *result = -1;
  }
  else if (tid == 0)
  {
    int max_i = -1;
    float max_l = -1000.0f;
    for (int i = lo; i < hi; i++)
    {
      if (!(mag[i] / mean > threshold)) continue;
      bool peak = true;
      for (int j = 1; j < 10 && i + j < hi; j++) if (mag[i + j] > mag[i]) { peak = false; break; }
      if (!peak) continue;
      if (mag[i] > max_l) { max_l = mag[i]; max_i = i; }
      i += 10;
    }
    *result = (max_l / mean < threshold) ? -1 : max_i;
  }
  __syncthreads();
}

template <int FMT>
__global__ void __launch_bounds__(FFT_THREADS, 4) k_prs_corr(const FrameDesc * __restrict__ frames, int n_frames, const RecInput * __restrict__ recs,
                                                             const float2 * __restrict__ w2048, const float2 * __restrict__ prs,
                                                             float thr_first, float thr_rest, const uint8_t * __restrict__ first_flags,
                                                             int strongest, int * __restrict__ start_index)
{
  __shared__ float2 smem[FFT_SMEM_F2];
  __shared__ float2 step[16];
  __shared__ float red[4];
  __shared__ int result;
  const int tid = threadIdx.x;
  __shared__ float2 tw2s[FFT_TW2_F2];
  FftTwiddles tw;
  fft_load_twiddles(tw, w2048, tw2s, tid);
  __syncthreads();
  for (int fi = blockIdx.x; fi < n_frames; fi += gridDim.x)
  {
    const FrameDesc fd = frames[fi];
    const RecInput rin = recs[fd.rec];
    float2 v[16];
    load_symbol<FMT>(v, rin.iq, rin.n, fd.eval, fd.f_sym0, fd.ph_eval, step, tid);
    const float thr = (first_flags != nullptr && first_flags[fi]) ? thr_first : thr_rest;
    prs_correlate_cta(v, tw, prs, thr, strongest, smem, red, &result, tid);
    if (tid == 0) start_index[fi] = result;
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------ coarse AFC (S3)
// smem holds the natural-order spectrum of symbol 0 on entry.
__device__ void coarse_afc_cta(const FftTwiddles & tw, const float2 * __restrict__ ref_arg_conj, float2 * smem, float * magw, int * result, int tid)
{
  float2 v[16];
  // d[i] = conj(X[i]) X[i+1], d[2047] = 0; IFFT(d) = conj(FFT(conj(d)))
#pragma unroll
  for (int n1 = 0; n1 < 16; n1++)
  {
    const int i = 128 * n1 + tid;
    if (i < T_U - 1)
    {
      const float2 a = smem[fft_nat(i)], b = smem[fft_nat(i + 1)];
      const float2 d = make_float2(a.x * b.x + a.y * b.y, a.x * b.y - a.y * b.x);
      v[n1] = make_float2(d.x, -d.y);
    }
    else v[n1] = make_float2(0.0f, 0.0f);
  }
  __syncthreads();
  fft2048_to_smem(v, tw, smem, tid);
#pragma unroll
  for (int n1 = 0; n1 < 16; n1++)
  {
    const int i = 128 * n1 + tid;
    const float2 sv = smem[fft_nat(i)];
    v[n1] = cmul(make_float2(sv.x, -sv.y), ref_arg_conj[i]);
  }
  __syncthreads();
  fft2048_to_smem(v, tw, smem, tid);
  // peak over bins -70..70 (phasereference.cpp:248-279)
  for (int i = tid; i < 143; i += FFT_THREADS)
  {
    const float2 c = smem[fft_nat((T_U + i - 71) & (T_U - 1))];
    magw[i] = sqrtf(c.x * c.x + c.y * c.y); // magw[i] = |bin i-71|, i = 0..142 (one guard bin each side)
  }
  __syncthreads();
  if (tid == 0)
  {
    int index = 100000;
    float mx = 0.0f, avg = 0.0f;
    for (int i = -70; i <= 70; i++)
    {
      const float val = magw[i + 71];
      if (val > mx) { mx = val; index = i; }
      avg += val;
    }
    avg /= 141.0f;
    if (mx < avg * 5.0f) *result = 100000;
    else
    {
      const float p0 = magw[index + 70], p1 = magw[index + 71], p2 = magw[index + 72];
      const float offset = (float)index + (p2 - p0) / (p0 + p1 + p2);
      *result = (int)(offset * 1000.0f);
    }
  }
  __syncthreads();
}

template <int FMT>
__global__ void __launch_bounds__(FFT_THREADS, 4) k_coarse_afc(const FrameDesc * __restrict__ frames, int n_frames, const RecInput * __restrict__ recs,
                                                               const float2 * __restrict__ w2048, const float2 * __restrict__ ref_arg_conj,
                                                               int * __restrict__ offset_hz)
{
  __shared__ float2 smem[FFT_SMEM_F2];
  __shared__ float2 step[16];
  __shared__ float magw[144];
  __shared__ int result;
  const int tid = threadIdx.x;
  __shared__ float2 tw2s[FFT_TW2_F2];
  FftTwiddles tw;
  fft_load_twiddles(tw, w2048, tw2s, tid);
  __syncthreads();
  for (int fi = blockIdx.x; fi < n_frames; fi += gridDim.x)
  {
    const FrameDesc fd = frames[fi];
    const RecInput rin = recs[fd.rec];
    float2 v[16];
    const int ph = mod_fs((long long)fd.ph_eval - (long long)fd.f_sym0 * (fd.sym0 - fd.eval));
    load_symbol<FMT>(v, rin.iq, rin.n, fd.sym0, fd.f_sym0, ph, step, tid);
    fft2048_to_smem(v, tw, smem, tid);
    coarse_afc_cta(tw, ref_arg_conj, smem, magw, &result, tid);
    if (tid == 0) offset_hz[fi] = result;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(FFT_THREADS, 4) k_coarse_afc_raw(const float2 * __restrict__ fft_nat_in, int n, const float2 * __restrict__ w2048,
                                                                   const float2 * __restrict__ ref_arg_conj, int * __restrict__ offset_hz)
{
  __shared__ float2 smem[FFT_SMEM_F2];
  __shared__ float magw[144];
  __shared__ int result;
  const int tid = threadIdx.x;
  __shared__ float2 tw2s[FFT_TW2_F2];
  FftTwiddles tw;
  fft_load_twiddles(tw, w2048, tw2s, tid);
  __syncthreads();
  for (int it = blockIdx.x; it < n; it += gridDim.x)
  {
    for (int i = tid; i < T_U; i += FFT_THREADS) smem[fft_nat(i)] = fft_nat_in[(size_t)it * T_U + i];
    __syncthreads();
    coarse_afc_cta(tw, ref_arg_conj, smem, magw, &result, tid);
    if (tid == 0) offset_hz[it] = result;
    __syncthreads();
  }
}

// ref_arg_conj = conj(IFFT(relative phase of the PRS)) (phasereference.cpp:58-66)
__global__ void __launch_bounds__(FFT_THREADS) k_init_ref_arg(const float2 * __restrict__ w2048, const float2 * __restrict__ prs, float2 * __restrict__ ref_arg_conj)
{
  __shared__ float2 smem[FFT_SMEM_F2];
  const int tid = threadIdx.x;
  __shared__ float2 tw2s[FFT_TW2_F2];
  FftTwiddles tw;
  fft_load_twiddles(tw, w2048, tw2s, tid);
  __syncthreads();
  float2 v[16];
#pragma unroll
  for (int n1 = 0; n1 < 16; n1++)
  {
    const int i = 128 * n1 + tid;
    if (i < T_U - 1)
    {
      const float2 a = prs[i], b = prs[i + 1];
      v[n1] = make_float2(a.x * b.x + a.y * b.y, -(a.x * b.y - a.y * b.x)); // conj(conj(a) b)
    }
    else v[n1] = make_float2(0.0f, 0.0f);
  }
  fft2048_to_smem(v, tw, smem, tid);
  // IFFT(d) = conj(smem); ref_arg_conj = conj(IFFT(d)) = smem
  for (int i = tid; i < T_U; i += FFT_THREADS) ref_arg_conj[i] = smem[fft_nat(i)];
}

// ------------------------------------------------------------------------------------------------ CP correlation (F2)
// cp[frame] = sum over symbols 1..75 and the 504 prefix samples of x[i+2048] conj(x[i]) on the RAW samples. The
// derotated sum the reference forms differs by the constant factor e^{-j 2 pi f / 1000} (f = integer Hz), which the
// host control loop applies.
//
// 8-bit input is summed in INTEGERS: a sample is ((I - c) / 128, (Q - c) / 128) with c = 127.38 (to_cf), so with a = x[i+2048],
// b = x[i] as bytes
//   16384 Re = P1 - c S1 + 2 N c^2,  P1 = sum(aI bI + aQ bQ),  S1 = sum(aI + aQ + bI + bQ),  N = number of products
//   16384 Im = P2 - c S2,            P2 = sum(aQ bI - aI bQ),  S2 = sum(aQ - aI + bI - bQ)
// and the four sums are dot products of byte vectors (IDP.4A): seven of them per TWO samples instead of ~20 instructions per
// sample for the conversion to float and the complex multiply-add, no rounding until the one conversion per frame, and a
// result that does not depend on which lane adds what (the two kernels below and their edge paths agree bit for bit by
// construction). The reference's float sum of the same 37 800 products carries a rounding error of ~1e-5 relative, as did the
// float form of this kernel; the integer form is the exact value of that sum.
struct CpInt
{
  int p1, p2, s1, s2;
};
__device__ __forceinline__ unsigned dp4a_uu(unsigned a, unsigned b, unsigned c)
{
  unsigned d;
  asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ int dp4a_us(unsigned a, unsigned b_signed, int c)
{
  int d;
  asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b_signed), "r"(c));
  return d;
}
// aw: bytes (I, Q, I, Q) of up to two samples of x[i+2048], bw: the same of x[i]; bytes outside the sum must be zero in both
__device__ __forceinline__ void cp_int_add(CpInt & t, unsigned aw, unsigned bw)
{
  t.p1 = (int)dp4a_uu(aw, bw, (unsigned)t.p1);
  const unsigned bs = __byte_perm(bw, 0u, 0x2301); // (Q, I, Q, I)
  t.p2 = (int)dp4a_uu(aw & 0xff00ff00u, bs, (unsigned)t.p2);
  t.p2 -= (int)dp4a_uu(aw & 0x00ff00ffu, bs, 0u);
  t.s1 = (int)dp4a_uu(aw, 0x01010101u, dp4a_uu(bw, 0x01010101u, (unsigned)t.s1));
  t.s2 = dp4a_us(aw, 0x01ff01ffu, dp4a_us(bw, 0xff01ff01u, t.s2)); // weights (-1, +1, -1, +1) and (+1, -1, +1, -1)
}
__device__ __forceinline__ int warp_sum_int(int v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// the per-warp sums of a frame (at most 10 symbols x 504 products: below 2^31) -> cp; thread 0, after a barrier
__device__ __forceinline__ float2 cp_int_finish(const CpInt * red, int n_syms)
{
  long long p1 = 0, p2 = 0, s1 = 0, s2 = 0;
  for (int w = 0; w < 8; w++) { p1 += red[w].p1; p2 += red[w].p2; s1 += red[w].s1; s2 += red[w].s2; }
  const double c = 127.38, n = (double)n_syms * (double)T_G;
  return make_float2((float)(((double)p1 - c * (double)s1 + 2.0 * n * c * c) * (1.0 / 16384.0)), (float)(((double)p2 - c * (double)s2) * (1.0 / 16384.0)));
}

template <int FMT>
__global__ void __launch_bounds__(256) k_cp_corr(const FrameDesc * __restrict__ frames, int n_frames, const RecInput * __restrict__ recs, float2 * __restrict__ cp)
{
  __shared__ float2 red[8];
  __shared__ CpInt redi[8];
  for (int fi = blockIdx.x; fi < n_frames; fi += gridDim.x)
  {
    const FrameDesc fd = frames[fi];
    const RecInput rin = recs[fd.rec];
    const long long base = fd.sym0 + T_U;
    float2 acc = make_float2(0.0f, 0.0f);
    CpInt ti = { 0, 0, 0, 0 };
    // a warp takes every eighth symbol; the 2 x 16 loads of a lane are issued before the first product (a strided loop with one
    // pair of 2-byte loads in flight per thread ran at a third of the HBM rate)
    typedef typename Raw<FMT>::type T;
    const int lane = threadIdx.x & 31;
    for (int sym = threadIdx.x >> 5; sym < fd.n_syms; sym += 8)
    {
      const T * pp = reinterpret_cast<const T *>(rin.iq) + base + (long long)sym * T_S + lane;
      typename Raw<FMT>::reg ra[16], rb[16];
#pragma unroll
      for (int k = 0; k < 16; k++)
      {
        if (lane + 32 * k < T_G) { ra[k] = pp[32 * k + T_U]; rb[k] = pp[32 * k]; }
        else { ra[k] = typename Raw<FMT>::reg(); rb[k] = typename Raw<FMT>::reg(); }
      }
#pragma unroll
      for (int k = 0; k < 16; k++)
      {
        if (lane + 32 * k < T_G)
        {
          if constexpr (FMT == FMT_U8) cp_int_add(ti, ra[k], rb[k]);
          else
          {
            const float2 a = to_cf(ra[k]), b = to_cf(rb[k]);
            acc.x += a.x * b.x + a.y * b.y;
            acc.y += a.y * b.x - a.x * b.y;
          }
        }
      }
    }
    if constexpr (FMT == FMT_U8)
    {
      ti.p1 = warp_sum_int(ti.p1); ti.p2 = warp_sum_int(ti.p2); ti.s1 = warp_sum_int(ti.s1); ti.s2 = warp_sum_int(ti.s2);
      if ((threadIdx.x & 31) == 0) redi[threadIdx.x >> 5] = ti;
      __syncthreads();
      if (threadIdx.x == 0) cp[fi] = cp_int_finish(redi, fd.n_syms);
    }
    else
    {
      acc.x = warp_sum(acc.x);
      acc.y = warp_sum(acc.y);
      if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
      __syncthreads();
      if (threadIdx.x == 0)
      {
        float2 s = red[0];
        for (int w = 1; w < 8; w++) { s.x += red[w].x; s.y += red[w].y; }
        cp[fi] = s;
      }
    }
    __syncthreads();
  }
}

// The same sums for 8-bit input with the samples brought in by the TMA engine: a warp keeps CPB_STAGES symbols in flight, each as
// two bulk copies (the prefix and the samples 2048 later, 1024 bytes from a 16-byte aligned start; both have the same offset in
// their copy) into the warp's own ring in shared memory, completion on an mbarrier per stage. A lane then takes 16 bytes (eight
// samples) of each copy at a time; the bytes of the first and the last 16 that lie outside the prefix are masked. No register
// waits for a load (k_cp_corr: 67 % of the stall samples on the 32 two-byte loads of a symbol, 3.6 TB/s), a warp has 8 KB in
// flight instead of 2, and the sums are exact integers, so the result equals k_cp_corr's. Symbols whose aligned copies could
// leave the recording take the direct loads.
constexpr int CPB_STAGES = 4;
constexpr int CPB_COPY = 1024;
constexpr int CPB_SMEM = 8 * CPB_STAGES * 2 * CPB_COPY;

__global__ void __launch_bounds__(256) k_cp_corr_bulk(const FrameDesc * __restrict__ frames, int n_frames, const RecInput * __restrict__ recs, float2 * __restrict__ cp)
{
  extern __shared__ __align__(128) unsigned char cpb_ring[];
  __shared__ unsigned long long cpb_bar[8 * CPB_STAGES];
  __shared__ CpInt red[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char * ring = cpb_ring + warp * (CPB_STAGES * 2 * CPB_COPY);
  const unsigned ring_s = smem_addr_u32(ring), bar_s = smem_addr_u32(cpb_bar + warp * CPB_STAGES);
  if (lane == 0)
  {
#pragma unroll
    for (int b = 0; b < CPB_STAGES; b++) mbar_init(bar_s + 8u * (unsigned)b, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  // the warp's symbols in order: frames blockIdx.x, blockIdx.x + gridDim.x, ..., symbols warp, warp + 8, ... of each
  struct Cursor
  {
    int fi, sym, n_syms;
    long long base, n;
    const unsigned char * iq;
  };
  auto enter = [&](Cursor & c) {
    // first frame from c.fi on that has a symbol for this warp
    while (c.fi < n_frames)
    {
      const FrameDesc & fd = frames[c.fi];
      c.n_syms = fd.n_syms;
      if (warp < c.n_syms)
      {
        const RecInput rin = recs[fd.rec];
        c.base = fd.sym0 + T_U;
        c.n = rin.n;
        c.iq = static_cast<const unsigned char *>(rin.iq);
        c.sym = warp;
        return;
      }
      c.fi += (int)gridDim.x;
    }
  };
  auto advance = [&](Cursor & c) {
    c.sym += 8;
    if (c.sym >= c.n_syms) { c.fi += (int)gridDim.x; enter(c); }
  };
  auto first_sample = [](const Cursor & c) { return c.base + (long long)c.sym * T_S; };
  auto by_copy = [&](const Cursor & c) { const long long s0 = first_sample(c); return s0 >= 8 && s0 + T_U + T_G + 8 <= c.n; };
  auto issue = [&](const Cursor & c, int b) {
    if (c.fi < n_frames && by_copy(c) && lane == 0)
    {
      const unsigned long long a = (unsigned long long)(c.iq + 2 * first_sample(c)) & ~15ull;
      const unsigned dst = ring_s + (unsigned)(b * 2 * CPB_COPY), bar = bar_s + 8u * (unsigned)b;
      mbar_expect_tx(bar, 2u * CPB_COPY);
      bulk_g2s(dst, reinterpret_cast<const void *>(a), CPB_COPY, bar);
      bulk_g2s(dst + CPB_COPY, reinterpret_cast<const void *>(a + 2ull * T_U), CPB_COPY, bar);
    }
  };

  Cursor ahead;
  ahead.fi = (int)blockIdx.x;
  ahead.sym = 0; ahead.n_syms = 0; ahead.base = 0; ahead.n = 0; ahead.iq = nullptr;
  enter(ahead);
  Cursor cur = ahead;
#pragma unroll 1
  for (int b = 0; b < CPB_STAGES && ahead.fi < n_frames; b++) { issue(ahead, b); advance(ahead); }
  int stage = 0;
  unsigned phase_bits = 0;

  for (int fi = blockIdx.x; fi < n_frames; fi += gridDim.x)
  {
    CpInt ti = { 0, 0, 0, 0 };
    const int n_syms = frames[fi].n_syms;
    while (cur.fi == fi)
    {
      if (by_copy(cur))
      {
        mbar_wait(bar_s + 8u * (unsigned)stage, (phase_bits >> stage) & 1u);
        phase_bits ^= 1u << stage;
        const int off = (int)((unsigned long long)(cur.iq + 2 * first_sample(cur)) & 15ull); // the prefix is bytes [off, off + 1008) of a copy
        const uint4 * sp = reinterpret_cast<const uint4 *>(ring + stage * 2 * CPB_COPY) + lane;
        uint4 va[2], vb[2];
#pragma unroll
        for (int it = 0; it < 2; it++) { vb[it] = sp[32 * it]; va[it] = sp[32 * it + CPB_COPY / 16]; }
        if (lane == 0)
        {
          // bytes [0, off) of the first 16 (off is even)
          unsigned * w = reinterpret_cast<unsigned *>(&va[0]);
          unsigned * u = reinterpret_cast<unsigned *>(&vb[0]);
#pragma unroll
          for (int j = 0; j < 4; j++)
          {
            const int drop = min(max(off - 4 * j, 0), 4); // leading bytes of word j that precede the prefix
            const unsigned m = drop >= 4 ? 0u : 0xffffffffu << (8 * drop);
            w[j] &= m;
            u[j] &= m;
          }
        }
        if (lane == 31)
        {
          // bytes [off - 16 + 16, 16) of the last 16, i.e. those from 1008 + off on: keep the first `off` bytes
          unsigned * w = reinterpret_cast<unsigned *>(&va[1]);
          unsigned * u = reinterpret_cast<unsigned *>(&vb[1]);
#pragma unroll
          for (int j = 0; j < 4; j++)
          {
            const int keep = min(max(off - 4 * j, 0), 4);
            const unsigned m = keep >= 4 ? 0xffffffffu : ~(0xffffffffu << (8 * keep));
            w[j] &= m;
            u[j] &= m;
          }
        }
#pragma unroll
        for (int it = 0; it < 2; it++)
        {
          cp_int_add(ti, va[it].x, vb[it].x);
          cp_int_add(ti, va[it].y, vb[it].y);
          cp_int_add(ti, va[it].z, vb[it].z);
          cp_int_add(ti, va[it].w, vb[it].w);
        }
      }
      else
      {
        const unsigned short * pp = reinterpret_cast<const unsigned short *>(cur.iq) + first_sample(cur) + lane;
        unsigned ra[16], rb[16];
#pragma unroll
        for (int k = 0; k < 16; k++)
        {
          if (lane + 32 * k < T_G) { ra[k] = pp[32 * k + T_U]; rb[k] = pp[32 * k]; }
          else { ra[k] = 0; rb[k] = 0; }
        }
#pragma unroll
        for (int k = 0; k < 16; k++) cp_int_add(ti, ra[k], rb[k]);
      }
      // the stage is free again: every lane has its values in registers
      __syncwarp();
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      issue(ahead, stage);
      if (ahead.fi < n_frames) advance(ahead);
      advance(cur);
      stage = stage + 1 == CPB_STAGES ? 0 : stage + 1;
    }
    ti.p1 = warp_sum_int(ti.p1); ti.p2 = warp_sum_int(ti.p2); ti.s1 = warp_sum_int(ti.s1); ti.s2 = warp_sum_int(ti.s2);
    if (lane == 0) red[warp] = ti;
    __syncthreads();
    if (threadIdx.x == 0) cp[fi] = cp_int_finish(red, n_syms);
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------ DQPSK demapper (D1-D4)
// OfdmDecoder::decode_symbol (ofdm_decoder.cpp:147-355) for whole recordings. The per-carrier IIR chains are sequential
// in time but independent across carriers, so the parallelism is (recordings or segments) x carriers:
//   * a run (DemapWork: consecutive frames of one recording) is 3 CTAs of 128 threads; a thread owns 4 adjacent carriers
//     = two pairs: one 32-byte piece of a spectrum row, one 8-byte store per soft-bit plane. The two carriers of a pair run
//     in the two halves of the packed FP32 instructions (FADD2 / FMUL2 / FFMA2); the two pairs are independent dependency
//     chains the scheduler interleaves;
//   * the only coupling between carriers, mMeanValue (sum of |r| over the PREVIOUS symbol, ofdm_decoder.cpp:256,294),
//     scales the OUTPUT only. Each warp publishes its partial sum of symbol g as one 64-bit word {g+1, sum} in a ring
//     in global memory (L2), keeps its unscaled r in a shared-memory stash, and writes the soft bits of symbol
//     g - LAG, whose scale (12 partial sums of symbol g - LAG - 1, added in a fixed order by every warp for itself)
//     was published several symbols ago: the tag check rarely fails (then the warp polls), and there is no barrier,
//     cluster or designated reducer;
//   * the launch is NOT cooperative: a CTA takes its work item from a ticket counter when it starts, so the CTAs a running
//     CTA may wait for (the other slices of its run) either run already or are the next to start as soon as any CTA
//     finishes: there is always a run with all slices resident, hence no deadlock, for any number of runs per launch;
//   * spectrum rows arrive through a per-thread cp.async ring in shared memory, 8 rows deep: the load of row q + 8 is issued
//     when row q is consumed and nothing reads a destination register in between;
//   * 6.5 MUFU per carrier and symbol: rsqrt|X|^2 (shared by two symbols), rcp for the arctangent, sqrt(meanPow),
//     rsqrt|z|^2, sqrt(|P|/|z|) and one reciprocal of the combined denominator; the arctangent is a degree-13 odd minimax
//     polynomial; x86 (i16)(float) semantics of the output conversion are checked once per thread and row.
// History (ms per 9984 frames): one CTA per recording with IEEE division / atan2 12.5; cluster of 4 CTAs over DSMEM 9.7;
// scalar FP32 with the ring 8.1; packed FP32, 2 carriers per thread, cooperative launch (k_demap4, round 1) 5.49 at 235 warp
// instructions per thread and symbol of which ~87 are the recurrences; this kernel 5.58 at 366 per FOUR carriers (-28 %
// instructions, same time: two warps per scheduler leave it bound by dependent-issue latency, profiles/r2_a_*).
constexpr int DM3_RING = 64;           // > 2 * LAG + 2: a slot is never overwritten while a slower warp may still read it
constexpr int DM3_ROW4 = K_CARR / 2;   // float4 per spectrum row

__device__ __forceinline__ float rcp_ftz(float a) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a)); return r; }
__device__ __forceinline__ float rsqrt_ftz(float a) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a)); return r; }
__device__ __forceinline__ float sqrt_ftz(float a) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a)); return r; }

__device__ __forceinline__ unsigned long long ld_volatile_global_b64(const unsigned long long * p)
{
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.b64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_volatile_global_b64(unsigned long long * p, unsigned long long v)
{
  asm volatile("st.relaxed.gpu.global.b64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__device__ __forceinline__ float2 f2(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }

struct CarrierPair
{
  float2 integ, stddev, mean_pow, mean_sigma, null_pow; // .x = carrier 2t, .y = carrier 2t + 1
};

// arg(z) mod pi/2 for both carriers (see folded_phase)
__device__ __forceinline__ float2 folded_phase2(float2 re, float2 im)
{
  const float ax0 = fabsf(re.x), ay0 = fabsf(im.x), ax1 = fabsf(re.y), ay1 = fabsf(im.y);
  const float2 mn = make_float2(fminf(ax0, ay0), fminf(ax1, ay1));
  const float2 t = mul2(mn, make_float2(rcp_ftz(fmaxf(ax0, ay0)), rcp_ftz(fmaxf(ax1, ay1))));
  const float2 z = mul2(t, t);
  float2 p = f2(0.00681177107617259f);
  p = fma2(p, z, f2(-0.033604156225919724f));
  p = fma2(p, z, f2(0.07962360233068466f));
  p = fma2(p, z, f2(-0.13233338296413422f));
  p = fma2(p, z, f2(0.19807815551757812f));
  p = fma2(p, z, f2(-0.3331736922264099f));
  p = fma2(p, z, f2(0.9999961256980896f));
  const float2 a = mul2(p, t);
  const bool m0 = (ay0 > ax0) != ((__float_as_int(re.x) ^ __float_as_int(im.x)) < 0);
  const bool m1 = (ay1 > ax1) != ((__float_as_int(re.y) ^ __float_as_int(im.y)) < 0);
  return make_float2(m0 ? PI_2_F - a.x : a.x, m1 ? PI_2_F - a.y : a.y);
}

// decode_symbol (ofdm_decoder.cpp:166-294) for the two carriers of a thread. xr/xi, rr/ri: real and imaginary parts of the
// symbol and of the phase reference; returns the unscaled soft values in o_re/o_im and |r| of both carriers in r_abs.
template <int SOFT>
__device__ __forceinline__ void dm4_pair(CarrierPair & st, float2 xr, float2 xi, float2 rr, float2 ri, float2 ref_abs, float2 ref_inv, float2 cterm,
                                         float2 & o_re, float2 & o_im, float2 & r_abs, float2 & pow_acc)
{
  constexpr float ALPHA = 0.005f;
  // raw = x conj(ref) / |ref|
  const float2 re = mul2(fma2(xi, ri, mul2(xr, rr)), ref_inv);
  const float2 im = mul2(fma2(neg2(xr), ri, mul2(xi, rr)), ref_inv);
  // rotation by -(clock term + integrator), minimax polynomial of ofdm_decoder.cpp:70-88
  const float2 t = add2(cterm, st.integ), a2 = mul2(t, t);
  const float2 rx = fma2(a2, fma2(a2, f2(3.679168224334716796875e-2f), f2(-0.495580852031707763671875f)), f2(0.9994032382965087890625f));
  const float2 ry = mul2(neg2(t), fma2(a2, f2(-0.16034401953220367431640625f), f2(0.99903142452239990234375f)));
  const float2 zr = fma2(neg2(im), ry, mul2(re, rx));
  const float2 zi = fma2(im, rx, mul2(re, ry));
  const float2 dv = add2(folded_phase2(zr, zi), f2(-PI_4_F));
  const float2 in = fma2(dv, f2(0.2f * ALPHA), st.integ);
  st.integ = make_float2(fminf(fmaxf(in.x, -20.0f * RAD_PER_DEG_F), 20.0f * RAD_PER_DEG_F), fminf(fmaxf(in.y, -20.0f * RAD_PER_DEG_F), 20.0f * RAD_PER_DEG_F));
  st.stddev = fma2(fma2(dv, dv, neg2(st.stddev)), f2(ALPHA), st.stddev);
  const float2 pw = fma2(zr, zr, mul2(zi, zi));
  st.mean_pow = fma2(add2(pw, neg2(st.mean_pow)), f2(ALPHA), st.mean_pow);
  pow_acc = fma2(pow_acc, f2(POW_ALL_DECAY), pw); // this carrier's share of mMeanPowerOvrAll (kernels.h, OfdmStateDev)
  const float2 lvl = make_float2(sqrt_ftz(st.mean_pow.x), sqrt_ftz(st.mean_pow.y));
  const float2 dr = fma2(lvl, f2(-0.70710678118654752440f), make_float2(fabsf(zr.x), fabsf(zr.y)));
  const float2 di = fma2(lvl, f2(-0.70710678118654752440f), make_float2(fabsf(zi.x), fabsf(zi.y)));
  st.mean_sigma = fma2(add2(fma2(dr, dr, mul2(di, di)), neg2(st.mean_sigma)), f2(ALPHA), st.mean_sigma);
  float2 sig = add2(st.mean_pow, neg2(st.null_pow));
  if (sig.x <= 0.0f) sig.x = 0.1f;
  if (sig.y <= 0.0f) sig.y = 0.1f;
  const float2 inv_z = make_float2(rsqrt_ftz(pw.x), rsqrt_ftz(pw.y));
  float2 w1;
  if (SOFT == 2) w1 = ref_abs;
  else
  {
    // 1 / ((nullPow / sig + 0.7) * meanSigma) = sig / ((nullPow + 0.7 sig) * meanSigma)
    const float2 den = mul2(fma2(sig, f2(0.7f), st.null_pow), st.mean_sigma);
    const float2 g = mul2(sig, make_float2(rcp_ftz(den.x), rcp_ftz(den.y)));
    if (SOFT == 1) w1 = mul2(ref_abs, g);
    else
    {
      const float2 q = mul2(ref_abs, inv_z); // sqrt(|z| |P|) / |z| = sqrt(|P| / |z|)
      w1 = mul2(mul2(make_float2(sqrt_ftz(q.x), sqrt_ftz(q.y)), lvl), g);
    }
  }
  r_abs = mul2(mul2(pw, inv_z), w1); // |z| w1, w1 >= 0
  o_re = mul2(zr, w1);
  o_im = mul2(zi, w1);
}

// x86 cvttss2si returns 0x80000000 out of range (to_i16): a value the GPU conversion saturated to 0x7fffffff must read 0 in
// its low half, not 0xffff (start-up transient of SOFTDEC2). Checked once per thread and row.
__device__ __forceinline__ void dm4_fix_saturated(int & a, int & b, int & c, int & e)
{
  a = a == 0x7fffffff ? 0 : a; b = b == 0x7fffffff ? 0 : b; c = c == 0x7fffffff ? 0 : c; e = e == 0x7fffffff ? 0 : e;
}

// ------------------------------------------------------------------------------------------------ the demapper kernel
constexpr int DM5_T = 128;                 // threads per CTA
constexpr int DM5_SLICES = K_CARR / 4 / DM5_T; // 3 CTAs per recording
constexpr int DM5_WARPS = K_CARR / 128;    // 12 warps per recording
constexpr int DM5_PF = 8;                  // spectrum rows in flight per thread

__device__ __forceinline__ float dm5_total(const unsigned long long * slot, unsigned long long w, unsigned tag, int lane)
{
  while (__any_sync(0xffffffffu, lane < DM5_WARPS && (unsigned)(w >> 32) != tag)) w = ld_volatile_global_b64(slot + (lane < DM5_WARPS ? lane : 0));
  float v = lane < DM5_WARPS ? __uint_as_float((unsigned)w) : 0.0f;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// QUAL: per-frame signal-quality capture (dabstar_decoder_set_frame_quality). After the null symbol of every complete frame
// whose soft bits it writes, the run stores the frame's FrameQualSnap into qsnap[descriptor index]: the state the host's
// quality figures are taken from. mMeanValue of that state is the total of the frame's last symbol, which is known only LAG
// symbols later (emit of d = symbols at the frame's end, the drain, or tot_last). A complete frame is 75 symbols, more than
// LAG, so at most one snapshot waits for its mMeanValue at any time.
template <int SOFT, int LAG, bool QUAL>
__global__ void __launch_bounds__(DM5_T, 4) k_demap5(const DemapWork * __restrict__ work, const FrameDesc * __restrict__ frames,
                                                      const uint8_t * __restrict__ null_is_tii, const float2 * __restrict__ X,
                                                      const int16_t * __restrict__ rel_of_k, OfdmStateDev * __restrict__ states,
                                                      int16_t * __restrict__ soft, unsigned long long * __restrict__ ring, unsigned * __restrict__ ticket,
                                                      FrameQualSnap * __restrict__ qsnap)
{
  constexpr int STASH = LAG + 1; // stash depth (power of two)
  constexpr int T = DM5_T;
  static_assert((STASH & (STASH - 1)) == 0, "stash depth must be a power of two");
  static_assert(DM3_RING > 2 * LAG + 2, "a ring slot must not be overwritten while a slower warp may still read it");
  extern __shared__ float4 dm5_smem[]; // [STASH][T][2] unscaled soft values of the last symbols | [DM5_PF][T][2] spectrum rows in flight | [STASH][T / 32] output rows
  __shared__ unsigned s_ticket;
  if (threadIdx.x == 0) s_ticket = atomicAdd(ticket, 1u);
  __syncthreads();
  float4 * stash = dm5_smem;
  float4 * rowbuf = dm5_smem + STASH * T * 2;
  int * orow_ring = reinterpret_cast<int *>(rowbuf + DM5_PF * T * 2) + (threadIdx.x >> 5);
  const int w = (int)s_ticket / DM5_SLICES, slice = (int)s_ticket - w * DM5_SLICES;
  const DemapWork wk = work[w];
  const int tid = threadIdx.x, lane = tid & 31;
  const int t_rec = slice * T + tid; // thread index within the recording: carriers 4 t_rec .. 4 t_rec + 3
  const int gw = t_rec >> 5;         // warp index within the recording
  const int k0 = 4 * t_rec;
  unsigned long long * my_ring = ring + (size_t)w * DM3_RING * DM5_WARPS;

  const OfdmStateDev & sd = states[wk.state_in];
  CarrierPair sa, sb;
  float2 pow_a = f2(0.f), pow_b = f2(0.f);
  if (wk.reset) sa = sb = CarrierPair{ f2(0.f), f2(0.f), f2(0.f), f2(0.f), f2(0.f) };
  else
  {
    const float4 v0 = *reinterpret_cast<const float4 *>(sd.integ + k0), v1 = *reinterpret_cast<const float4 *>(sd.stddev + k0),
                 v2 = *reinterpret_cast<const float4 *>(sd.mean_pow + k0), v3 = *reinterpret_cast<const float4 *>(sd.mean_sigma + k0),
                 v4 = *reinterpret_cast<const float4 *>(sd.null_pow + k0), v5 = *reinterpret_cast<const float4 *>(sd.pow_acc + k0);
    sa = CarrierPair{ make_float2(v0.x, v0.y), make_float2(v1.x, v1.y), make_float2(v2.x, v2.y), make_float2(v3.x, v3.y), make_float2(v4.x, v4.y) };
    sb = CarrierPair{ make_float2(v0.z, v0.w), make_float2(v1.z, v1.w), make_float2(v2.z, v2.w), make_float2(v3.z, v3.w), make_float2(v4.z, v4.w) };
    pow_a = make_float2(v5.x, v5.y);
    pow_b = make_float2(v5.z, v5.w);
  }
  const float mean_value0 = sd.mean_value; // not touched by reset() (ofdm_decoder.cpp:90-101)
  const float pow_carry0 = wk.reset ? 1.0f : sd.pow_carry; // mMeanPowerOvrAll = 1 at reset() (ofdm_decoder.cpp:98)
  const float2 gka = make_float2((float)(K_CARR / 2 - rel_of_k[k0]) / (float)(K_CARR / 2), (float)(K_CARR / 2 - rel_of_k[k0 + 1]) / (float)(K_CARR / 2));
  const float2 gkb = make_float2((float)(K_CARR / 2 - rel_of_k[k0 + 2]) / (float)(K_CARR / 2), (float)(K_CARR / 2 - rel_of_k[k0 + 3]) / (float)(K_CARR / 2));
  constexpr float W2 = SOFT == 0 ? -100.0f : -140.0f;

  const int total_rows = wk.n_frames * X_ROWS;
  const float4 * rows = reinterpret_cast<const float4 *>(X + (size_t)(total_rows > 0 ? frames[wk.desc_first].xslot : 0) * X_ROWS * K_CARR) + 2 * t_rec;
  // (the two 16-byte halves of a thread's row / stash entry are interleaved at a 32-byte stride: twice the ideal wavefronts; separate
  // planes of contiguous 16-byte accesses were measured, 5.76 instead of 5.56 ms)
  const unsigned rowbuf_addr = smem_addr_u32(rowbuf + 2 * tid);
#pragma unroll
  for (int i = 0; i < DM5_PF; i++)
  {
    if (i < total_rows)
    {
      cp_async16(rowbuf_addr + (unsigned)(i * T) * 32u, rows + (size_t)i * DM3_ROW4);
      cp_async16(rowbuf_addr + (unsigned)(i * T) * 32u + 16u, rows + (size_t)i * DM3_ROW4 + 1);
    }
    cp_async_commit();
  }

  float2 rra = f2(0.f), ria = f2(0.f), ref_abs_a = f2(0.f), ref_inv_a = f2(0.f);
  float2 rrb = f2(0.f), rib = f2(0.f), ref_abs_b = f2(0.f), ref_inv_b = f2(0.f);
  int g = 0;               // symbols decoded so far; tag of symbol g is g + 1
  int q = 0;               // spectrum rows consumed so far
  unsigned long long pre = 0; // ring words (lane l < 12: warp l) of the symbol whose total scales this iteration's output

  // soft bits of symbol d (its unscaled values are in the stash); total = sum |r| of symbol d - 1 (unused for d = 0)
  auto emit = [&](int d, int o_row, float total) {
    if (o_row < 0) return; // warm-up frame of a segment: the state advances, nothing is written
    const float w2 = d == 0 ? rcp_ftz(mean_value0) * W2 : rcp_ftz(total) * (W2 * (float)K_CARR);
    const float4 ra = stash[((d & (STASH - 1)) * T + tid) * 2], rb = stash[((d & (STASH - 1)) * T + tid) * 2 + 1]; // (re0, re1, im0, im1) of each pair
    const float2 are = mul2(make_float2(ra.x, ra.y), f2(w2)), aim = mul2(make_float2(ra.z, ra.w), f2(w2));
    const float2 bre = mul2(make_float2(rb.x, rb.y), f2(w2)), bim = mul2(make_float2(rb.z, rb.w), f2(w2));
    int a0 = __float2int_rz(are.x), a1 = __float2int_rz(are.y), a2 = __float2int_rz(aim.x), a3 = __float2int_rz(aim.y);
    int b0 = __float2int_rz(bre.x), b1 = __float2int_rz(bre.y), b2 = __float2int_rz(bim.x), b3 = __float2int_rz(bim.y);
    if (max(max(max(a0, a1), max(a2, a3)), max(max(b0, b1), max(b2, b3))) == 0x7fffffff) { dm4_fix_saturated(a0, a1, a2, a3); dm4_fix_saturated(b0, b1, b2, b3); }
    int16_t * o = soft + (size_t)o_row * SYM_BITS;
    reinterpret_cast<uint2 *>(o)[t_rec] = make_uint2(__byte_perm((unsigned)a0, (unsigned)a1, 0x5410), __byte_perm((unsigned)b0, (unsigned)b1, 0x5410));
    reinterpret_cast<uint2 *>(o + K_CARR)[t_rec] = make_uint2(__byte_perm((unsigned)a2, (unsigned)a3, 0x5410), __byte_perm((unsigned)b2, (unsigned)b3, 0x5410));
  };
  auto wsum = [](float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
  };
  // the next spectrum row of this thread (its load was requested DM5_PF rows ago); requests row q + DM5_PF
  float4 cur_a, cur_b;
  auto next_row = [&]() {
    cp_async_wait<DM5_PF - 1>();
    const unsigned slot = (unsigned)((q & (DM5_PF - 1)) * T);
    cur_a = rowbuf[(slot + tid) * 2];
    cur_b = rowbuf[(slot + tid) * 2 + 1];
    if (q + DM5_PF < total_rows)
    {
      cp_async16(rowbuf_addr + slot * 32u, rows + (size_t)(q + DM5_PF) * DM3_ROW4);
      cp_async16(rowbuf_addr + slot * 32u + 16u, rows + (size_t)(q + DM5_PF) * DM3_ROW4 + 1);
    }
    cp_async_commit();
    q++;
  };
  // this row is the phase reference of the next symbol
  auto set_reference = [&]() {
    rra = make_float2(cur_a.x, cur_a.y); ria = make_float2(cur_a.z, cur_a.w);
    rrb = make_float2(cur_b.x, cur_b.y); rib = make_float2(cur_b.z, cur_b.w);
    const float2 pa = fma2(rra, rra, mul2(ria, ria)), pb = fma2(rrb, rrb, mul2(rib, rib));
    ref_inv_a = make_float2(rsqrt_ftz(pa.x), rsqrt_ftz(pa.y));
    ref_inv_b = make_float2(rsqrt_ftz(pb.x), rsqrt_ftz(pb.y));
    ref_abs_a = mul2(pa, ref_inv_a);
    ref_abs_b = mul2(pb, ref_inv_b);
  };
  float part_prev = 0.0f; // this thread's |r| sum of symbol g - 1, published (reduced over the warp) one symbol late
  const bool upper = (lane & 16) != 0;
  int q_wait_g = -1, q_wait = 0; // QUAL: symbol count at the end of the snapshot that waits for its mMeanValue, and its index
  auto q_mean_value = [&](int d, float total) {
    if (QUAL && d == q_wait_g)
    {
      if (t_rec == 0) qsnap[q_wait].mean_value = total / (float)K_CARR;
      q_wait_g = -1;
    }
  };

  for (int fi = 0; fi < wk.n_frames; fi++)
  {
    const FrameDesc fd = frames[wk.desc_first + fi];
    const float cfac = fd.clock_err / 1024.0f * PI_F;
    const float2 cterm_a = mul2(f2(cfac), gka), cterm_b = mul2(f2(cfac), gkb);
    const int n_syms = fd.n_syms;
    const int out_row0 = fi < wk.warmup ? -(1 << 30) : fd.slot * 75;
    const bool tii = null_is_tii != nullptr && null_is_tii[wk.desc_first + fi];
    next_row();
    set_reference(); // store_reference_symbol_0
    for (int sym = 1; sym <= 75; sym++)
    {
      next_row();
      if (sym > n_syms) continue; // the recording ends inside this frame
      const int d = g - LAG; // symbol whose soft bits are written in this iteration
      // ONE shuffle chain, independent of this symbol's arithmetic, reduces two values: this warp's share of sum |r| of the PREVIOUS symbol (lower half warp) and
      // the total of symbol d - 1 from the ring words fetched one iteration ago (upper half warp)
      const float b_in = lane < DM5_WARPS ? __uint_as_float((unsigned)pre) : 0.0f;
      const bool tags_ok = __all_sync(0xffffffffu, lane >= DM5_WARPS || (unsigned)(pre >> 32) == (unsigned)d);
      const unsigned long long pre_used = pre;
      if (d >= 0 && lane < DM5_WARPS) pre = ld_volatile_global_b64(my_ring + (size_t)(d & (DM3_RING - 1)) * DM5_WARPS + lane);
      float v = (upper ? b_in : part_prev) + __shfl_xor_sync(0xffffffffu, upper ? part_prev : b_in, 16);
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      const float tot_fast = __shfl_sync(0xffffffffu, v, 16);
      float2 a_re, a_im, a_abs, b_re, b_im, b_abs;
      dm4_pair<SOFT>(sa, make_float2(cur_a.x, cur_a.y), make_float2(cur_a.z, cur_a.w), rra, ria, ref_abs_a, ref_inv_a, cterm_a, a_re, a_im, a_abs, pow_a);
      dm4_pair<SOFT>(sb, make_float2(cur_b.x, cur_b.y), make_float2(cur_b.z, cur_b.w), rrb, rib, ref_abs_b, ref_inv_b, cterm_b, b_re, b_im, b_abs, pow_b);
      part_prev = (a_abs.x + a_abs.y) + (b_abs.x + b_abs.y);
      stash[((g & (STASH - 1)) * T + tid) * 2] = make_float4(a_re.x, a_re.y, a_im.x, a_im.y);
      stash[((g & (STASH - 1)) * T + tid) * 2 + 1] = make_float4(b_re.x, b_re.y, b_im.x, b_im.y);
      if (lane == 0) orow_ring[(g & (STASH - 1)) * (T >> 5)] = out_row0 + (sym - 1);
      __syncwarp();
      if (lane == 0 && g > 0)
        st_volatile_global_b64(my_ring + (size_t)((g - 1) & (DM3_RING - 1)) * DM5_WARPS + gw,
                               ((unsigned long long)(unsigned)g << 32) | (unsigned long long)__float_as_uint(v));
      if (d >= 0)
      {
        float tot = tot_fast;
        if (d > 0 && !tags_ok) tot = dm5_total(my_ring + (size_t)((d - 1) & (DM3_RING - 1)) * DM5_WARPS, pre_used, (unsigned)d, lane);
        emit(d, orow_ring[(d & (STASH - 1)) * (T >> 5)], tot);
        q_mean_value(d, tot);
      }
      g++;
      set_reference();
    }
    next_row(); // null symbol
    if (n_syms == 75 && !tii)
    {
      // store_null_symbol_without_tii (ofdm_decoder.cpp:114-130)
      constexpr float MIN_POW = (1.0f / 32767.0f) * (1.0f / 32767.0f);
      const float2 xra = make_float2(cur_a.x, cur_a.y), xia = make_float2(cur_a.z, cur_a.w), xrb = make_float2(cur_b.x, cur_b.y), xib = make_float2(cur_b.z, cur_b.w);
      const float2 pa = add2(fma2(xra, xra, mul2(xia, xia)), f2(MIN_POW)), pb = add2(fma2(xrb, xrb, mul2(xib, xib)), f2(MIN_POW));
      sa.null_pow = fma2(add2(pa, neg2(sa.null_pow)), f2(0.05f), sa.null_pow);
      sb.null_pow = fma2(add2(pb, neg2(sb.null_pow)), f2(0.05f), sb.null_pow);
    }
    if (QUAL && out_row0 >= 0 && n_syms == 75)
    {
      FrameQualSnap & qs = qsnap[wk.desc_first + fi];
      *reinterpret_cast<float4 *>(qs.stddev + k0) = make_float4(sa.stddev.x, sa.stddev.y, sb.stddev.x, sb.stddev.y);
      *reinterpret_cast<float4 *>(qs.null_pow + k0) = make_float4(sa.null_pow.x, sa.null_pow.y, sb.null_pow.x, sb.null_pow.y);
      *reinterpret_cast<float4 *>(qs.pow_acc + k0) = make_float4(pow_a.x, pow_a.y, pow_b.x, pow_b.y);
      if (t_rec == 0) qs.pow_carry = pow_carry0 * powf(POW_ALL_DECAY, (float)g);
      q_wait_g = g;
      q_wait = wk.desc_first + fi;
    }
  }
  cp_async_wait<0>();
  // the last symbol's share has not been published yet
  if (g > 0)
  {
    const float part = wsum(part_prev);
    if (lane == 0)
      st_volatile_global_b64(my_ring + (size_t)((g - 1) & (DM3_RING - 1)) * DM5_WARPS + gw,
                             ((unsigned long long)(unsigned)g << 32) | (unsigned long long)__float_as_uint(part));
  }
  // drain: the last LAG symbols
#pragma unroll
  for (int i = LAG - 1; i >= 0; i--)
  {
    const int d = g - 1 - i;
    if (d < 0) continue;
    float tot = 0.0f;
    if (d >= 1)
    {
      const unsigned long long * slot = my_ring + (size_t)((d - 1) & (DM3_RING - 1)) * DM5_WARPS;
      unsigned long long word = 0;
      if (lane < DM5_WARPS) word = ld_volatile_global_b64(slot + lane);
      tot = dm5_total(slot, word, (unsigned)d, lane);
    }
    emit(d, orow_ring[(d & (STASH - 1)) * (T >> 5)], tot);
    q_mean_value(d, tot);
  }
  if (!QUAL && wk.state_out < 0) return; // a segment that does not end the window: its state is not the recording's
  // mMeanValue after the last symbol, fetched BEFORE anything is stored: with state_out == state_in the other slices of the
  // recording read mean_value when they start, which may be later than this (the launch is not cooperative); whoever can
  // see the last symbol's total has been waited for by it, i.e. all slices have started and read their input state
  float tot_last = mean_value0 * (float)K_CARR;
  if (gw == 0 && g > 0)
  {
    unsigned long long word = 0;
    const unsigned long long * slot = my_ring + (size_t)((g - 1) & (DM3_RING - 1)) * DM5_WARPS;
    if (lane < DM5_WARPS) word = ld_volatile_global_b64(slot + lane);
    tot_last = dm5_total(slot, word, (unsigned)g, lane);
  }
  if (QUAL)
  {
    q_mean_value(g, tot_last); // (the last frame's snapshot: its total is tot_last, also when no state is stored)
    if (wk.state_out < 0) return;
  }
  OfdmStateDev & so = states[wk.state_out];
  *reinterpret_cast<float4 *>(so.integ + k0) = make_float4(sa.integ.x, sa.integ.y, sb.integ.x, sb.integ.y);
  *reinterpret_cast<float4 *>(so.stddev + k0) = make_float4(sa.stddev.x, sa.stddev.y, sb.stddev.x, sb.stddev.y);
  *reinterpret_cast<float4 *>(so.mean_pow + k0) = make_float4(sa.mean_pow.x, sa.mean_pow.y, sb.mean_pow.x, sb.mean_pow.y);
  *reinterpret_cast<float4 *>(so.mean_sigma + k0) = make_float4(sa.mean_sigma.x, sa.mean_sigma.y, sb.mean_sigma.x, sb.mean_sigma.y);
  *reinterpret_cast<float4 *>(so.null_pow + k0) = make_float4(sa.null_pow.x, sa.null_pow.y, sb.null_pow.x, sb.null_pow.y);
  *reinterpret_cast<float4 *>(so.pow_acc + k0) = make_float4(pow_a.x, pow_a.y, pow_b.x, pow_b.y);
  if (gw == 0 && lane == 0) so.mean_value = g > 0 ? tot_last / (float)K_CARR : mean_value0;
  if (t_rec == 0) so.pow_carry = pow_carry0 * powf(POW_ALL_DECAY, (float)g); // (only this thread reads or writes pow_carry)
}

// ------------------------------------------------------------------------------------------------ time sync (S1)
// TimeSyncer::read_samples_until_end_of_level_drop (timesyncer.cpp:40-90) on top of SampleReader's level IIR
// (sample_reader.cpp:236, alpha = 1e-5). One CTA per recording; the stream is scanned in blocks of 1024 samples.
constexpr int DIP_THREADS = 256;
constexpr int DIP_BLOCK = 1024;
constexpr float LEVEL_ALPHA = 0.00001f;

template <int FMT> __device__ __forceinline__ float sample_abs(const void * iq, long long i)
{
  const float2 v = load_sample<FMT>(iq, i);
  return sqrtf(v.x * v.x + v.y * v.y);
}
// The same in two halves, so that a batch of loads is issued before the first conversion: the IEEE square root carries a
// branch (its slow path), and a load is not moved across it (ncu: 63 % of this kernel's stall samples sat on the instruction
// after each load, one memory latency per sample).
template <int FMT> __device__ __forceinline__ typename Raw<FMT>::reg sample_raw(const void * iq, long long i)
{
  return (typename Raw<FMT>::reg)reinterpret_cast<const typename Raw<FMT>::type *>(iq)[i];
}
template <int FMT> __device__ __forceinline__ float raw_abs(typename Raw<FMT>::reg r)
{
  const float2 v = to_cf(r);
  return sqrtf(v.x * v.x + v.y * v.y);
}

template <int FMT>
__global__ void __launch_bounds__(DIP_THREADS) k_dip_search(const DipWork * __restrict__ work, const RecInput * __restrict__ recs, DipResult * __restrict__ out)
{
  __shared__ float mag[DIP_BLOCK + 64];
  __shared__ float lvl[DIP_BLOCK];
  __shared__ float2 scan_ab[DIP_THREADS];
  __shared__ float redf[DIP_THREADS / 32];
  __shared__ int found;
  const DipWork wk = work[blockIdx.x];
  const RecInput rin = recs[wk.rec];
  const int tid = threadIdx.x;
  const long long p0 = wk.pos;
  const float loga = log1pf(-LEVEL_ALPHA);

  // sLevel at p0: IIR over everything read so far (initial value 0.1, sample_reader.h:91); older than 2^21 samples is < 1e-9.
  const long long hist = p0 < (1LL << 21) ? p0 : (1LL << 21);
  // weight of sample p0 - 1 - i is (1 - alpha)^i. Eight samples of a thread are in flight at a time (a re-synchronisation deep
  // in a stream sums 2^21 samples, one CTA per recording: with one 2-byte load per iteration the kernel was a chain of
  // memory latencies); their weights are one expf times the constants (1 - alpha)^(256 u).
  float acc = 0.0f;
  {
    float ru[8];
#pragma unroll
    for (int u = 0; u < 8; u++) ru[u] = expf((float)(DIP_THREADS * u) * loga);
    long long i = tid;
    for (; i + 7LL * DIP_THREADS < hist; i += 8LL * DIP_THREADS)
    {
      typename Raw<FMT>::reg rw[8];
#pragma unroll
      for (int u = 0; u < 8; u++) rw[u] = sample_raw<FMT>(rin.iq, p0 - 1 - (i + (long long)u * DIP_THREADS));
      float m[8];
#pragma unroll
      for (int u = 0; u < 8; u++) m[u] = raw_abs<FMT>(rw[u]);
      const float w = expf((float)i * loga);
#pragma unroll
      for (int u = 0; u < 8; u++) acc = fmaf(m[u], w * ru[u], acc);
    }
    for (; i < hist; i += DIP_THREADS) acc = fmaf(sample_abs<FMT>(rin.iq, p0 - 1 - i), expf((float)i * loga), acc);
  }
  acc = warp_sum(acc);
  if ((tid & 31) == 0) redf[tid >> 5] = acc;
  __syncthreads();
  float s_level = 0.0f;
  for (int w = 0; w < DIP_THREADS / 32; w++) s_level += redf[w];
  s_level = LEVEL_ALPHA * s_level + (hist == p0 ? 0.1f * expf((float)(p0 + wk.abs0) * loga) : 0.0f);
  __syncthreads();

  // phase 0: searching the dip (first check after 50 samples), phase 1: searching its end
  int phase = 0;
  long long dip_i = -1;
  int status = -1;
  long long end_pos = p0;
  const float a1 = 1.0f - LEVEL_ALPHA;
  // |x| of a block's own 1024 samples, fetched one block ahead (the loads of block b + 1 are in flight while block b is
  // evaluated); the 49 samples of window history in front of a block are the tail of the previous block's array
  typename Raw<FMT>::reg nx[DIP_BLOCK / DIP_THREADS]; // raw: converted when the block is filed, a block later
  auto fetch = [&](long long b0) {
    const bool inside = p0 + b0 + DIP_BLOCK <= rin.n;
#pragma unroll
    for (int u = 0; u < DIP_BLOCK / DIP_THREADS; u++) nx[u] = inside ? sample_raw<FMT>(rin.iq, p0 + b0 + tid + u * DIP_THREADS) : typename Raw<FMT>::reg();
  };
  fetch(0);
  if (tid < 49) mag[tid] = 0.0f; // nothing in front of the search
  for (long long b0 = 0; status < 0; b0 += DIP_BLOCK)
  {
    if (p0 + b0 + DIP_BLOCK > rin.n) { status = 3; end_pos = rin.n; break; }
    if (b0 > 0)
    {
      float keep = 0.0f;
      if (tid < 49) keep = mag[DIP_BLOCK + tid];
      __syncthreads();
      if (tid < 49) mag[tid] = keep;
    }
#pragma unroll
    for (int u = 0; u < DIP_BLOCK / DIP_THREADS; u++) mag[49 + tid + u * DIP_THREADS] = raw_abs<FMT>(nx[u]);
    __syncthreads();
    fetch(b0 + DIP_BLOCK);
    // level IIR s_i = a s_{i-1} + alpha |x_i| as a scan of affine maps, 4 samples per thread
    float A = 1.0f, B = 0.0f;
#pragma unroll
    for (int q = 0; q < 4; q++) { const float m = mag[49 + 4 * tid + q]; B = a1 * B + LEVEL_ALPHA * m; A *= a1; }
    // inclusive scan of the maps (composition: first this thread's predecessors, then its own): shuffles inside a warp, the eight
    // warp totals through shared memory
    {
      const int lane = tid & 31, wp = tid >> 5;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1)
      {
        const float pa = __shfl_up_sync(0xffffffffu, A, o), pb = __shfl_up_sync(0xffffffffu, B, o);
        if (lane >= o) { B = fmaf(A, pb, B); A *= pa; }
      }
      if (lane == 31) scan_ab[wp] = make_float2(A, B);
      __syncthreads();
      // level in front of this warp: the block's start level through the totals of the warps before it
      float s = s_level;
      for (int w = 0; w < wp; w++) { const float2 ab = scan_ab[w]; s = fmaf(ab.x, s, ab.y); }
      // level in front of this thread: through the inclusive map of the lane before it
      const float ea = __shfl_up_sync(0xffffffffu, A, 1), eb = __shfl_up_sync(0xffffffffu, B, 1);
      if (lane > 0) s = fmaf(ea, s, eb);
#pragma unroll
      for (int q = 0; q < 4; q++) { s = a1 * s + LEVEL_ALPHA * mag[49 + 4 * tid + q]; lvl[4 * tid + q] = s; }
      if (tid == DIP_THREADS - 1) scan_ab[DIP_THREADS / 32].x = s; // level after the block
    }
    if (tid == 0) found = 0x7fffffff;
    __syncthreads();
    const float s_after = scan_ab[DIP_THREADS / 32].x;
    // evaluate both phases inside this block (the dip end may follow in the same block)
    int from = 0;
    while (true)
    {
      int best = 0x7fffffff;
      {
        // window sums of the thread's four samples: the first directly (two chains), the others by sliding, as the reference's
        // running sum does (timesyncer.cpp:57-62); mag[i..i+49] = samples gi-49..gi
        float c0 = 0.0f, c1 = 0.0f;
#pragma unroll 5
        for (int j = 0; j < 50; j += 2) { c0 += mag[4 * tid + j]; c1 += mag[4 * tid + j + 1]; }
        float c = c0 + c1;
#pragma unroll
        for (int q = 0; q < 4; q++)
        {
          const int i = 4 * tid + q;
          const long long gi = b0 + i;
          if (q > 0) c += mag[i + 49] - mag[i - 1];
          if (i < from || (phase == 0 && gi < 49) || best != 0x7fffffff) continue;
          const float mean = c / 50.0f;
          const bool hit = phase == 0 ? !(mean > 0.55f * lvl[i]) : !(mean < 0.75f * lvl[i]);
          if (hit) best = i;
        }
      }
      if (best != 0x7fffffff) atomicMin(&found, best);
      __syncthreads();
      const int f = found;
      __syncthreads();
      if (tid == 0) found = 0x7fffffff;
      __syncthreads();
      // limits: dip within T_F loop reads (timesyncer.cpp:66-69), end within T_N + 70 (timesyncer.cpp:82-85)
      if (phase == 0)
      {
        const long long lim = 49 + (long long)T_F; // last index whose condition is still evaluated
        const long long gi = f == 0x7fffffff ? (long long)1 << 60 : b0 + f;
        if (gi <= lim) { phase = 1; dip_i = gi; from = f; continue; }
        if (b0 + DIP_BLOCK - 1 >= lim + 1) { status = 1; end_pos = p0 + lim + 2; }
        break;
      }
      else
      {
        const long long lim = dip_i + T_N + 70;
        const long long gi = f == 0x7fffffff ? (long long)1 << 60 : b0 + f;
        if (gi <= lim) { status = 0; end_pos = p0 + gi + 1; }
        else if (b0 + DIP_BLOCK - 1 >= lim + 1) { status = 2; end_pos = p0 + lim + 2; }
        break;
      }
    }
    s_level = s_after;
    __syncthreads();
  }
  if (tid == 0)
  {
    if (end_pos > rin.n) { end_pos = rin.n; status = 3; }
    out[blockIdx.x].pos = end_pos;
    out[blockIdx.x].status = status;
    out[blockIdx.x].s_level = s_level;
  }
}

// ------------------------------------------------------------------------------------------------ file sample formats (I1)
// XmlReader::readElements_* (xml_filereader/xml_reader.cpp:254-800) for the formats the FFT kernel does not read natively.
// One thread per complex sample; the 8-bit containers go through a 256-entry table computed on the host with the
// reference's own expressions, the wider ones are assembled byte by byte (either byte order) and divided by 2^(bits-1)
// (an exact multiplication by the reciprocal).
__device__ __forceinline__ float ingest_value(const unsigned char * p, int container, int msb_first, float inv_scaler, const float * __restrict__ lut)
{
  switch (container)
  {
  case 0: case 1: case 6: return lut[p[0]];
  case 7: // libsndfile PCM_32 -> float: v / 2^31 (positive scaler, unlike the XML reader's wrapped one)
  {
    const unsigned v = ((unsigned)p[3] << 24) | (p[2] << 16) | (p[1] << 8) | p[0];
    return (float)(int)v * 4.656612873077393e-10f;
  }
  case 2:
  {
    const int v = msb_first ? ((p[0] << 8) | p[1]) : ((p[1] << 8) | p[0]);
    return (float)(short)v * inv_scaler;
  }
  case 3:
  {
    int v = msb_first ? ((p[0] << 16) | (p[1] << 8) | p[2]) : ((p[2] << 16) | (p[1] << 8) | p[0]);
    if (v & 0x800000) v |= (int)0xFF000000;
    return (float)v * inv_scaler;
  }
  case 4:
  {
    const unsigned v = msb_first ? (((unsigned)p[0] << 24) | (p[1] << 16) | (p[2] << 8) | p[3]) : (((unsigned)p[3] << 24) | (p[2] << 16) | (p[1] << 8) | p[0]);
    return (float)(int)v * inv_scaler;
  }
  default:
  {
    const unsigned v = msb_first ? (((unsigned)p[0] << 24) | (p[1] << 16) | (p[2] << 8) | p[3]) : (((unsigned)p[3] << 24) | (p[2] << 16) | (p[1] << 8) | p[0]);
    return __uint_as_float(v);
  }
  }
}

__global__ void __launch_bounds__(256) k_ingest_convert(const unsigned char * __restrict__ src, int container, int msb_first, int iq_order, float inv_scaler,
                                                        const float * __restrict__ lut, long long n, float2 * __restrict__ dst)
{
  const int bytes = (container <= 1 || container == 6) ? 1 : (container == 2 ? 2 : (container == 3 ? 3 : 4));
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
  {
    float2 o;
    if (iq_order <= 1)
    {
      const float a = ingest_value(src + (2 * i) * bytes, container, msb_first, inv_scaler, lut);
      const float b = ingest_value(src + (2 * i + 1) * bytes, container, msb_first, inv_scaler, lut);
      o = iq_order == 0 ? make_float2(a, b) : make_float2(b, a);
    }
    else
    {
      const float a = ingest_value(src + i * bytes, container, msb_first, inv_scaler, lut);
      o = iq_order == 2 ? make_float2(a, 0.0f) : make_float2(0.0f, a);
    }
    dst[i] = o;
  }
}

// Sample-rate conversion of the file readers without liquid-dsp (xml_reader.cpp:70-76,215-224; wav_reader.cpp:66-83,
// 196-206): every block of N = rate / 1000 input samples becomes 2048 output samples by linear interpolation,
//   out[2048 b + j] = x[b N + base_j + 1 - shift] * frac_j + x[b N + base_j - shift] * (1 - frac_j)
// (shift = 1 for the XML reader, whose buffer starts with the previous block's last sample and with 0 before the first
// block; 0 for the WAV reader). Two roundings per product and one per sum, as the scalar x86 code does it (no FMA).
__global__ void __launch_bounds__(256) k_resample_linear(const float2 * __restrict__ in, long long n_in, int block_in, int shift,
                                                         const short * __restrict__ base, const float * __restrict__ frac,
                                                         long long n_out, float2 * __restrict__ out)
{
  for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < n_out; o += (long long)gridDim.x * blockDim.x)
  {
    const long long b = o >> 11;
    const int j = (int)(o & 2047);
    const long long lo = b * block_in + base[j] - shift;
    const float r = frac[j], r1 = __fsub_rn(1.0f, r);
    const float2 hi_v = lo + 1 < n_in ? in[lo + 1] : make_float2(0.f, 0.f);
    const float2 lo_v = lo >= 0 ? in[lo] : make_float2(0.f, 0.f);
    out[o] = make_float2(__fadd_rn(__fmul_rn(hi_v.x, r), __fmul_rn(lo_v.x, r1)), __fadd_rn(__fmul_rn(hi_v.y, r), __fmul_rn(lo_v.y, r1)));
  }
}

template <typename F> cudaError_t dispatch_fmt(int fmt, F && f)
{
  switch (fmt)
  {
  case FMT_CF32: f(std::integral_constant<int, FMT_CF32>()); break;
  case FMT_U8: f(std::integral_constant<int, FMT_U8>()); break;
  case FMT_I16: f(std::integral_constant<int, FMT_I16>()); break;
  default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

inline int fft_grid(int n_items) { return n_items < N_SM * 4 ? n_items : N_SM * 4; }
} // namespace

// ------------------------------------------------------------------------------------------------ launchers
cudaError_t launch_init_ref_arg(cudaStream_t s, const DeviceTables & t, unsigned long long * lc)
{
  k_init_ref_arg<<<1, FFT_THREADS, 0, s>>>(t.w2048, t.prs, t.ref_arg_conj);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

cudaError_t launch_fft_batch(cudaStream_t s, const DeviceTables & t, const float2 * in, float2 * out, int n, int sign, unsigned long long * lc)
{
  if (n <= 0) return cudaSuccess;
  k_fft_batch<<<fft_grid(n), FFT_THREADS, 0, s>>>(in, out, n, sign, t.w2048);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

cudaError_t launch_fft_frames(cudaStream_t s, const DeviceTables & t, const FrameDesc * frames, int n_frames, const RecInput * recs, int fmt,
                              float2 * X, int max_ctas_per_sm, unsigned long long * lc)
{
  if (n_frames <= 0) return cudaSuccess;
  const int n_items = n_frames * X_ROWS;
  if (lc) (*lc)++;
  return dispatch_fmt(fmt, [&](auto F) {
    constexpr int FMT = decltype(F)::value;
    constexpr int stage = 2 * fft_stage_bytes<FMT>();
    const LaunchProps lp = launch_props((const void *)k_fft_frames<FMT>, FFT_THREADS, stage, stage); // per device: resident CTAs per SM of this instantiation
    int per_sm = lp.err == cudaSuccess && lp.ctas_per_sm > 0 ? lp.ctas_per_sm : 4;
    if (max_ctas_per_sm > 0) per_sm = std::min(per_sm, max_ctas_per_sm);
    k_fft_frames<FMT><<<std::min(n_items, lp.n_sm * per_sm), FFT_THREADS, stage, s>>>(frames, n_items, recs, t.w2048, t.fft_slot_w, t.fft_slot_r, X);
  });
}

cudaError_t launch_reorder_frames(cudaStream_t s, const DeviceTables & t, const float2 * fft_nat, int n_frames, float2 * X, unsigned long long * lc)
{
  if (n_frames <= 0) return cudaSuccess;
  k_reorder_frames<<<n_frames * X_ROWS, 256, 0, s>>>(fft_nat, n_frames * X_ROWS, t.bin_of_k, X);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

// exchange ring of the per-symbol sums (one word per warp of a recording and ring slot) + the ticket counter of k_demap5
size_t demap_ring_bytes(int n_work) { return sizeof(unsigned long long) * (size_t)std::max(n_work, 1) * DM3_RING * DM5_WARPS + 256; }
static size_t demap5_smem_bytes(int lag) { return sizeof(float4) * 2 * (size_t)(lag + 1 + DM5_PF) * DM5_T + sizeof(int) * (size_t)(lag + 1) * (DM5_T / 32); }
template <int LAG, bool QUAL> static const void * demap5_fn(int soft_bit_type)
{
  return soft_bit_type == 0 ? (const void *)k_demap5<0, LAG, QUAL> : (soft_bit_type == 1 ? (const void *)k_demap5<1, LAG, QUAL> : (const void *)k_demap5<2, LAG, QUAL>);
}
template <int LAG> static const void * demap5_fn(int soft_bit_type, bool qual) { return qual ? demap5_fn<LAG, true>(soft_bit_type) : demap5_fn<LAG, false>(soft_bit_type); }

cudaError_t launch_demap(cudaStream_t s, const DeviceTables & t, const DemapWork * work, int n_work, const FrameDesc * frames,
                         const uint8_t * null_is_tii, const float2 * X, OfdmStateDev * states, int soft_bit_type, int16_t * soft,
                         unsigned long long * ring, FrameQualSnap * qsnap, unsigned long long * lc)
{
  if (n_work <= 0) return cudaSuccess;
  if (soft_bit_type < 0 || soft_bit_type > 2) return cudaErrorInvalidValue;
  if (lc) (*lc)++;
  if (ring == nullptr) return cudaErrorInvalidValue;
  // symbols between a symbol's arithmetic and the write of its soft bits: the stash is (lag + 1) x 4 KB of shared memory per
  // CTA, so a shorter lag trades waiting on the slowest warp of a run against resident CTAs per SM (2 / 3 / 4 at lag 15 / 7 /
  // 3). Measured (profiles/README.md): 288 CTAs (96 recordings) 5.57 / 5.61 / 7.07 ms, 576 CTAs (192 segments) - / 7.83 / 6.08 ms:
  // the longest lag whose residency still holds the whole grid. DABSTAR_DEMAP_LAG = 3 | 7 | 15 overrides (A/B switch).
  static const int lag_env = getenv("DABSTAR_DEMAP_LAG") ? atoi(getenv("DABSTAR_DEMAP_LAG")) : 0;
  const int grid_ctas = n_work * DM5_SLICES;
  const int lag = lag_env == 3 || lag_env == 7 || lag_env == 15 ? lag_env : (grid_ctas <= 2 * N_SM ? 15 : (grid_ctas <= 3 * N_SM ? 7 : 3));
  const bool qual = qsnap != nullptr;
  const void * fn = lag == 3 ? demap5_fn<3>(soft_bit_type, qual) : (lag == 15 ? demap5_fn<15>(soft_bit_type, qual) : demap5_fn<7>(soft_bit_type, qual));
  const size_t smem = demap5_smem_bytes(lag);
  const LaunchProps lp = launch_props(fn, DM5_T, smem, smem); // opt-in for the dynamic shared memory, once per device
  if (lp.err != cudaSuccess) return lp.err;
  cudaError_t e = cudaMemsetAsync(ring, 0, demap_ring_bytes(n_work), s); // ring tags and the ticket counter
  if (e != cudaSuccess) return e;
  unsigned * ticket = reinterpret_cast<unsigned *>(reinterpret_cast<unsigned char *>(ring) + demap_ring_bytes(n_work) - 256);
  const int16_t * rel = t.rel_of_k;
  void * args[] = { (void *)&work, (void *)&frames, (void *)&null_is_tii, (void *)&X, (void *)&rel, (void *)&states, (void *)&soft, (void *)&ring, (void *)&ticket, (void *)&qsnap };
  return cudaLaunchKernel(fn, dim3((unsigned)(n_work * DM5_SLICES)), dim3(DM5_T), args, smem, s);
}

// The sums of the host's quality_from_state (engine.cu) over one snapshot, in its order and precision: serial float sums over
// k = 0..1535 and the double weighted sum of mMeanPowerOvrAll from k = 1535 down. The explicit roundings keep nvcc from
// contracting to FMA, so the figures the host forms from them equal those of the end-of-run state bit for bit.
__global__ void __launch_bounds__(128) k_frame_quality(const FrameDesc * __restrict__ frames, int n_frames, const FrameQualSnap * __restrict__ qsnap,
                                                       FrameQual * __restrict__ out)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_frames || frames[i].n_syms != 75) return; // a cut frame has no snapshot
  const FrameQualSnap & q = qsnap[i];
  double acc = 0.0, w = 1.0;
  for (int k = K_CARR - 1; k >= 0; k--)
  {
    acc = __dadd_rn(acc, __dmul_rn(w, (double)q.pow_acc[k]));
    w = __dmul_rn(w, 1.0 - POW_ALL_BETA);
  }
  float sum_noise = 0.0f, sd = 0.0f;
  for (int k = 0; k < K_CARR; k++)
  {
    sum_noise = __fadd_rn(sum_noise, q.null_pow[k]);
    sd = __fadd_rn(sd, q.stddev[k]);
  }
  out[frames[i].slot] = FrameQual{ sd, sum_noise, (float)__dadd_rn((double)q.pow_carry, __dmul_rn(POW_ALL_BETA, acc)), q.mean_value };
}

cudaError_t launch_frame_quality(cudaStream_t s, const FrameDesc * frames, int n_frames, const FrameQualSnap * qsnap, FrameQual * out, unsigned long long * lc)
{
  if (n_frames <= 0) return cudaSuccess;
  k_frame_quality<<<(n_frames + 127) / 128, 128, 0, s>>>(frames, n_frames, qsnap, out);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

cudaError_t launch_cp_corr(cudaStream_t s, const FrameDesc * frames, int n_frames, const RecInput * recs, int fmt, float2 * cp, unsigned long long * lc)
{
  if (n_frames <= 0) return cudaSuccess;
  if (lc) (*lc)++;
  // DABSTAR_CP_BULK=0: the direct-load kernel for 8-bit input too (read per launch: A/B measurements, and the parity test of the two)
  const char * ev = getenv("DABSTAR_CP_BULK");
  const bool bulk = ev == nullptr || atoi(ev) != 0;
  if (fmt == FMT_U8 && bulk)
  {
    const LaunchProps lp = launch_props((const void *)k_cp_corr_bulk, 256, CPB_SMEM, CPB_SMEM);
    if (lp.err != cudaSuccess) return lp.err;
    const int slots = lp.n_sm * (lp.ctas_per_sm > 0 ? lp.ctas_per_sm : 1);
    k_cp_corr_bulk<<<n_frames < slots ? n_frames : slots, 256, CPB_SMEM, s>>>(frames, n_frames, recs, cp);
    return cudaGetLastError();
  }
  const int grid = n_frames < N_SM * 8 ? n_frames : N_SM * 8;
  return dispatch_fmt(fmt, [&](auto F) { k_cp_corr<decltype(F)::value><<<grid, 256, 0, s>>>(frames, n_frames, recs, cp); });
}

cudaError_t launch_prs_corr(cudaStream_t s, const DeviceTables & t, const FrameDesc * frames, int n_frames, const RecInput * recs, int fmt,
                            float threshold_first, float threshold_rest, const uint8_t * first_flags, int strongest, int * start_index, unsigned long long * lc)
{
  if (n_frames <= 0) return cudaSuccess;
  if (lc) (*lc)++;
  return dispatch_fmt(fmt, [&](auto F) {
    k_prs_corr<decltype(F)::value><<<fft_grid(n_frames), FFT_THREADS, 0, s>>>(frames, n_frames, recs, t.w2048, t.prs, threshold_first, threshold_rest, first_flags, strongest, start_index);
  });
}

cudaError_t launch_coarse_afc(cudaStream_t s, const DeviceTables & t, const FrameDesc * frames, int n_frames, const RecInput * recs, int fmt,
                              int * offset_hz, unsigned long long * lc)
{
  if (n_frames <= 0) return cudaSuccess;
  if (lc) (*lc)++;
  return dispatch_fmt(fmt, [&](auto F) {
    k_coarse_afc<decltype(F)::value><<<fft_grid(n_frames), FFT_THREADS, 0, s>>>(frames, n_frames, recs, t.w2048, t.ref_arg_conj, offset_hz);
  });
}

cudaError_t launch_coarse_afc_raw(cudaStream_t s, const DeviceTables & t, const float2 * fft_nat, int n, int * offset_hz, unsigned long long * lc)
{
  if (n <= 0) return cudaSuccess;
  k_coarse_afc_raw<<<fft_grid(n), FFT_THREADS, 0, s>>>(fft_nat, n, t.w2048, t.ref_arg_conj, offset_hz);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

cudaError_t launch_ingest_convert(cudaStream_t s, const void * src, int container, int msb_first, int iq_order, float inv_scaler, const float * lut,
                                  long long n_samples, float2 * dst, unsigned long long * lc)
{
  if (n_samples <= 0) return cudaSuccess;
  const long long blocks = (n_samples + 255) / 256;
  k_ingest_convert<<<(unsigned)std::min<long long>(blocks, N_SM * 16), 256, 0, s>>>(static_cast<const unsigned char *>(src), container, msb_first, iq_order, inv_scaler, lut,
                                                                                    n_samples, dst);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

cudaError_t launch_fft_null(cudaStream_t s, const DeviceTables & t, const FrameDesc * frames, int n_frames, const RecInput * recs, int fmt, float2 * out,
                            unsigned long long * lc)
{
  if (n_frames <= 0) return cudaSuccess;
  if (lc) (*lc)++;
  return dispatch_fmt(fmt, [&](auto F) { k_fft_null<decltype(F)::value><<<fft_grid(n_frames), FFT_THREADS, 0, s>>>(frames, n_frames, recs, t.w2048, out); });
}

cudaError_t launch_resample_linear(cudaStream_t s, const float2 * in, long long n_in, int block_in, int shift, const short * base, const float * frac,
                                   long long n_out, float2 * out, unsigned long long * lc)
{
  if (n_out <= 0) return cudaSuccess;
  const long long blocks = (n_out + 255) / 256;
  k_resample_linear<<<(unsigned)std::min<long long>(blocks, N_SM * 16), 256, 0, s>>>(in, n_in, block_in, shift, base, frac, n_out, out);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

cudaError_t launch_dip_search(cudaStream_t s, const DipWork * work, int n, const RecInput * recs, int fmt, DipResult * out, unsigned long long * lc)
{
  if (n <= 0) return cudaSuccess;
  if (lc) (*lc)++;
  return dispatch_fmt(fmt, [&](auto F) { k_dip_search<decltype(F)::value><<<n, DIP_THREADS, 0, s>>>(work, recs, out); });
}
} // namespace dab
