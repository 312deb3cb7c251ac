// common.cuh — shared constants and small device helpers for the sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dab
{
// Mode-I constants (reference: common/glob_defs.h:40-55, common/dab_constants.h:55)
constexpr int L_SYMS = 76;
constexpr int K_CARR = 1536;
constexpr int T_U = 2048;
constexpr int T_G = 504;
constexpr int T_S = 2552;
constexpr int T_N = 2656;
constexpr int T_F = 196608;
constexpr int SYM_BITS = 3072;
constexpr int CIF_BITS = 55296;
constexpr int FRAME_SOFT = 75 * SYM_BITS;  // int16 soft bits per frame: symbols 1..75
constexpr int FIC_SOFT = 9216;             // symbols 1..3
constexpr int FIC_IN = 2304;
constexpr int FIC_OUT = 768;
constexpr int FS = 2048000;
constexpr int X_ROWS = 77;                 // symbol 0, 1..75, null
constexpr int N_SM = 148;

constexpr float PI_F = 3.14159265358979323846f;
constexpr float PI_2_F = 1.57079632679489661923f;
constexpr float PI_4_F = 0.78539816339744830962f;
constexpr float TWO_PI_F = 6.28318530717958647692f;
constexpr float RAD_PER_DEG_F = 0.01745329251994329577f;

enum { FMT_CF32 = 0, FMT_U8 = 1, FMT_I16 = 2 };

// Complex arithmetic. On the device these are the packed FP32 instructions of sm_100 (FADD2 / FMUL2 / FFMA2 work on an
// aligned register pair = one complex number; an operand may be a broadcast scalar or have its halves swapped for free),
// so a complex add is ONE instruction and a complex multiply three (two with a prepared constant). The host versions
// (index-arithmetic tests) are the plain formulas; results differ by rounding only (FMA contraction).
#if defined(__CUDA_ARCH__) && __CUDA_ARCH__ >= 1000
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ float2 cmul(float2 a, float2 b)
{
  const float2 t = __fmul2_rn(a, make_float2(b.x, b.x));                           // (a.x b.x, a.y b.x)
  const float2 u = __fmul2_rn(make_float2(a.y, a.x), make_float2(b.y, b.y));       // (a.y b.y, a.x b.y)
  return __ffma2_rn(u, make_float2(-1.0f, 1.0f), t);
}
__device__ __forceinline__ float2 cmul_conj(float2 a, float2 b) // a * conj(b)
{
  const float2 t = __fmul2_rn(a, make_float2(b.x, b.x));                           // (a.x b.x, a.y b.x)
  const float2 u = __fmul2_rn(make_float2(a.y, a.x), make_float2(b.y, b.y));       // (a.y b.y, a.x b.y)
  return __ffma2_rn(u, make_float2(1.0f, -1.0f), t);
}
// a * (c + j s) for a compile-time constant: (a.x c - a.y s, a.y c + a.x s) = a * c + swap(a) * (-s, s)
__device__ __forceinline__ float2 cmul_const(float2 a, float c, float s)
{
  return __ffma2_rn(make_float2(a.y, a.x), make_float2(-s, s), __fmul2_rn(a, make_float2(c, c)));
}
// -j a
__device__ __forceinline__ float2 cmul_mj(float2 a) { return __fmul2_rn(make_float2(a.y, a.x), make_float2(1.0f, -1.0f)); }
// a - j b and a + j b
__device__ __forceinline__ float2 csub_j(float2 a, float2 b) { return __ffma2_rn(make_float2(b.y, b.x), make_float2(1.0f, -1.0f), a); }
__device__ __forceinline__ float2 cadd_j(float2 a, float2 b) { return __ffma2_rn(make_float2(b.y, b.x), make_float2(-1.0f, 1.0f), a); }
#else
__host__ __device__ inline float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__host__ __device__ inline float2 cmul_conj(float2 a, float2 b) { return make_float2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y); } // a * conj(b)
__host__ __device__ inline float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__host__ __device__ inline float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__host__ __device__ inline float2 cmul_const(float2 a, float c, float s) { return cmul(a, make_float2(c, s)); }
__host__ __device__ inline float2 cmul_mj(float2 a) { return make_float2(a.y, -a.x); }
__host__ __device__ inline float2 csub_j(float2 a, float2 b) { return make_float2(a.x + b.y, a.y - b.x); }
__host__ __device__ inline float2 cadd_j(float2 a, float2 b) { return make_float2(a.x - b.y, a.y + b.x); }
#endif

// One frame of one recording as the kernels see it. Built on the host by the control loop (decoder.cu),
// which restates DabProcessor's AFC/clock bookkeeping (main/dab_processor.cpp:191-265).
// Oscillator convention (ofdm/sample_reader.cpp:276-281): for every sample read, phase = (phase - f) mod FS
// first, then out = v * e^{j 2 pi phase / FS}. ph_* is the phase BEFORE the first sample of the segment.
struct FrameDesc
{
  long long sym0;      // sample index (within the recording) of the first useful sample of symbol 0
  long long eval;      // sample index of the 2048-sample window handed to the PRS correlator
  int rec;             // recording index
  int slot;            // persistent frame slot in the soft-bit / FIB buffers (global index over all recordings)
  int xslot;           // row block of this frame in the window's spectrum buffer X
  int f_sym0, ph_eval; // integer Hz and oscillator phase before sample `eval`
  int f_data, ph_data; // ... before the first sample of symbol 1 (its cyclic prefix)
  int f_null, ph_null; // ... before the first sample of the null symbol
  float clock_err;     // iClockErr handed to decode_symbol in this frame
  int n_syms;          // data symbols available (75 unless the recording ends inside the frame)
  int pad;
};

struct RecInput
{
  const void * iq;     // device pointer, interleaved I,Q in `fmt`
  long long n;         // samples
};
} // namespace dab
