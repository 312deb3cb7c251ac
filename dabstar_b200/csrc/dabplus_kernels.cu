// dabplus_kernels.cu — DAB+ outer code on the GPU: Reed-Solomon RS(120,110) over GF(2^8), Fire code, access-unit CRCs.
//
// Reference (SURVEY.md section 8f.2): Mp4Processor::add_to_frame / _process_reed_solomon_frame / _process_super_frame
// (backend/audio/mp4processor.cpp:95-334), ReedSolomon(8, 0435, 0, 1, 10)::dec(.., 135) (backend/reed_solomon.cpp:140-440,
// backend/galois.cpp:36-143), FirecodeChecker (backend/firecode_checker.cpp:41-184), check_crc_bytes (backend/crc.cpp:75-96).
//
// The reference walks the logical frames of a sub-channel one by one: a five-frame window is tested with the Fire code,
// decoded (bit_rate / 8 interleaved code words), dissected into access units, and the outcome decides where the next
// window starts. That dependency is handled by speculation, as the decoder handles frame positions: the walk of the
// synchronisation state machine (dabplus.cuh) runs on the device, one thread per stream, taking every window it has no
// outcome for as a success; only the windows it attempts are decoded, and walk and decode alternate until a walk attempts
// nothing new (engine.cu: run_dabplus). A stream keeps its five-frame stride through single failures, so the first walk is
// final unless synchronisation runs out. The Reed-Solomon decoder restates the reference's own sequence (Horner syndromes
// with its zero shortcut, its Berlekamp-Massey variant, Chien search, Forney with the same early exits), because the
// corrected bytes are handed on whatever the decoder returns: uncorrectable words leave with whatever corrections were
// applied before the decoder gave up.
#include "kernels.h"
#include "dabplus.cuh"
#include "stream_search.cuh"

#include <cstring>
#include <vector>

namespace dab
{
namespace
{
constexpr int RS_NN = 255, RS_ROOTS = 10, RS_PAD = 135, RS_DATA = 110, RS_LEN = 120;

struct GfTables
{
  uint8_t exp[256], log[256]; // log[0] = 255 stands for log(0), exp[255] = 0
  uint16_t fc[256];           // Fire code CRC table, polynomial 0x782f
  uint8_t mulr[10][256];      // mulr[r][x] = x alpha^r (syndrome Horner steps)
};

__host__ __device__ inline int gf_modnn(int x)
{
  while (x >= RS_NN) { x -= RS_NN; x = (x >> 8) + (x & RS_NN); }
  return x;
}
__host__ __device__ inline unsigned gf_mul(const GfTables & t, unsigned a, unsigned b) { return (a == 0 || b == 0) ? 0u : t.exp[gf_modnn(t.log[a] + t.log[b])]; }
__host__ __device__ inline unsigned gf_div(const GfTables & t, unsigned a, unsigned b) { return a == 0 ? 0u : t.exp[gf_modnn(RS_NN + t.log[a] - t.log[b])]; }
__host__ __device__ inline int gf_pow_power(int a, int n) { return a == 0 ? 0 : (a * n) % RS_NN; }

// Fire code remainder over x[2..10] then x[0..1] (firecode_checker.cpp:142-156)
__host__ __device__ inline unsigned fire_crc(const GfTables & t, const uint8_t * x)
{
  unsigned crc = 0;
  for (int i = 2; i < 11; i++) crc = ((crc << 8) ^ t.fc[(crc >> 8) ^ x[i]]) & 0xffffu;
  for (int i = 0; i < 2; i++) crc = ((crc << 8) ^ t.fc[(crc >> 8) ^ x[i]]) & 0xffffu;
  return crc;
}

// One code word: syn[] are its ten syndromes (not all zero). Corrections go to out[pos * stride] for data positions.
// Returns what ReedSolomon::dec returns: number of corrected symbols, or -1.
__device__ int rs_correct(const GfTables & t, const uint8_t (&syn)[RS_ROOTS], uint8_t * out, int stride)
{
  uint8_t lambda[RS_ROOTS + 1], root_tab[RS_ROOTS], loc_tab[RS_ROOTS], omega[RS_ROOTS + 1];
  int deg_lambda = 0;
  {
    // Berlekamp-Massey as ReedSolomon::computeLambda runs it (ten coefficients, corrector shifted every round)
    uint8_t corr[RS_ROOTS], old[RS_ROOTS];
    unsigned K = 1, L = 0;
    for (int i = 0; i < RS_ROOTS; i++) { corr[i] = 0; lambda[i] = 0; }
    lambda[RS_ROOTS] = 0;
    unsigned error = syn[0];
    lambda[0] = 1;
    corr[1] = 1;
    while (K < RS_ROOTS)
    {
      for (int i = 0; i < RS_ROOTS; i++) old[i] = lambda[i];
      for (int i = 0; i < RS_ROOTS; i++) lambda[i] ^= (uint8_t)gf_mul(t, error, corr[i]);
      if (2 * L < K && error != 0)
      {
        L = K - L;
        for (int i = 0; i < RS_ROOTS; i++) corr[i] = (uint8_t)gf_div(t, old[i], error);
      }
      for (int i = RS_ROOTS - 1; i >= 1; i--) corr[i] = corr[i - 1];
      corr[0] = 0;
      error = syn[K];
      for (unsigned i = 1; i <= K; i++) error ^= gf_mul(t, syn[K - i], lambda[i]);
      K++;
    }
    for (int i = 0; i < RS_ROOTS; i++) lambda[i] ^= (uint8_t)gf_mul(t, error, corr[i]);
    for (int i = 0; i < RS_ROOTS; i++) { if (lambda[i] != 0) deg_lambda = i; lambda[i] = t.log[lambda[i]]; }
  }
  int root_count = 0;
  {
    // Chien search over all 255 positions (computeErrors, iprim = 1: location = index - 1)
    uint8_t work[RS_ROOTS + 1];
    for (int i = 0; i <= RS_ROOTS; i++) work[i] = lambda[i];
    for (int i = 1; i <= RS_NN; i++)
    {
      unsigned result = 1;
      for (int j = deg_lambda; j > 0; j--)
        if (work[j] != RS_NN)
        {
          work[j] = (uint8_t)gf_modnn(work[j] + j);
          result ^= t.exp[work[j]];
        }
      if (result != 0) continue;
      if (root_count < RS_ROOTS) { root_tab[root_count] = (uint8_t)i; loc_tab[root_count] = (uint8_t)(i - 1); }
      root_count++;
    }
    if (root_count != deg_lambda) return -1;
  }
  int deg_omega = 0;
  for (int i = 0; i < RS_ROOTS; i++)
  {
    unsigned tmp = 0;
    for (int j = deg_lambda < i ? deg_lambda : i; j >= 0; j--)
      if (t.log[syn[i - j]] != RS_NN && lambda[j] != RS_NN) tmp ^= t.exp[gf_modnn(t.log[syn[i - j]] + lambda[j])];
    if (tmp != 0) deg_omega = i;
    omega[i] = t.log[tmp];
  }
  omega[RS_ROOTS] = RS_NN;
  for (int j = root_count - 1; j >= 0; j--)
  {
    unsigned num1 = 0;
    for (int i = deg_omega; i >= 0; i--)
      if (omega[i] != RS_NN) num1 ^= t.exp[gf_modnn(omega[i] + gf_pow_power(i, root_tab[j]))];
    const unsigned num2 = t.exp[gf_modnn(gf_pow_power(root_tab[j], RS_NN - 1) + RS_NN)];
    unsigned den = 0;
    for (int i = (deg_lambda < RS_ROOTS - 1 ? deg_lambda : RS_ROOTS - 1) & ~1; i >= 0; i -= 2)
      if (lambda[i + 1] != RS_NN) den ^= t.exp[gf_modnn(lambda[i + 1] + gf_pow_power(i, root_tab[j]))];
    if (den == 0) return -1;
    if (num1 != 0)
    {
      if (loc_tab[j] >= RS_NN - RS_ROOTS) root_count--;
      else
      {
        int e = gf_modnn(t.log[num1] + t.log[num2]);
        e = gf_modnn(e + (RS_NN - t.log[den]));
        const int pos = (int)loc_tab[j] - RS_PAD; // positions inside the 135 leading zeros are "corrected" in the reference's scratch block only
        if (pos >= 0) out[(size_t)pos * stride] ^= t.exp[e];
      }
    }
  }
  return root_count;
}

__device__ inline void load_tables(GfTables & t, const GfTables * __restrict__ tabs)
{
  for (int i = threadIdx.x; i < (int)(sizeof(GfTables) / 4); i += blockDim.x) reinterpret_cast<unsigned *>(&t)[i] = reinterpret_cast<const unsigned *>(tabs)[i];
  __syncthreads();
}

// thread = window of any stream: the Fire code on its raw header
__global__ void __launch_bounds__(128) k_dabplus_scan(const DabplusStream * __restrict__ st, int n_streams, long long n_windows, const GfTables * __restrict__ tabs,
                                                      uint8_t * __restrict__ state)
{
  __shared__ GfTables t;
  load_tables(t, tabs);
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_windows) return;
  const DabplusStream & s = st[find_stream(st, n_streams, g, [](const DabplusStream & x) { return x.win0; })];
  const uint8_t * raw = s.src + (size_t)(g - s.win0) * 3 * s.bit_rate;
  state[g] = fire_crc(t, raw) == 0 ? SF_PRE_OK : 0;
}

// thread = stream: the processor's walk over what is known; attempted windows without an outcome are appended to the decode list
__global__ void __launch_bounds__(128) k_dabplus_walk(const DabplusStream * __restrict__ st, int n_streams, const uint8_t * __restrict__ state, int * __restrict__ att,
                                                      DabplusMeta * __restrict__ meta, int * __restrict__ att_n, DabplusEntry * __restrict__ list, int * __restrict__ slot)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_streams) return;
  const DabplusStream & s = st[i];
  const uint8_t * sw = state + s.win0;
  int * a = att + s.att0;
  const int n = superframe_walk(sw, s.n_frames, a);
  att_n[i] = n;
  int todo = 0;
  for (int k = 0; k < n; k++) todo += (sw[a[k]] & SF_DECODED) ? 0 : 1;
  if (todo == 0) return;
  const long long sf_bytes = 110LL * (s.bit_rate / 8);
  unsigned long long e = atomicAdd(&meta->entries, (unsigned long long)todo);
  unsigned long long b = atomicAdd(&meta->bytes, (unsigned long long)todo * sf_bytes);
  for (int k = 0; k < n; k++)
  {
    if (sw[a[k]] & SF_DECODED) continue;
    list[e] = DabplusEntry{ b, i, a[k] };
    slot[s.win0 + a[k]] = (int)e;
    e++;
    b += sf_bytes;
  }
}

// thread = (listed window, code word j < 24): gather with the super-frame interleave, decode, scatter the 110 data bytes
__global__ void __launch_bounds__(128) k_dabplus_rs(const DabplusStream * __restrict__ st, const DabplusEntry * __restrict__ list, int n_list, const GfTables * __restrict__ tabs,
                                                    uint8_t * __restrict__ payload, int8_t * __restrict__ ler)
{
  __shared__ GfTables t;
  load_tables(t, tabs);
  const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (long long)n_list * DABPLUS_MAX_RS_DIMS) return;
  const int e = (int)(id / DABPLUS_MAX_RS_DIMS), j = (int)(id - (long long)e * DABPLUS_MAX_RS_DIMS);
  const DabplusEntry le = list[e];
  const DabplusStream & s = st[le.stream];
  const int rs_dims = s.bit_rate / 8;
  if (j >= rs_dims) return;
  const uint8_t * in = s.src + (size_t)le.window * 3 * s.bit_rate + j; // byte k of the code word at in[k * rs_dims]
  uint8_t * out = payload + le.pay_off + j;                            // mOutVec[j + k * rs_dims]
  // Horner for the ten roots alpha^0..alpha^9 in one pass; the 135 leading zeros leave every accumulator at zero.
  // mulr[r][x] = x alpha^r (mulr[r][0] = 0) is the reference's  s == 0 ? d : d ^ exp[modnn(log[s] + r)]  in one lookup.
  unsigned s_[RS_ROOTS];
#pragma unroll
  for (int r = 0; r < RS_ROOTS; r++) s_[r] = 0;
  for (int k = 0; k < RS_LEN; k++)
  {
    const unsigned d = in[(size_t)k * rs_dims];
    if (k < RS_DATA) out[(size_t)k * rs_dims] = (uint8_t)d;
#pragma unroll
    for (int r = 0; r < RS_ROOTS; r++) s_[r] = d ^ t.mulr[r][s_[r]];
  }
  uint8_t syn[RS_ROOTS];
  unsigned any = 0;
#pragma unroll
  for (int r = 0; r < RS_ROOTS; r++) { syn[r] = (uint8_t)s_[r]; any |= s_[r]; }
  ler[id] = any == 0 ? (int8_t)0 : (int8_t)rs_correct(t, syn, out, rs_dims);
}

// thread = listed window: Fire code on the raw and on the decoded super-frame header, header fields, access-unit CRCs
__global__ void __launch_bounds__(128) k_dabplus_check(const DabplusStream * __restrict__ st, const DabplusEntry * __restrict__ list, int n_list, const GfTables * __restrict__ tabs,
                                                       const uint16_t * __restrict__ fc_syn, uint8_t * __restrict__ payload, const int8_t * __restrict__ ler,
                                                       SuperFrameRec * __restrict__ rec, uint8_t * __restrict__ state)
{
  __shared__ GfTables t;
  load_tables(t, tabs);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_list) return;
  const DabplusEntry le = list[e];
  const DabplusStream & s = st[le.stream];
  const int rs_dims = s.bit_rate / 8, w = le.window;
  SuperFrameRec r;
  memset(&r, 0, sizeof(r));
  r.first_frame = w;
  const uint8_t * raw = s.src + (size_t)w * 3 * s.bit_rate;
  uint8_t * o = payload + le.pay_off;
  const int sf_bytes = RS_DATA * rs_dims;
  r.pre_ok = fire_crc(t, raw) == 0;                       // FirecodeChecker::check on the undecoded block (mp4processor.cpp:133)
  for (int j = 0; j < rs_dims; j++)
  {
    const int l = ler[(size_t)e * DABPLUS_MAX_RS_DIMS + j];
    if (l < 0) r.rs_errors++; else r.rs_corrections += l;
  }
  // check_and_correct_6bits on the decoded header (firecode_checker.cpp:166-184)
  uint8_t x[11];
  for (int i = 0; i < 11; i++) x[i] = o[i];
  const unsigned syn = fire_crc(t, x);
  bool ok = syn == 0;
  if (!ok)
  {
    const unsigned e = fc_syn[syn];
    if (e & 0xffu)
    {
      const int bit = (int)(e >> 8);
      x[bit / 8] ^= (uint8_t)((e & 0xffu) >> (bit % 8));
      x[bit / 8 + 1] ^= (uint8_t)((e & 0xffu) << (8 - (bit % 8)));
      for (int i = 0; i < 11; i++) o[i] = x[i];
      ok = true;
    }
  }
  r.ok = ok;
  if (ok)
  {
    bool diff = false;
    for (int i = 0; i < 11; i++) diff = diff || (x[i] != raw[i]);
    r.fc_corrected = diff;
    r.dac_rate = (x[2] >> 6) & 1; r.sbr_flag = (x[2] >> 5) & 1; r.aac_channel_mode = (x[2] >> 4) & 1; r.ps_flag = (x[2] >> 3) & 1; r.mpeg_surround = x[2] & 7;
    int * a = r.au_start;
    switch (2 * r.dac_rate + r.sbr_flag)
    {
    case 0: r.num_aus = 4; a[0] = 8; a[1] = x[3] * 16 + (x[4] >> 4); a[2] = (x[4] & 0xf) * 256 + x[5]; a[3] = x[6] * 16 + (x[7] >> 4); a[4] = sf_bytes; break;
    case 1: r.num_aus = 2; a[0] = 5; a[1] = x[3] * 16 + (x[4] >> 4); a[2] = sf_bytes; break;
    case 2: r.num_aus = 6; a[0] = 11; a[1] = x[3] * 16 + (x[4] >> 4); a[2] = (x[4] & 0xf) * 256 + x[5]; a[3] = x[6] * 16 + (x[7] >> 4);
            a[4] = (x[7] & 0xf) * 256 + x[8]; a[5] = x[9] * 16 + (x[10] >> 4); a[6] = sf_bytes; break;
    default: r.num_aus = 3; a[0] = 6; a[1] = x[3] * 16 + (x[4] >> 4); a[2] = (x[4] & 0xf) * 256 + x[5]; a[3] = sf_bytes; break;
    }
    for (int u = 0; u < r.num_aus; u++)
    {
      const int len = a[u + 1] - a[u] - 2;
      if (len > 960 || len < 0) { r.au_state[u] = 0; continue; }     // mp4processor.cpp:326
      if (a[u] + len + 2 > sf_bytes) { r.au_state[u] = 2; continue; } // would leave the super-frame
      unsigned crc = 0xffffu;                                         // calc_crc: 0x1021, all ones, complemented (crc.cpp:75-86)
      for (int i = 0; i < len; i++)
      {
        crc ^= (unsigned)o[a[u] + i] << 8;
        for (int b = 0; b < 8; b++) crc = (crc & 0x8000u) ? ((crc << 1) ^ 0x1021u) : (crc << 1);
        crc &= 0xffffu;
      }
      crc = ~crc & 0xffffu;
      r.au_state[u] = crc == (((unsigned)o[a[u] + len] << 8) | o[a[u] + len + 1]) ? 1 : 2;
    }
  }
  rec[e] = r;
  state[s.win0 + w] |= (uint8_t)(SF_DECODED | (ok ? SF_OK : 0));
}

// block = output record: the attempted windows' records and super-frames in stream order
__global__ void __launch_bounds__(128) k_dabplus_compact(const DabplusStream * __restrict__ st, int n_streams, const int * __restrict__ att, const int * __restrict__ slot,
                                                         const DabplusEntry * __restrict__ list, const SuperFrameRec * __restrict__ rec, const uint8_t * __restrict__ payload,
                                                         SuperFrameRec * __restrict__ out_rec, uint8_t * __restrict__ out_pay)
{
  const long long k = blockIdx.x;
  const int si = find_stream(st, n_streams, k, [](const DabplusStream & x) { return x.out_rec0; });
  const DabplusStream & s = st[si];
  const int i = (int)(k - s.out_rec0);
  const int e = slot[s.win0 + att[s.att0 + i]];
  const int sf_bytes = RS_DATA * (s.bit_rate / 8);
  const uint8_t * src = payload + list[e].pay_off;
  uint8_t * dst = out_pay + s.out_pay0 + (long long)i * sf_bytes;
  for (int b = threadIdx.x; b < sf_bytes; b += blockDim.x) dst[b] = src[b];
  if (threadIdx.x == 0) out_rec[k] = rec[e];
}
} // namespace

// Host side of the tables: GF(2^8) with generator 0435 (galois.cpp:36-62), Fire code CRC table and the 65536-entry
// burst syndrome table, filled in the reference's order so that the FIRST burst producing a syndrome is kept
// (firecode_checker.cpp:46-140, pattern list firecode_checker.h:57-70).
void dabplus_host_tables(std::vector<uint8_t> & gf_blob, std::vector<uint16_t> & fc_syn)
{
  GfTables t;
  memset(&t, 0, sizeof(t));
  unsigned sr = 1;
  t.log[0] = RS_NN;
  t.exp[RS_NN] = 0;
  for (int i = 0; i < RS_NN; i++)
  {
    t.log[sr] = (uint8_t)i;
    t.exp[i] = (uint8_t)sr;
    sr <<= 1;
    if (sr & 0x100) sr ^= 0x11D;
    sr &= 0xff;
  }
  for (int i = 0; i < 256; i++)
  {
    unsigned crc = (unsigned)i << 8;
    for (int j = 0; j < 8; j++) crc = (crc & 0x8000u) ? ((crc << 1) ^ 0x782fu) : (crc << 1);
    t.fc[i] = (uint16_t)crc;
  }
  for (int r = 0; r < RS_ROOTS; r++)
    for (int x = 0; x < 256; x++) t.mulr[r][x] = x == 0 ? 0 : t.exp[gf_modnn(t.log[x] + r)];
  gf_blob.resize(sizeof(t));
  memcpy(gf_blob.data(), &t, sizeof(t));
  // burst patterns of up to 6 bits, grouped by the bit shifts they are tried at
  static const uint8_t P[124] = {
    17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 30, 31, 34, 36, 38, 40, 42, 44, 46, 50, 52, 54, 56, 60, 62, 68, 72, 76, 84, 88, 92, 100, 104, 108, 120, 124, 136, 152, 168,
    184, 200, 216, 248, 33, 35, 37, 39, 41, 43, 45, 49, 51, 53, 55, 57, 59, 61, 63, 66, 70, 74, 78, 82, 86, 90, 98, 102, 106, 110, 114, 118, 122, 126, 132, 140, 148, 156,
    164, 172, 180, 196, 204, 212, 220, 228, 236, 244, 252, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 29, 32, 48, 58, 64, 80, 96, 112, 116, 128, 144, 160, 176, 192,
    208, 224, 232, 240 };
  fc_syn.assign(65536, 0);
  uint8_t e[11] = { 0 };
  const struct { int shift, first, last, bytes; } pass[4] = { { 0, 0, 124, 11 }, { 4, 0, 45, 10 }, { 2, 45, 75, 10 }, { 6, 60, 90, 10 } };
  for (const auto & ps : pass)
    for (int i = 0; i < ps.bytes; i++)
      for (int j = ps.first; j < ps.last; j++)
      {
        if (ps.shift == 0) e[i] = P[j];
        else { e[i] = (uint8_t)(P[j] >> ps.shift); e[i + 1] = (uint8_t)(P[j] << (8 - ps.shift)); }
        const unsigned s = fire_crc(t, e);
        if (fc_syn[s] == 0) fc_syn[s] = (uint16_t)(((i * 8 + ps.shift) << 8) + P[j]);
        e[i] = 0;
        if (ps.shift != 0) e[i + 1] = 0;
      }
}

cudaError_t launch_dabplus_scan(cudaStream_t s, const DabplusStream * st, int n_streams, long long n_windows, const void * gf_tables, uint8_t * state, unsigned long long * lc)
{
  if (n_windows <= 0) return cudaSuccess;
  k_dabplus_scan<<<(unsigned)((n_windows + 127) / 128), 128, 0, s>>>(st, n_streams, n_windows, static_cast<const GfTables *>(gf_tables), state);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

cudaError_t launch_dabplus_walk(cudaStream_t s, const DabplusStream * st, int n_streams, const uint8_t * state, int * att, DabplusMeta * meta, int * att_n,
                                DabplusEntry * list, int * slot, unsigned long long * lc)
{
  if (n_streams <= 0) return cudaSuccess;
  k_dabplus_walk<<<(n_streams + 127) / 128, 128, 0, s>>>(st, n_streams, state, att, meta, att_n, list, slot);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

cudaError_t launch_dabplus_decode(cudaStream_t s, const DabplusStream * st, const DabplusEntry * list, int n_list, const void * gf_tables, const uint16_t * fc_syn,
                                  uint8_t * payload, int8_t * ler, SuperFrameRec * rec, uint8_t * state, unsigned long long * lc)
{
  if (n_list <= 0) return cudaSuccess;
  const GfTables * t = static_cast<const GfTables *>(gf_tables);
  const long long words = (long long)n_list * DABPLUS_MAX_RS_DIMS;
  k_dabplus_rs<<<(unsigned)((words + 127) / 128), 128, 0, s>>>(st, list, n_list, t, payload, ler);
  k_dabplus_check<<<(n_list + 127) / 128, 128, 0, s>>>(st, list, n_list, t, fc_syn, payload, ler, rec, state);
  if (lc) (*lc) += 2;
  return cudaGetLastError();
}

cudaError_t launch_dabplus_compact(cudaStream_t s, const DabplusStream * st, int n_streams, long long n_out, const int * att, const int * slot, const DabplusEntry * list,
                                   const SuperFrameRec * rec, const uint8_t * payload, SuperFrameRec * out_rec, uint8_t * out_pay, unsigned long long * lc)
{
  if (n_out <= 0) return cudaSuccess;
  k_dabplus_compact<<<(unsigned)n_out, 128, 0, s>>>(st, n_streams, att, slot, list, rec, payload, out_rec, out_pay);
  if (lc) (*lc)++;
  return cudaGetLastError();
}
} // namespace dab
