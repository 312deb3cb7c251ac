// pfec_kernels.cu — packet-mode FEC of DAB sub-channels on the GPU: the FEC frames of every stream located, and the 12 rows of
// each RS(204,188)-corrected, before the packet pass walks the corrected bytes (engine.cu: run_packet_fec).
//
// Every slot decides on its own whether an FEC-packet run starts there (pfec.cuh: pfec_run_start over the fit codes of its
// neighbours), so locating needs no walk: k_pfec_code and k_pfec_start take one thread per slot. k_pfec_list compacts each
// stream's runs in stream order with a block-wide scan (block_scan.cuh) and marks their slots in the FEC mask the packet scan
// reads. k_pfec_correct gives every frame 16 lanes, 12 of which decode one row each with per-root syndrome tables in shared
// memory; a row with more than 8 errors is left as received.
#include "kernels.h"
#include "stream_search.cuh"
#include "block_scan.cuh"

#include <cstring>
#include <vector>

namespace dab
{
namespace
{
__device__ inline long long pfec_slots(const PfecStream & s) { return (long long)s.n_frames * (s.bit_rate / 8); }

// thread = slot of any stream: its fit code
__global__ void __launch_bounds__(256) k_pfec_code(const PfecStream * __restrict__ st, int n_streams, long long n_slots, uint8_t * __restrict__ code)
{
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_slots) return;
  const PfecStream & s = st[find_stream(st, n_streams, g, [](const PfecStream & x) { return x.slot0; })];
  code[g] = (uint8_t)pfec_slot_code(s.src + (g - s.slot0) * PFEC_SLOT);
}

// thread = slot of any stream: does a run start there
__global__ void __launch_bounds__(256) k_pfec_start(const PfecStream * __restrict__ st, int n_streams, long long n_slots, const uint8_t * __restrict__ code,
                                                    uint8_t * __restrict__ start)
{
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_slots) return;
  const PfecStream & s = st[find_stream(st, n_streams, g, [](const PfecStream & x) { return x.slot0; })];
  start[g] = pfec_run_start(code + s.slot0, pfec_slots(s), g - s.slot0) ? 1 : 0;
}

// runs before a chunk and the last of them (-1 none)
struct PfecCarry
{
  int count, last;
};
__device__ inline PfecCarry pfec_then(PfecCarry a, PfecCarry b) { return PfecCarry{ a.count + b.count, b.last >= 0 ? b.last : a.last }; }

constexpr int PFEC_LIST_THREADS = 256;
// block = stream
__global__ void __launch_bounds__(PFEC_LIST_THREADS) k_pfec_list(const PfecStream * __restrict__ st, const uint8_t * __restrict__ code,
                                                                 const uint8_t * __restrict__ start, PfecStage * __restrict__ stage, int * __restrict__ cnt,
                                                                 uint8_t * __restrict__ mask)
{
  __shared__ PfecCarry sh[32];
  const PfecStream & s = st[blockIdx.x];
  const int n = (int)pfec_slots(s), per = (n + (int)blockDim.x - 1) / (int)blockDim.x;
  const int i0 = min(n, (int)threadIdx.x * per), i1 = min(n, i0 + per);
  const uint8_t * sc = code + s.slot0;
  const uint8_t * ss = start + s.slot0;
  PfecCarry mine{ 0, -1 };
  for (int i = i0; i < i1; i++)
    if (ss[i]) { mine.count++; mine.last = i; }
  PfecCarry total;
  const PfecCarry in = block_exclusive_scan(mine, PfecCarry{ 0, -1 }, pfec_then, sh, &total);
  int k = in.count, prev = in.last;
  for (int i = i0; i < i1; i++)
  {
    if (!ss[i]) continue;
    stage[s.stage0 + k++] = PfecStage{ i, pfec_score(sc, n, i), pfec_incomplete(i, prev, n) ? 1 : 0 };
    prev = i;
    for (int j = i; j < i + PFEC_RUN && j < n; j++) mask[s.slot0 + j] = 1;
  }
  if (threadIdx.x == 0) cnt[blockIdx.x] = total.count;
}

constexpr int PFEC_LANES = 16; // per frame: one row each for lanes 0..11
constexpr int PFEC_CORRECT_THREADS = 128;
// 16 lanes = output frame: its 12 rows decoded and corrected, then (lane 0) its record
__global__ void __launch_bounds__(PFEC_CORRECT_THREADS) k_pfec_correct(const PfecStream * __restrict__ st, int n_streams, long long n_out,
                                                                       const PfecTables * __restrict__ tabs, const PfecStage * __restrict__ stage,
                                                                       PfecRec * __restrict__ rec)
{
  __shared__ PfecTables t;
  for (int i = threadIdx.x; i < (int)(sizeof(PfecTables) / 4); i += blockDim.x) reinterpret_cast<unsigned *>(&t)[i] = reinterpret_cast<const unsigned *>(tabs)[i];
  __syncthreads();
  const long long k = (long long)blockIdx.x * (PFEC_CORRECT_THREADS / PFEC_LANES) + threadIdx.x / PFEC_LANES;
  const int r = threadIdx.x % PFEC_LANES;
  if (k >= n_out) return; // all 16 lanes of a frame leave together
  const PfecStream & s = st[find_stream(st, n_streams, k, [](const PfecStream & x) { return x.out0; })];
  const PfecStage g = stage[s.stage0 + (k - s.out0)];
  int fixed = 0, failed = 0, bytes = 0;
  if (!g.incomplete && r < PFEC_ROWS)
  {
    int col[PFEC_T];
    uint8_t val[PFEC_T];
    const uint8_t * src = s.src;
    const long long run = g.run;
    const int m = pfec_row_decode(t, [&](int c) { return (unsigned)src[pfec_byte(run, r, c)]; }, col, val);
    if (m < 0) failed = 1;
    else if (m > 0)
    {
      fixed = 1;
      bytes = m;
      for (int i = 0; i < m; i++) s.dst[pfec_byte(run, r, col[i])] ^= val[i];
    }
  }
  const unsigned grp = 0xffffu << (threadIdx.x & 16);
  for (int d = 1; d < PFEC_LANES; d <<= 1)
  {
    fixed += __shfl_xor_sync(grp, fixed, d, PFEC_LANES);
    failed += __shfl_xor_sync(grp, failed, d, PFEC_LANES);
    bytes += __shfl_xor_sync(grp, bytes, d, PFEC_LANES);
  }
  if (r) return;
  const int n = s.n_frames * (s.bit_rate / 8), spf = s.bit_rate / 8;
  PfecRec o;
  o.first_slot = g.run - PFEC_ADT_SLOTS;
  o.run_slot = g.run;
  o.first_frame = max(0, o.first_slot) / spf;
  o.last_frame = (min(g.run + PFEC_RUN, n) - 1) / spf;
  o.status = g.incomplete ? PFEC_INCOMPLETE : failed ? PFEC_PARTIAL : fixed ? PFEC_CORRECTED : PFEC_CLEAN;
  o.rows_corrected = fixed;
  o.rows_failed = failed;
  o.bytes_corrected = bytes;
  o.headers_matched = g.score;
  o.reserved = 0;
  rec[k] = o;
}
} // namespace

void pfec_host_tables(std::vector<uint8_t> & blob)
{
  PfecTables t;
  memset(&t, 0, sizeof t);
  pfec_tables(t);
  blob.resize(sizeof t);
  memcpy(blob.data(), &t, sizeof t);
}

cudaError_t launch_pfec_locate(cudaStream_t s, const PfecStream * st, int n_streams, long long n_slots, uint8_t * code, uint8_t * start, unsigned long long * lc)
{
  if (n_slots <= 0) return cudaSuccess;
  const unsigned grid = (unsigned)((n_slots + 255) / 256);
  k_pfec_code<<<grid, 256, 0, s>>>(st, n_streams, n_slots, code);
  k_pfec_start<<<grid, 256, 0, s>>>(st, n_streams, n_slots, code, start);
  if (lc) (*lc) += 2;
  return cudaGetLastError();
}

cudaError_t launch_pfec_list(cudaStream_t s, const PfecStream * st, int n_streams, const uint8_t * code, const uint8_t * start, PfecStage * stage, int * cnt,
                             uint8_t * mask, unsigned long long * lc)
{
  if (n_streams <= 0) return cudaSuccess;
  k_pfec_list<<<n_streams, PFEC_LIST_THREADS, 0, s>>>(st, code, start, stage, cnt, mask);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

cudaError_t launch_pfec_correct(cudaStream_t s, const PfecStream * st, int n_streams, long long n_out, const void * tables, const PfecStage * stage, PfecRec * rec,
                                unsigned long long * lc)
{
  if (n_out <= 0) return cudaSuccess;
  constexpr int per = PFEC_CORRECT_THREADS / PFEC_LANES;
  k_pfec_correct<<<(unsigned)((n_out + per - 1) / per), PFEC_CORRECT_THREADS, 0, s>>>(st, n_streams, n_out, static_cast<const PfecTables *>(tables), stage, rec);
  if (lc) (*lc)++;
  return cudaGetLastError();
}
} // namespace dab
