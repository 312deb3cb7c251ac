// mp2_kernels.cu — MPEG-1 / MPEG-2 LSF audio layer II frames of DAB (MP2) sub-channels on the GPU: header, allocation, SCFSI and
// CRC-16 of every audio-frame slot, the walk over each stream's slots, and the compaction of records and OK frames.
//
// A DAB audio frame starts at the first bit of a logical frame and fills it (48 kHz), or it and the next (24 kHz; ETSI EN 300 401
// clause 7). So every logical frame is classified on its own (k_mp2_scan, mp2.cuh: mp2_classify), and the only dependency left,
// whether a slot is the second half of an OK 24 kHz frame, is resolved by a scan over 2-state maps, one block per stream
// (k_mp2_walk, built on mp2_walk_step). The records and the OK frames' bytes are then compacted in stream order (k_mp2_compact)
// for one copy to the host (engine.cu: run_mp2).
#include "kernels.h"
#include "stream_search.cuh"
#include "block_scan.cuh"

namespace dab
{
namespace
{
// thread = logical frame of any stream: classify the slot that would start there
__global__ void __launch_bounds__(128) k_mp2_scan(const Mp2Stream * __restrict__ st, int n_streams, long long n_slots, uint8_t * __restrict__ cls, int2 * __restrict__ crc,
                                                  uint32_t * __restrict__ hdr)
{
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_slots) return;
  const Mp2Stream & s = st[find_stream(st, n_streams, g, [](const Mp2Stream & x) { return x.slot0; })];
  const long long i = g - s.slot0, fb = 3LL * s.bit_rate;
  const Mp2Slot r = mp2_classify(s.src + i * fb, (s.n_frames - i) * fb, s.bit_rate);
  cls[g] = mp2_class_byte(r);
  crc[g] = make_int2(r.crc_stored, r.crc_computed);
  hdr[g] = r.header;
}

// The walk as a scan over 2-state maps (block_scan.cuh). A slot is in state 0 (it starts a record) or 1 (it is the second half
// of an OK 24 kHz frame); slot 0 is in state 0. A slot in state 1 hands state 0 to the next; one in state 0 hands on 1 exactly
// when mp2_walk_step makes its record span two logical frames.
constexpr int MP2_WALK_THREADS = 256;
__device__ inline unsigned next_state(const uint8_t * cls, int i, int n, unsigned state)
{
  int status;
  return state == 0 && mp2_walk_step(cls[i], i, n, &status) == 2 ? 1u : 0u;
}

// block = stream: each thread takes a contiguous chunk of its slots; the scanned maps give the chunk's entry state, a scan of the
// chunks' record and byte counts gives where its records go; the records are staged at the stream's own slot range
__global__ void __launch_bounds__(MP2_WALK_THREADS) k_mp2_walk(const Mp2Stream * __restrict__ st, const uint8_t * __restrict__ cls_all, const int2 * __restrict__ crc,
                                                               const uint32_t * __restrict__ hdr, Mp2Rec * __restrict__ stage, long long * __restrict__ stage_off,
                                                               Mp2Count * __restrict__ cnt)
{
  __shared__ unsigned sh_map[32];
  __shared__ Mp2Count sh_cnt[32];
  const Mp2Stream & s = st[blockIdx.x];
  const int n = s.n_frames, per = (n + (int)blockDim.x - 1) / (int)blockDim.x;
  const int i0 = min(n, (int)threadIdx.x * per), i1 = min(n, i0 + per);
  const uint8_t * cls = cls_all + s.slot0;
  const long long fb = 3LL * s.bit_rate;
  unsigned a = 0, b = 1; // the chunk's states entered with 0 and with 1
  for (int i = i0; i < i1; i++)
  {
    a = next_state(cls, i, n, a);
    b = next_state(cls, i, n, b);
  }
  const unsigned entry = block_exclusive_scan(a | (b << 1), MAP_IDENTITY, map_then, sh_map, (unsigned *)nullptr) & 1u;
  Mp2Count mine{ 0, 0 };
  unsigned state = entry;
  for (int i = i0; i < i1; i++)
  {
    if (state == 0)
    {
      int status;
      const int span = mp2_walk_step(cls[i], i, n, &status);
      mine.recs++;
      if (status == MP2_OK) mine.bytes += span * fb;
    }
    state = next_state(cls, i, n, state);
  }
  Mp2Count total;
  const Mp2Count off = block_exclusive_scan(mine, Mp2Count{ 0, 0 }, [](Mp2Count x, Mp2Count y) { return Mp2Count{ x.recs + y.recs, x.bytes + y.bytes }; }, sh_cnt, &total);
  long long k = s.slot0 + off.recs, bytes = off.bytes;
  state = entry;
  for (int i = i0; i < i1; i++)
  {
    if (state == 0)
    {
      int status;
      const int span = mp2_walk_step(cls[i], i, n, &status);
      const int2 c = crc[s.slot0 + i];
      stage[k] = Mp2Rec{ i, span, status, hdr[s.slot0 + i], c.x, c.y };
      stage_off[k] = status == MP2_OK ? bytes : -1;
      if (status == MP2_OK) bytes += span * fb;
      k++;
    }
    state = next_state(cls, i, n, state);
  }
  if (threadIdx.x == 0) cnt[blockIdx.x] = total;
}

// warp = output record: the record, and its frame's bytes if it is OK
constexpr int MP2_COMPACT_WARPS = 4;
__global__ void __launch_bounds__(32 * MP2_COMPACT_WARPS) k_mp2_compact(const Mp2Stream * __restrict__ st, int n_streams, long long n_out, const Mp2Rec * __restrict__ stage,
                                                                        const long long * __restrict__ stage_off, Mp2Rec * __restrict__ out_rec, uint8_t * __restrict__ out_pay)
{
  const long long k = (long long)blockIdx.x * MP2_COMPACT_WARPS + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (k >= n_out) return;
  const Mp2Stream & s = st[find_stream(st, n_streams, k, [](const Mp2Stream & x) { return x.out_rec0; })];
  const long long j = s.slot0 + (k - s.out_rec0);
  const Mp2Rec r = stage[j];
  if (lane == 0) out_rec[k] = r;
  const long long off = stage_off[j];
  if (off < 0) return;
  const long long fb = 3LL * s.bit_rate, n = r.n_frames * fb;
  const uint8_t * src = s.src + r.first_frame * fb;
  uint8_t * dst = out_pay + s.out_pay0 + off;
  for (long long b = lane; b < n; b += 32) dst[b] = src[b];
}
} // namespace

cudaError_t launch_mp2_scan(cudaStream_t s, const Mp2Stream * st, int n_streams, long long n_slots, uint8_t * cls, int2 * crc, uint32_t * hdr, unsigned long long * lc)
{
  if (n_slots <= 0) return cudaSuccess;
  k_mp2_scan<<<(unsigned)((n_slots + 127) / 128), 128, 0, s>>>(st, n_streams, n_slots, cls, crc, hdr);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

cudaError_t launch_mp2_walk(cudaStream_t s, const Mp2Stream * st, int n_streams, const uint8_t * cls, const int2 * crc, const uint32_t * hdr, Mp2Rec * stage,
                            long long * stage_off, Mp2Count * cnt, unsigned long long * lc)
{
  if (n_streams <= 0) return cudaSuccess;
  k_mp2_walk<<<n_streams, MP2_WALK_THREADS, 0, s>>>(st, cls, crc, hdr, stage, stage_off, cnt);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

cudaError_t launch_mp2_compact(cudaStream_t s, const Mp2Stream * st, int n_streams, long long n_out, const Mp2Rec * stage, const long long * stage_off,
                               Mp2Rec * out_rec, uint8_t * out_pay, unsigned long long * lc)
{
  if (n_out <= 0) return cudaSuccess;
  k_mp2_compact<<<(unsigned)((n_out + MP2_COMPACT_WARPS - 1) / MP2_COMPACT_WARPS), 32 * MP2_COMPACT_WARPS, 0, s>>>(st, n_streams, n_out, stage, stage_off, out_rec, out_pay);
  if (lc) (*lc)++;
  return cudaGetLastError();
}
} // namespace dab
