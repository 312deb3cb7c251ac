// block_scan.cuh — the block-wide scan the stream walks (MP2 slots, packet-mode groups) are built on, and the composition of
// the 2-state maps a walk is scanned as.
#pragma once
#include <cstdint>

namespace dab
{
// __shfl_up_sync of any value made of 32-bit words
template <typename T> __device__ inline T shfl_up(T v, int d)
{
  static_assert(sizeof(T) % 4 == 0, "shfl_up: T must be made of 32-bit words");
  union U { T t; unsigned w[sizeof(T) / 4]; };
  U u;
  u.t = v;
#pragma unroll
  for (int i = 0; i < (int)(sizeof(T) / 4); i++) u.w[i] = __shfl_up_sync(0xffffffffu, u.w[i], d);
  return u.t;
}

// Block-wide exclusive scan of one value per thread (blockDim.x a multiple of 32): op(a, b) combines an earlier a with a later b;
// *total (may be null) gets the combination of all values. sh: 32 entries of shared memory.
template <typename T, typename Op> __device__ T block_exclusive_scan(T v, T id, Op op, T * sh, T * total)
{
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  T x = v;
  for (int d = 1; d < 32; d <<= 1)
  {
    const T y = shfl_up(x, d);
    if (lane >= d) x = op(y, x);
  }
  if (lane == 31) sh[w] = x;
  __syncthreads();
  if (w == 0)
  {
    T t = lane < nw ? sh[lane] : id;
    for (int d = 1; d < 32; d <<= 1)
    {
      const T y = shfl_up(t, d);
      if (lane >= d) t = op(y, t);
    }
    sh[lane] = t;
  }
  __syncthreads();
  T before = shfl_up(x, 1);
  if (lane == 0) before = id;
  const T r = op(w > 0 ? sh[w - 1] : id, before);
  if (total) *total = sh[nw - 1];
  __syncthreads(); // sh is reused by the next scan
  return r;
}

// A walk over 2 states as a scan: the map of a run of items holds in bit s the state after the run when it is entered in state
// s. Maps compose, so the entry state of every chunk of items comes from a block-wide scan of the chunks' maps.
constexpr unsigned MAP_IDENTITY = 2u; // 0 -> 0, 1 -> 1
__device__ inline unsigned map_then(unsigned a, unsigned b) { return ((b >> (a & 1u)) & 1u) | (((b >> ((a >> 1) & 1u)) & 1u) << 1); } // b after a
} // namespace dab
