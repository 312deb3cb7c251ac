// stream_search.cuh — the batched outer-code passes (DAB+, MP2) lay their streams' items (windows, slots, output records) end
// to end in one index space and give every stream the first index of its range; a thread finds its stream by binary search.
#pragma once

namespace dab
{
// the stream whose range [key(s), key(s + 1)) holds i: the last s with key(s) <= i (streams with an empty range share the key of the next)
template <typename S, typename K> __device__ inline int find_stream(const S * __restrict__ st, int n, long long i, K key)
{
  int lo = 0, hi = n - 1;
  while (lo < hi)
  {
    const int mid = (lo + hi + 1) >> 1;
    if (key(st[mid]) <= i) lo = mid; else hi = mid - 1;
  }
  return lo;
}
} // namespace dab
