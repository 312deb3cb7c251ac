// dabplus.cuh — which five-frame windows of a DAB+ sub-channel Mp4Processor attempts (mp4processor.cpp:95-180), as one
// function the device walk kernel and the host tests share.
#pragma once
#include <cstdint>

namespace dab
{
// per-window state of the DAB+ pass (dabplus_kernels.cu)
enum : uint8_t
{
  SF_PRE_OK = 1,  // the Fire code holds on the window's raw header (FirecodeChecker::check, mp4processor.cpp:133)
  SF_DECODED = 2, // the window has been through Reed-Solomon and the header repair: SF_OK is known
  SF_OK = 4,      // ... and the repair succeeded (_process_reed_solomon_frame returned true)
};

// Mp4Processor::add_to_frame's synchronisation over n_frames logical frames; window w covers frames w..w+4. A window whose
// outcome is not known yet (no SF_DECODED) is taken to succeed. Writes the attempted windows in order to attempted[] (room for
// n_frames - 4: once synchronisation has run out, the next window may be attempted one frame later) and returns their count.
__host__ __device__ inline int superframe_walk(const uint8_t * state, int n_frames, int * attempted)
{
  int in_buf = 0, sync = 0, n = 0;
  for (int f = 0; f < n_frames; f++)
  {
    if (++in_buf < 5) continue;
    const int w = f - 4;
    const unsigned s = state[w];
    if (sync == 0)
    {
      if (s & SF_PRE_OK) sync = 4;
      else { in_buf = 4; continue; }
    }
    in_buf = 0;
    attempted[n++] = w;
    if (!(s & SF_DECODED) || (s & SF_OK)) sync = 4;
    else if (--sync == 0) in_buf = 4;
  }
  return n;
}
} // namespace dab
