// viterbi.cuh — K=7 rate-1/4 Viterbi decoder, one warp per terminated code word.
//
// Replaces ViterbiSpiral::deconvolve (support/viterbi_spiral/viterbi_spiral.cpp:95-126, viterbi_scalar.h:9-94)
// together with the callers' index work around it: FicDecoder's depuncturing / PRBS / CRC / BER
// (decoder/fic_decoder.cpp:178-262), Protection::deconvolve (protection/protection.cpp:46-59) and Backend's
// 16-CIF time de-interleaver and energy dispersal (backend/backend.cpp:129-158).
//
// Mapping: lane i owns butterfly i (old states i and i+32 -> new states 2i and 2i+1), i.e. two path
// metrics per lane. Metrics live in the upper 16 bits of a register: the reference's 32-bit metrics never
// differ by more than 6*1020+1000 between states, so arithmetic modulo 2^16 with signed comparison gives
// the same decisions and needs no renormalisation. Ties keep path 0 (decision = (m0 - m1) > 0), as the
// scalar reference does (the AVX2 variant of the reference differs, SURVEY.md section 0).
// Per step: one broadcast LDS of the four clamped symbols, XOR + DP4A branch metric, two shuffles that
// bring the packed metrics of the two predecessor lanes, add-compare-select, two ballots -> one 64-bit
// survivor word in shared memory (bit i = decision of state 2i, bit 32+i = state 2i+1).
// Chain back: 32 steps at a time, lane j prefetches the survivor word of step T-j, the state recursion
// s' = (s>>1)|(k<<5) then runs out of registers (shuffles are off the dependent chain).
#pragma once
#include "common.cuh"

namespace dab
{
constexpr int VIT_MAX_SEG = 6;

// Where the soft inputs of a code word come from. A profile is one (L_i, PI_i) puncturing recipe
// (EEP/UEP/FIC) or the identity (already depunctured input).
struct VitProfile
{
  int n_bits;                  // information bits N (768 for a FIC, 24*bitRate for MSC)
  int n_seg;                   // puncturing segments incl. the 24-position tail
  int seg_pos[VIT_MAX_SEG + 1];// first Viterbi-input position of segment s (seg_pos[n_seg] = 4(N+6))
  int seg_kept[VIT_MAX_SEG];   // kept soft bits before segment s
  unsigned seg_mask[VIT_MAX_SEG]; // puncturing vector of the segment, bit j = position j mod 32 kept
  int n_kept;                  // total kept soft bits
  int tab_off;                 // first entry of this profile in the step table (vit_step_entry), one entry per trellis step
};

// Step-table entry of trellis step t: kept soft bits before Viterbi-input position 4t (bits 0..27) and which of the
// positions 4t..4t+3 are kept (bits 28..31). Built on the host when a profile is registered; the batched kernels read
// it instead of searching the puncturing segments per position.
__host__ __device__ inline unsigned vit_step_entry_make(int kept_before, unsigned mask4) { return (unsigned)kept_before | (mask4 << 28); }

enum { VIT_SRC_LINEAR = 0, VIT_SRC_TIME_DEINTERLEAVE = 1 };
enum { VIT_FLAG_PRBS = 1, VIT_FLAG_FIC = 2 };

struct VitJob
{
  long long src;       // int16 index of kept soft bit 0 (LINEAR) or of the recording's frame slot 0 (TIME_DEINTERLEAVE)
  long long out;       // byte index of decoded bit 0
  int profile;
  int src_mode;
  int flags;
  int cif_first;       // TIME_DEINTERLEAVE: CIF index (4*slot + c) read by bits whose interleave delay row is 0
  int row_mask;        // bit m set: the CIF of row m exists (otherwise the de-interleaver memory is still zero)
  int frag_off;        // startCU * 64
  int aux;             // FIC: index of the FIC block (crc_ok[3*aux..], ber[2*aux..])
  int skip_plus1;      // TIME_DEINTERLEAVE, EtiGenerator only: CIF (skip_plus1 - 1) is missing from the de-interleaver history
                       // (rows at or after it read one CIF later, row index -1 reads the dropped CIF itself); 0 = Backend
};

// A Backend's jobs in compact form (expanded on the device, k_expand_backend_jobs): logical frames g_first .. g_first + n_jobs - 1
// of a sub-channel whose Backend exists from CIF g_start on.
struct BackendJobRange
{
  long long src, out;  // as VitJob::src; byte index of the first decoded bit of the range
  int profile, n_bits; // n_bits = 24 * bit rate
  int g_start, g_first, n_jobs;
  int frag_off;
  int job_first;       // index of the range's first job in the launch's job array
  int pad;
};

// CIF read by de-interleaver row m of a job (see VitJob::skip_plus1 and decoder.cu, ETI section)
__host__ __device__ inline int vit_row_cif(int cif_first, int skip_plus1, int m)
{
  int cif = cif_first + m;
  if (skip_plus1 > 0)
  {
    const int skip = skip_plus1 - 1;
    cif = cif < 0 ? skip : (cif >= skip ? cif + 1 : cif);
  }
  return cif;
}

// Time de-interleaver row of fragment bit i (backend/backend.cpp:129): out_r[i] = in_{r-16+map[i&15]}[i]
__host__ __device__ inline int time_map(int i)
{
  // {0,8,4,12,2,10,6,14,1,9,5,13,3,11,7,15} = 4-bit reversal
  const int x = i & 15;
  return ((x & 1) << 3) | ((x & 2) << 1) | ((x & 4) >> 1) | ((x & 8) >> 3);
}

// int16 offset of CIF g (g = 4*slot + c) inside a recording's soft-bit buffer [slot][75][3072]
__host__ __device__ inline long long cif_offset(int g) { return (long long)(g >> 2) * FRAME_SOFT + FIC_SOFT + (long long)(g & 3) * CIF_BITS; }

// Kept-bit index of Viterbi-input position p, or -1 if the position is punctured.
__host__ __device__ inline int vit_src_index(const VitProfile & pr, int p)
{
  int pos = pr.seg_pos[0], kept = pr.seg_kept[0];
  unsigned m = pr.seg_mask[0];
#pragma unroll
  for (int i = 1; i < VIT_MAX_SEG; i++)
    if (i < pr.n_seg && p >= pr.seg_pos[i]) { pos = pr.seg_pos[i]; kept = pr.seg_kept[i]; m = pr.seg_mask[i]; }
  const int q = p - pos;
  if (!((m >> (q & 31)) & 1u)) return -1;
#ifdef __CUDA_ARCH__
  return kept + (q >> 5) * __popc(m) + __popc(m & ((1u << (q & 31)) - 1u));
#else
  return kept + (q >> 5) * __builtin_popcount(m) + __builtin_popcount(m & ((1u << (q & 31)) - 1u));
#endif
}

// Expected symbols of butterfly i as a byte mask (byte j = 0xFF when generator j outputs 1 on the branch
// old state i -> new state 2i). Generators {109, 79, 83, 109} on the register (2i): viterbi_spiral.cpp:27-37.
__host__ __device__ inline unsigned vit_branch_mask(int i)
{
  const int poly[4] = { 109, 79, 83, 109 };
  unsigned m = 0;
  for (int j = 0; j < 4; j++)
  {
    unsigned x = (unsigned)((2 * i) & poly[j]);
    x ^= x >> 4; x ^= x >> 2; x ^= x >> 1;
    if (x & 1u) m |= 0xFFu << (8 * j);
  }
  return m;
}

// One add-compare-select of butterfly i. a, b: metrics of old states i, i+32 in the upper 16 bits.
// metric: branch metric (0..1020). Outputs the survivors for new states 2i, 2i+1 (upper 16 bits) and the decisions.
__host__ __device__ inline void vit_acs(unsigned a, unsigned b, unsigned metric, unsigned & n0, unsigned & n1, bool & d0, bool & d1)
{
  const unsigned M = metric << 16, Mb = (1020u - metric) << 16;
  const unsigned m0 = a + M, m1 = b + Mb, m2 = a + Mb, m3 = b + M;
  d0 = (int)(m0 - m1) > 0;
  d1 = (int)(m2 - m3) > 0;
  n0 = d0 ? m1 : m0;
  n1 = d1 ? m3 : m2;
}

// Chain-back step on the rotated state r = (s >> 1) | ((s & 1) << 5): survivor word w has the decision of
// state s at bit r. Returns the decoded bit and updates r for the predecessor state s' = (s >> 1) | (k << 5).
__host__ __device__ inline unsigned vit_traceback_step(unsigned long long w, unsigned & r)
{
  const unsigned k = (unsigned)(w >> r) & 1u;
  // s = ((r & 31) << 1) | (r >> 5); s' = (s >> 1) | (k << 5) = (r & 31) | (k << 5); r' = (s' >> 1) | ((s' & 1) << 5)
  const unsigned sp = (r & 31u) | (k << 5);
  r = (sp >> 1) | ((sp & 1u) << 5);
  return k;
}
} // namespace dab
