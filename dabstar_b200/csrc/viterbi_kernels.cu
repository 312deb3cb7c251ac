// viterbi_kernels.cu — warp-per-code-word Viterbi with fused depuncture / time de-interleave gather,
// energy dispersal, FIB CRC and BER re-encode. See viterbi.cuh for the algorithm and reference citations.
#include "viterbi.cuh"
#include "viterbi_tpc.cuh"
#include "kernels.h"
#include "devcache.h"

#include <cstdlib>

namespace dab
{
namespace
{
constexpr unsigned FULL = 0xffffffffu;
constexpr int VIT_SMEM_PER_STEP = 14; // bytes of shared memory per trellis step and warp

__device__ __forceinline__ unsigned clamp_sym(int v)
{
  // viterbi_scalar.h:34-40: `i16 tmp = in; tmp += 127;` wraps in 16 bits before the clamp (inputs above 32640 become 0)
  v = (int)(short)(v + 127);
  return (unsigned)min(max(v, 0), 255);
}

__device__ __forceinline__ unsigned parity8(unsigned x)
{
  return __popc(x) & 1u;
}

// Job j of a launch: either an entry of the job list, or (fic_frames != nullptr) FIC block (j & 3) of frame descriptor
// j >> 2. Returns false when the frame ends before that FIC block.
__device__ __forceinline__ bool load_job(const VitJob * __restrict__ jobs, const FrameDesc * __restrict__ fic_frames, int j, VitJob & job)
{
  if (fic_frames != nullptr)
  {
    const FrameDesc & fd = fic_frames[j >> 2];
    const int b = j & 3, n_fic = min(4, fd.n_syms * SYM_BITS / FIC_IN);
    if (b >= n_fic) return false;
    job.src = (long long)fd.slot * FRAME_SOFT + (long long)b * FIC_IN;
    job.out = (long long)fd.slot * (4 * FIC_OUT) + (long long)b * FIC_OUT;
    job.profile = 0;
    job.src_mode = VIT_SRC_LINEAR;
    job.flags = VIT_FLAG_PRBS | VIT_FLAG_FIC;
    job.cif_first = job.row_mask = job.frag_off = 0;
    job.aux = 4 * fd.slot + b;
    job.skip_plus1 = 0;
  }
  else job = jobs[j];
  return true;
}

// Raw soft input of kept bit idx of a job (0 where the time de-interleaver memory is still empty).
__device__ __forceinline__ int job_soft(const VitJob & job, const int16_t * __restrict__ soft, int idx)
{
  if (job.src_mode == VIT_SRC_LINEAR) return soft[job.src + idx];
  const int m = time_map(idx);
  if (!((job.row_mask >> m) & 1)) return 0;
  return soft[job.src + cif_offset(vit_row_cif(job.cif_first, job.skip_plus1, m)) + job.frag_off + idx];
}

// Eight consecutive energy-dispersal bits as a byte, first bit most significant: bit 7 - j = prbs[i + j] (i a multiple of 8)
__device__ __forceinline__ unsigned prbs_byte_msb(const uint8_t * __restrict__ prbs, int i)
{
  const uint2 w = *reinterpret_cast<const uint2 *>(prbs + i); // one 0/1 byte per bit
  // bytes b0..b3 of a word times 0x08040201: the top byte of the product is 8 b0 + 4 b1 + 2 b2 + b3 (no carries reach it)
  const unsigned n0 = ((w.x * 0x08040201u) >> 24) & 0x0fu, n1 = ((w.y * 0x08040201u) >> 24) & 0x0fu;
  return (n0 << 4) | n1;
}

// shared memory per warp: survivors u64[cap] | symbols u32[cap] | decoded bits u8[cap] | input signs, 1 bit per position (cap/2 bytes)
// fic_frames != nullptr: job j is FIC block (j & 3) of frame descriptor j >> 2 (no job list needed)
__global__ void __launch_bounds__(256) k_viterbi(const VitJob * __restrict__ jobs, const FrameDesc * __restrict__ fic_frames, int n_jobs, const VitProfile * __restrict__ profiles,
                                                 const int16_t * __restrict__ soft, uint8_t * __restrict__ out_bits,
                                                 const uint8_t * __restrict__ prbs, uint8_t * __restrict__ crc_ok,
                                                 int * __restrict__ ber, int cap)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  unsigned char * base = smem_raw + (size_t)warp * (size_t)cap * VIT_SMEM_PER_STEP;
  unsigned long long * surv = reinterpret_cast<unsigned long long *>(base);
  unsigned * syms = reinterpret_cast<unsigned *>(base + (size_t)cap * 8);
  unsigned char * syms8 = reinterpret_cast<unsigned char *>(syms);
  unsigned char * dbits = base + (size_t)cap * 12;
  unsigned * sgn = reinterpret_cast<unsigned *>(base + (size_t)cap * 13);

  const unsigned xmask = vit_branch_mask(lane);
  const unsigned sel = (lane & 1) ? 0x3244u : 0x1044u; // PRMT: chosen 16-bit half -> upper half, zeros below
  const int src_a = lane >> 1, src_b = 16 + (lane >> 1);

  for (int j = blockIdx.x * warps + warp; j < n_jobs; j += gridDim.x * warps)
  {
    VitJob job;
    if (!load_job(jobs, fic_frames, j, job)) continue;
    const VitProfile pr = profiles[job.profile];
    const int n_bits = pr.n_bits, steps = n_bits + 6;

    // ---- gather: depuncture (+ time de-interleave) and clamp to u8
    for (int p0 = 0; p0 < 4 * steps; p0 += 32)
    {
      const int p = p0 + lane;
      int v = 0;
      if (p < 4 * steps)
      {
        const int idx = vit_src_index(pr, p);
        if (idx >= 0)
        {
          v = job_soft(job, soft, idx);
        }
        syms8[p] = (unsigned char)clamp_sym(v);
      }
      const unsigned pos = __ballot_sync(FULL, v > 0); // sign of the raw input, for calculate_BER
      if (lane == 0) sgn[p0 >> 5] = pos;
    }
    __syncwarp();

    // ---- forward pass
    unsigned a = (lane == 0 ? 0u : 1000u) << 16; // old[i]   (start metrics 0 / 1000, viterbi_spiral.cpp:98-101)
    unsigned b = 1000u << 16;                    // old[i+32]
    for (int t = 0; t < steps; t++)
    {
      const unsigned metric = __dp4a(syms[t] ^ xmask, 0x01010101u, 0u);
      unsigned n0, n1;
      bool d0, d1;
      vit_acs(a, b, metric, n0, n1, d0, d1);
      const unsigned w0 = __ballot_sync(FULL, d0), w1 = __ballot_sync(FULL, d1);
      if (lane == 0) surv[t] = (unsigned long long)w0 | ((unsigned long long)w1 << 32);
      const unsigned pk = __byte_perm(n0, n1, 0x7632); // low half = n0 >> 16, high half = n1 >> 16
      const unsigned va = __shfl_sync(FULL, pk, src_a), vb = __shfl_sync(FULL, pk, src_b);
      a = __byte_perm(va, 0u, sel);
      b = __byte_perm(vb, 0u, sel);
    }
    __syncwarp();

    // ---- chain back from state 0, 32 decisions per round
    unsigned r = 0;
    for (int top = steps - 1; top >= 6; top -= 32)
    {
      const int e = top - lane;
      const unsigned long long w = e >= 0 ? surv[e] : 0ull;
      unsigned mine = 0;
#pragma unroll 8
      for (int q = 0; q < 32; q++)
      {
        const unsigned long long wq = __shfl_sync(FULL, w, q);
        const unsigned k = vit_traceback_step(wq, r);
        if (q == lane) mine = k;
      }
      const int t = e - 6;
      if (t >= 0)
      {
        if (job.flags & VIT_FLAG_FIC) dbits[t] = (unsigned char)mine;
        out_bits[job.out + t] = (unsigned char)(mine ^ ((job.flags & VIT_FLAG_PRBS) ? prbs[t] : 0));
      }
    }

    if (job.flags & VIT_FLAG_FIC)
    {
      __syncwarp();
      // BER: re-encode and compare with the sign of the kept inputs (viterbi_spiral.cpp:128-164)
      int errors = 0;
      for (int i = lane; i < steps; i += 32)
      {
        unsigned sr = 0;
#pragma unroll
        for (int q = 0; q < 8; q++)
        {
          const int ii = i - q;
          if (ii >= 0 && ii < n_bits) sr |= (unsigned)dbits[ii] << q;
        }
        const int poly[4] = { 109, 79, 83, 109 };
#pragma unroll
        for (int g = 0; g < 4; g++)
        {
          if (vit_src_index(pr, 4 * i + g) < 0) continue;
          const unsigned hard = (sgn[(4 * i + g) >> 5] >> ((4 * i + g) & 31)) & 1u;
          errors += hard != parity8(sr & (unsigned)poly[g]);
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) errors += __shfl_xor_sync(FULL, errors, o);
      if (lane == 0) { ber[2 * job.aux] = pr.n_kept; ber[2 * job.aux + 1] = errors; }
      // CRC of the three FIBs on the descrambled bits (backend/crc.cpp:98-132)
      if (lane < 3)
      {
        unsigned reg = 0xffff;
        const int o = lane * 256;
        for (int i = 0; i < 256; i++)
        {
          const unsigned bit = (unsigned)(dbits[o + i] ^ prbs[o + i]) ^ (i >= 240 ? 1u : 0u);
          const unsigned fb = ((reg >> 15) & 1u) ^ bit;
          reg = (reg << 1) & 0xffffu;
          if (fb) reg ^= 0x1021u;
        }
        crc_ok[3 * job.aux + lane] = reg == 0;
      }
    }
    __syncwarp();
  }
}

// ================================================================================================ thread per code word
// Three kernels (algorithm and reference citations: viterbi_tpc.cuh):
//   k_vit_gather_kb : depuncture (+ 16-CIF time de-interleave) + clamp; writes the 4 symbols of every trellis step as one
//                     32-bit word, [step][code word], through a shared-memory transpose (coalesced on both sides)
//   k_vit_tpc       : forward pass (decision words to [step][code word]) and chain back, energy dispersal fused into the
//                     packed byte store
//   k_fic_post      : FIB CRC and BER re-encode of FIC blocks (warp per block)
constexpr int GATHER_STEPS = 128; // trellis steps per CTA tile
// Every CTA first files, per code word and de-interleave delay row, where kept bit 0 of that row lives (shared memory).
// ncu on a gather that did this address arithmetic per bit (CIF offset, row mask, source mode) showed it issue bound at
// 155 warp instructions per lane and trellis step (profiles/r1_g2_ncu_gather_summary.txt). Staging the 47 CIF rows of a
// CTA in shared memory was measured twice (bit exact, 19.5 instead of 16.9 ms for the MSC pass of the full ensemble) and
// dropped.
__device__ int16_t g_zero_row[CIF_BITS]; // what a delay row reads while its CIF precedes the Backend (backend.cpp:129-161: the memory starts as zeros)

// The kept soft bits of a code word are consecutive in the source, only the trellis steps they belong to are irregular. So
// each warp first copies the kept bits of its code word's 128 steps into shared memory as clamped bytes — lane L takes kept
// bits 4L..4L+3 (mod 128) from the 128-aligned start, which fixes the four de-interleave delay rows of a lane for the whole
// code word: four pointer fetches per code word instead of one per bit, loads at constant offsets, no work for punctured
// positions — and then builds each step's word from the four bytes at the step's first kept bit (two shared-memory words
// and a funnel shift) with one PRMT whose selector puts 127 (erasure) into the punctured positions. A gather that fetched
// a row pointer and issued a predicated load per mother-code bit was still issue bound: 260 against 139 instructions per
// code word and lane, MSC gather 3.83 against 3.57 ms (profiles/README.md).
constexpr int GK_WORDS = (4 * GATHER_STEPS + 128) / 4 + 1; // kept bytes of a tile from the aligned start, + the funnel shift's second word
constexpr int GK_ITERS = (4 * GATHER_STEPS + 128) / 128;
constexpr int GK_BATCH = 3; // 128-bit groups of a code word whose loads are in flight together

// soft bit at p if k < lim; unspecified otherwise (such bytes are never selected)
__device__ __forceinline__ int ld_soft_lt(const int16_t * p, int k, int lim)
{
  int v;
  asm volatile("{\n\t.reg .pred q;\n\tsetp.lt.s32 q, %2, %3;\n\t@q ld.global.nc.s16 %0, [%1];\n\t}" : "=r"(v) : "l"(p), "r"(k), "r"(lim));
  return v;
}

__global__ void __launch_bounds__(256, 4) k_vit_gather_kb(const VitJob * __restrict__ jobs, const FrameDesc * __restrict__ fic_frames, int job_first, int n_jobs,
                                                       const VitProfile * __restrict__ profiles, const unsigned * __restrict__ step_tab,
                                                       const int16_t * __restrict__ soft, unsigned * __restrict__ sym, int stride, int rows)
{
  constexpr int H = GATHER_STEPS / 32;
  __shared__ unsigned tile[32][GATHER_STEPS + 1];
  // per code word: kept bit 0 of de-interleave delay row m (a linear source has the same pointer in all 16 rows; one
  // pad entry per code word keeps the lane-per-code-word stores off a single bank)
  __shared__ const int16_t * rowptr[32][17];
  __shared__ int sh_steps[32], sh_tab[32], sh_ka[32], sh_k1[32];
  __shared__ unsigned char sh_lin[32]; // the code word's kept bits are contiguous and 8-byte aligned: four per load
  __shared__ unsigned kb[8][GK_WORDS];
  __shared__ unsigned sel_lut[16];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int jb = blockIdx.x * 32, t0 = blockIdx.y * GATHER_STEPS;

  {
    // lane = code word, warp = two of the 16 delay rows
    VitJob job;
    const bool valid = jb + lane < n_jobs && load_job(jobs, fic_frames, job_first + jb + lane, job);
#pragma unroll
    for (int q = 0; q < 2; q++)
    {
      const int m = 2 * warp + q;
      const int16_t * p = g_zero_row;
      if (valid)
      {
        if (job.src_mode == VIT_SRC_LINEAR) p = soft + job.src;
        else if ((job.row_mask >> m) & 1) p = soft + job.src + cif_offset(vit_row_cif(job.cif_first, job.skip_plus1, m)) + job.frag_off;
      }
      rowptr[lane][m] = p;
    }
    if (warp == 0)
    {
      const VitProfile * pr = profiles + (valid ? job.profile : 0);
      const int steps = valid ? pr->n_bits + 6 : 0;
      const unsigned * tab = step_tab + pr->tab_off;
      int k0 = 0, k1 = 0; // kept bits [k0, k1) belong to the tile's steps
      if (t0 < steps)
      {
        k0 = (int)(tab[t0] & 0x0fffffffu);
        k1 = t0 + GATHER_STEPS < steps ? (int)(tab[t0 + GATHER_STEPS] & 0x0fffffffu) : pr->n_kept;
      }
      sh_steps[lane] = steps;
      sh_tab[lane] = pr->tab_off;
      sh_ka[lane] = k0 & ~127;
      sh_k1[lane] = k1;
      sh_lin[lane] = valid && job.src_mode == VIT_SRC_LINEAR && (pr->n_kept & 3) == 0 && ((uintptr_t)(soft + job.src) & 7) == 0;
    }
    if (threadIdx.x < 16)
    {
      // PRMT selector of a keep mask: the n-th kept position takes byte n of the four kept bytes, a punctured one byte 4 (= 127)
      unsigned s = 0, n = 0;
#pragma unroll
      for (int g = 0; g < 4; g++) s |= (((threadIdx.x >> g) & 1) ? n++ : 4u) << (4 * g);
      sel_lut[threadIdx.x] = s;
    }
  }
  __syncthreads();

  unsigned * kbw = kb[warp];
  // What depends only on the code word's profile and the tile is kept across the warp's code words (the jobs of a launch are
  // ordered by sub-channel: a CTA of mixed profiles is the exception): the kept-bit range, and per step the position of
  // its four bytes in kbw, the funnel-shift count and the PRMT selector.
  int cur_tab = -1, cur_steps = -1, ka = 0, span = 0, kl = 0, rem = 0;
  unsigned kpos[H], kshift[H], ksel[H];
  int ridx[4];
#pragma unroll
  for (int g = 0; g < 4; g++) ridx[g] = (int)(__brev((unsigned)(4 * lane + g)) >> 28); // time_map: 4-bit reversal of k & 15
#pragma unroll 1
  for (int c = 0; c < 4; c++)
  {
    const int jr = 4 * warp + c;
    if (sh_tab[jr] != cur_tab || sh_steps[jr] != cur_steps)
    {
      cur_tab = sh_tab[jr];
      cur_steps = sh_steps[jr];
      ka = sh_ka[jr];
      span = sh_k1[jr] - ka;  // kept bits from the aligned start to the end of the tile
      kl = ka + 4 * lane;
      rem = span - 4 * lane;  // the lane's bit 128 i + g exists if 128 i + g < rem
      const unsigned * tab = step_tab + cur_tab;
#pragma unroll
      for (int h = 0; h < H; h++)
      {
        const int t = t0 + lane + 32 * h;
        const unsigned w = tab[max(min(t, cur_steps - 1), 0)];
        const unsigned e = t < cur_steps ? w : (unsigned)ka; // no step: nothing kept, four erasures
        const int rel = (int)(e & 0x0fffffffu) - ka;
        kpos[h] = (unsigned)(rel >> 2);
        kshift[h] = (unsigned)rel << 3;
        ksel[h] = sel_lut[e >> 28];
      }
    }
    // ---- kept bits -> clamped bytes; every load of the code word is issued before the first is used
    // (three 128-bit groups of the code word at a time: all of a rate-1/2 tile, and it keeps the kernel at 64 registers)
    if (sh_lin[jr])
    {
      const uint2 * p = reinterpret_cast<const uint2 *>(rowptr[jr][0] + kl);
#pragma unroll
      for (int i0 = 0; i0 < GK_ITERS; i0 += GK_BATCH)
      {
        uint2 a[GK_BATCH];
#pragma unroll
        for (int i = i0; i < i0 + GK_BATCH && i < GK_ITERS; i++)
          if (128 * i < span && 128 * i < rem) a[i - i0] = __ldg(p + 32 * i); // the code word has a multiple of four kept bits
        asm volatile("" ::: "memory");
#pragma unroll
        for (int i = i0; i < i0 + GK_BATCH && i < GK_ITERS; i++)
        {
          if (128 * i < span)
          {
            const unsigned lo = __vmins2(__vmaxs2(__vadd2(a[i - i0].x, 0x007f007fu), 0u), 0x00ff00ffu);
            const unsigned hi = __vmins2(__vmaxs2(__vadd2(a[i - i0].y, 0x007f007fu), 0u), 0x00ff00ffu);
            kbw[32 * i + lane] = __byte_perm(lo, hi, 0x6420);
          }
        }
      }
    }
    else
    {
      const int16_t * p[4];
#pragma unroll
      for (int g = 0; g < 4; g++) p[g] = rowptr[jr][ridx[g]] + kl + g;
#pragma unroll
      for (int i0 = 0; i0 < GK_ITERS; i0 += GK_BATCH)
      {
        int a[GK_BATCH][4];
#pragma unroll
        for (int i = i0; i < i0 + GK_BATCH && i < GK_ITERS; i++)
        {
          if (128 * i < span)
          {
#pragma unroll
            for (int g = 0; g < 4; g++) a[i - i0][g] = ld_soft_lt(p[g] + 128 * i, 128 * i + g, rem);
          }
        }
        asm volatile("" ::: "memory");
#pragma unroll
        for (int i = i0; i < i0 + GK_BATCH && i < GK_ITERS; i++)
        {
          if (128 * i < span)
          {
            // viterbi_scalar.h:34-40: in + 127 wraps in 16 bits before the clamp to 0..255 (the 16-bit halves taken by the PRMT)
            unsigned lo = __byte_perm((unsigned)(a[i - i0][0] + 127), (unsigned)(a[i - i0][1] + 127), 0x5410);
            unsigned hi = __byte_perm((unsigned)(a[i - i0][2] + 127), (unsigned)(a[i - i0][3] + 127), 0x5410);
            lo = __vmins2(__vmaxs2(lo, 0u), 0x00ff00ffu);
            hi = __vmins2(__vmaxs2(hi, 0u), 0x00ff00ffu);
            kbw[32 * i + lane] = __byte_perm(lo, hi, 0x6420);
          }
        }
      }
    }
    __syncwarp();
    // ---- the four symbols of each step
#pragma unroll
    for (int h = 0; h < H; h++)
    {
      const unsigned v = __funnelshift_r(kbw[kpos[h]], kbw[kpos[h] + 1], kshift[h]);
      tile[jr][lane + 32 * h] = __byte_perm(v, 0x7f7f7f7fu, ksel[h]);
    }
    __syncwarp();
  }
  __syncthreads();
  unsigned * dst = sym + (size_t)(t0 + warp) * stride + jb + lane;
  const unsigned * src = &tile[lane][warp];
#pragma unroll
  for (int q = 0; q < GATHER_STEPS / 8; q++)
  {
    if (t0 + warp + 8 * q < rows) *dst = src[8 * q];
    dst += (size_t)8 * stride;
  }
}

__global__ void __launch_bounds__(32) k_vit_tpc(const VitJob * __restrict__ jobs, const FrameDesc * __restrict__ fic_frames, int job_first, int n_jobs,
                                                const VitProfile * __restrict__ profiles, const unsigned * __restrict__ sym,
                                                unsigned long long * __restrict__ surv, int stride, uint8_t * __restrict__ out_bits,
                                                const uint8_t * __restrict__ prbs)
{
  __shared__ unsigned char pos_lut[5][64]; // bit of the decision word that holds the decision of state y, per step type
  for (int i = threadIdx.x; i < 5 * 64; i += 32) pos_lut[i >> 6][i & 63] = (unsigned char)tpc_decision_bit(i >> 6, i & 63);
  __syncwarp();
  const int jl = blockIdx.x * 32 + threadIdx.x;
  if (jl >= n_jobs) return;
  VitJob job;
  if (!load_job(jobs, fic_frames, job_first + jl, job)) return;
  const int n_bits = profiles[job.profile].n_bits, steps = n_bits + 6;
  const unsigned * sp = sym + jl;
  unsigned long long * vp = surv + jl;

  // ---- forward pass, five steps per iteration; the symbols of the next TWO iterations are in flight meanwhile: the
  // symbol rows are followed by TPC_READ_AHEAD rows that are read and never used, and the decision rows are padded to a
  // multiple of 5, so neither the loads nor the stores of an iteration need a bound (launch_viterbi lays the workspace out)
  unsigned S[32];
  tpc_init(S);
  const size_t row = (size_t)(unsigned)stride;
  unsigned cur[5], nx1[5];
#pragma unroll
  for (int i = 0; i < 5; i++) { cur[i] = sp[i * row]; nx1[i] = sp[(5 + i) * row]; }
  const unsigned * pn = sp + 10 * row;
  unsigned long long * pv = vp;
  int to_renorm = TPC_RENORM / 5;
#pragma unroll 1
  for (int t0 = 0; t0 < steps; t0 += 5)
  {
    unsigned nx2[5];
#pragma unroll
    for (int i = 0; i < 5; i++) nx2[i] = pn[i * row];
    pn += 5 * row;
    unsigned long long dec[5];
    const bool renorm = --to_renorm == 0;
    if (renorm) to_renorm = TPC_RENORM / 5;
    tpc_five_steps(S, cur, dec, renorm);
#pragma unroll
    for (int i = 0; i < 5; i++)
    {
      pv[i * row] = dec[i];
      cur[i] = nx1[i];
      nx1[i] = nx2[i];
    }
    pv += 5 * row;
  }

  // ---- chain back from state 0; decoded bit i is the decision read at step i + 6 (viterbi_scalar.h:84-93).
  // The decision words of the next CB steps are loaded while the current CB are walked (the addresses do not depend on
  // the state, only the walk itself is serial); the forward pass's registers are free here, so CB = 16 words of 8 bytes.
  unsigned y = 0;
  const bool scramble = (job.flags & VIT_FLAG_PRBS) != 0;
  uint8_t * out = out_bits + job.out;
  constexpr int CB = 16;
  if (((unsigned long long)(uintptr_t)out & 7) == 0 && n_bits % CB == 0 && n_bits >= CB)
  {
    unsigned long long w[CB], wn[CB];
#pragma unroll
    for (int q = 0; q < CB; q++) w[q] = vp[(size_t)(n_bits - CB + 6 + q) * stride];
    int ty7 = (n_bits + 5) % 5; // type of step i + CB + 5 for i = n_bits - CB
#pragma unroll 1
    for (int i = n_bits - CB; i >= 0; i -= CB)
    {
      const int ip = i >= CB ? i - CB : 0;
#pragma unroll
      for (int q = 0; q < CB; q++) wn[q] = vp[(size_t)(ip + 6 + q) * stride];
      unsigned b[CB / 4];
#pragma unroll
      for (int q = 0; q < CB / 4; q++) b[q] = 0;
      int ty = ty7;
#pragma unroll
      for (int q = CB - 1; q >= 0; q--)
      {
        const unsigned k = tpc_traceback_step(w[q], pos_lut[ty][y], y);
        b[q >> 2] |= k << (8 * (q & 3));
        ty = ty == 0 ? 4 : ty - 1;
      }
      ty7 = ty;
#pragma unroll
      for (int q = 0; q < CB / 8; q++)
      {
        unsigned lo = b[2 * q], hi = b[2 * q + 1];
        if (scramble) { const uint2 pw = *reinterpret_cast<const uint2 *>(prbs + i + 8 * q); lo ^= pw.x; hi ^= pw.y; }
        *reinterpret_cast<uint2 *>(out + i + 8 * q) = make_uint2(lo, hi);
      }
#pragma unroll
      for (int q = 0; q < CB; q++) w[q] = wn[q];
    }
  }
  else
  {
    for (int i = n_bits - 1; i >= 0; i--)
    {
      const unsigned k = tpc_traceback_step(vp[(size_t)(i + 6) * stride], pos_lut[(i + 6) % 5][y], y);
      out[i] = (uint8_t)(k ^ (scramble ? prbs[i] : 0));
    }
  }
}

// FIB CRC (backend/crc.cpp:98-132) and BER re-encode (viterbi_spiral.cpp:128-164) of decoded FIC blocks. One warp per
// block: the decoded bits are packed into 32-bit words with ballots; every lane then re-encodes the trellis steps
// lane, lane + 32, ... from an 8-bit window of that vector (the generators bit-reversed, so no reversal of the window)
// and compares with the sign of the kept soft inputs; the three FIB CRCs run byte-wise from a table in shared memory.
constexpr int POST_WARPS = 8;
constexpr int POST_WORDS = 40; // >= 1 (zero word in front) + ceil((max FIC-like n_bits + 6) / 32) + 1

__global__ void __launch_bounds__(POST_WARPS * 32) k_fic_post(const VitJob * __restrict__ jobs, const FrameDesc * __restrict__ fic_frames, int job_first, int n_jobs,
                                                              const VitProfile * __restrict__ profiles, const unsigned * __restrict__ step_tab,
                                                              const int16_t * __restrict__ soft, const uint8_t * __restrict__ out_bits,
                                                              const uint8_t * __restrict__ prbs, uint8_t * __restrict__ crc_ok, int * __restrict__ ber)
{
  __shared__ unsigned short crc_tab[256];
  __shared__ unsigned vec[POST_WARPS][POST_WORDS];
  {
    // CRC-16/CCITT table, polynomial 0x1021, most significant bit first
    unsigned r = threadIdx.x << 8;
#pragma unroll
    for (int b = 0; b < 8; b++) r = (r & 0x8000u) ? ((r << 1) ^ 0x1021u) : (r << 1);
    crc_tab[threadIdx.x] = (unsigned short)r;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int jl = blockIdx.x * POST_WARPS + warp;
  if (jl >= n_jobs) return;
  VitJob job;
  if (!load_job(jobs, fic_frames, job_first + jl, job)) return;
  if (!(job.flags & VIT_FLAG_FIC)) return;
  const VitProfile & pr = profiles[job.profile];
  const int n_bits = pr.n_bits, steps = n_bits + 6;
  if (steps + 64 > 32 * POST_WORDS) return; // not a FIC-sized block
  const uint8_t * ob = out_bits + job.out;
  const bool scr = (job.flags & VIT_FLAG_PRBS) != 0;
  unsigned * v = vec[warp];
  // v[1 + c] bit b = decoded bit 32 c + b before energy dispersal; zero outside [0, n_bits)
  const int n_words = (steps + 31) / 32 + 2;
  for (int c = 0; c + 1 < n_words; c++)
  {
    const int i = 32 * c + lane;
    const unsigned bit = i < n_bits ? (unsigned)(ob[i] ^ (scr ? prbs[i] : 0)) : 0u;
    const unsigned wv = __ballot_sync(FULL, bit & 1u);
    if (lane == 0) v[1 + c] = wv;
  }
  if (lane == 0) v[0] = 0;
  __syncwarp();
  if (ber != nullptr)
  {
    // window bit j = decoded bit i - 7 + j; the encoder register has bit q = decoded bit i - q, so generator g sees
    // parity(window & reverse8(g)): reverse8 of {109, 79, 83, 109} = {0xB6, 0xF2, 0xCA, 0xB6}
    const unsigned * tab = step_tab + pr.tab_off;
    int errors = 0;
    for (int i = lane; i < steps; i += 32)
    {
      const int p = i - 7 + 32; // bit position of the window start in v[]
      const unsigned long long two = (unsigned long long)v[p >> 5] | ((unsigned long long)v[(p >> 5) + 1] << 32);
      const unsigned win = (unsigned)(two >> (p & 31)) & 0xffu;
      const unsigned e = tab[i];
      int k = (int)(e & 0x0fffffffu);
      const unsigned rp[4] = { 0xB6u, 0xF2u, 0xCAu, 0xB6u };
#pragma unroll
      for (int g = 0; g < 4; g++)
      {
        if (!((e >> (28 + g)) & 1u)) continue;
        const unsigned hard = job_soft(job, soft, k) > 0;
        k++;
        errors += hard != (__popc(win & rp[g]) & 1u);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) errors += __shfl_xor_sync(FULL, errors, o);
    if (lane == 0) { ber[2 * job.aux] = pr.n_kept; ber[2 * job.aux + 1] = errors; }
  }
  if (crc_ok != nullptr && lane < 3 && 256 * (lane + 1) <= n_bits)
  {
    // FIB `lane`: 32 bytes, first bit = most significant; all-ones start, the last two bytes inverted, pass <=> 0
    unsigned reg = 0xffffu;
    for (int b = 0; b < 32; b++)
    {
      const int i = 256 * lane + 8 * b; // multiple of 8: the byte does not straddle words
      unsigned byte = (v[1 + (i >> 5)] >> (i & 31)) & 0xffu;
      byte = __brev(byte) >> 24;                                   // decoded bit i -> bit 7
      byte ^= prbs_byte_msb(prbs, i);                              // the CRC runs on the descrambled bits
      if (b >= 30) byte ^= 0xffu;
      reg = ((reg << 8) & 0xffffu) ^ crc_tab[((reg >> 8) ^ byte) & 0xffu];
    }
    crc_ok[3 * job.aux + lane] = reg == 0;
  }
}
// One Backend (sub-channel of a recording) = one range of per-CIF jobs; the job list of a full ensemble has several hundred
// thousand entries, so it is written here instead of on the host (Backend::_process_segment start-up: logical frame g needs
// CIFs g-16 .. g-1 ... g; rows whose CIF precedes the Backend's creation read zeros, backend.cpp:129-161).
__global__ void __launch_bounds__(128) k_expand_backend_jobs(const BackendJobRange * __restrict__ ranges, VitJob * __restrict__ jobs)
{
  const BackendJobRange r = ranges[blockIdx.x];
  for (int i = threadIdx.x; i < r.n_jobs; i += blockDim.x)
  {
    const int g = r.g_first + i;
    VitJob j;
    j.src = r.src;
    j.out = r.out + (long long)i * r.n_bits;
    j.profile = r.profile;
    j.src_mode = VIT_SRC_TIME_DEINTERLEAVE;
    j.flags = VIT_FLAG_PRBS;
    j.cif_first = g - 16;
    const int lo = max(0, r.g_start - (g - 16));
    j.row_mask = lo >= 16 ? 0 : ((0xFFFF << lo) & 0xFFFF);
    j.frag_off = r.frag_off;
    j.aux = 0;
    j.skip_plus1 = 0;
    jobs[r.job_first + i] = j;
  }
}
// Protection::deconvolve over n logical frames at a constant stride (stage tap): job i reads its fragment at i * src_stride and
// writes at i * n_bits; written on the device because a million 48-byte jobs built and staged by the host cost more than decoding them.
__global__ void __launch_bounds__(256) k_linear_jobs(VitJob * __restrict__ jobs, int n, long long src_stride, int n_bits, int profile)
{
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
  {
    VitJob j;
    j.src = (long long)i * src_stride;
    j.out = (long long)i * n_bits;
    j.profile = profile;
    j.src_mode = VIT_SRC_LINEAR;
    j.flags = 0;
    j.cif_first = 0;
    j.row_mask = 0;
    j.frag_off = 0;
    j.aux = 0;
    j.skip_plus1 = 0;
    jobs[i] = j;
  }
}
// EtiGenerator::_process_sub_channel storage loop (eti_generator.cpp:403-411): 8 decoded bits (one per byte) -> one byte, first bit most significant
__global__ void __launch_bounds__(256) k_pack_bits(const uint8_t * __restrict__ bits, uint8_t * __restrict__ out, long long n_bytes)
{
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_bytes; i += (long long)gridDim.x * blockDim.x)
  {
    const uint2 w = *reinterpret_cast<const uint2 *>(bits + 8 * i);
    // bytes b0..b3 of a word times 0x08040201: the top byte of the product is 8 b0 + 4 b1 + 2 b2 + b3
    out[i] = (uint8_t)(((((w.x & 0x01010101u) * 0x08040201u) >> 24) << 4) | (((w.y & 0x01010101u) * 0x08040201u) >> 24));
  }
}
} // namespace

cudaError_t launch_expand_backend_jobs(cudaStream_t stream, const BackendJobRange * ranges, int n_ranges, VitJob * jobs, unsigned long long * launch_counter)
{
  if (n_ranges <= 0) return cudaSuccess;
  k_expand_backend_jobs<<<(unsigned)n_ranges, 128, 0, stream>>>(ranges, jobs);
  if (launch_counter) (*launch_counter)++;
  return cudaGetLastError();
}

cudaError_t launch_linear_jobs(cudaStream_t stream, VitJob * jobs, int n, long long src_stride, int n_bits, int profile, unsigned long long * launch_counter)
{
  if (n <= 0) return cudaSuccess;
  k_linear_jobs<<<(unsigned)std::min((n + 255) / 256, N_SM * 8), 256, 0, stream>>>(jobs, n, src_stride, n_bits, profile);
  if (launch_counter) (*launch_counter)++;
  return cudaGetLastError();
}

cudaError_t launch_pack_bits(cudaStream_t stream, const uint8_t * bits, uint8_t * out, long long n_bytes, unsigned long long * launch_counter)
{
  if (n_bytes <= 0) return cudaSuccess;
  const long long blocks = (n_bytes + 255) / 256;
  k_pack_bits<<<(unsigned)(blocks < N_SM * 16 ? blocks : N_SM * 16), 256, 0, stream>>>(bits, out, n_bytes);
  if (launch_counter) (*launch_counter)++;
  return cudaGetLastError();
}

int viterbi_smem_bytes(int max_steps, int warps)
{
  const int cap = (max_steps + 15) & ~15;
  return cap * VIT_SMEM_PER_STEP * warps;
}

// Workspace of the thread-per-code-word path for one launch of n_jobs code words of at most max_steps trellis steps:
// symbols u32[rows][stride] + decision words u64[rows][stride], rows = max_steps rounded up to 5, stride = jobs rounded up to 32.
static inline int tpc_rows(int max_steps) { return (max_steps + 4) / 5 * 5; }
constexpr int TPC_READ_AHEAD = 10; // symbol rows k_vit_tpc reads beyond the last block of five
static inline size_t tpc_bytes_per_job(int rows) { return (size_t)(rows + TPC_READ_AHEAD) * 4 + (size_t)rows * 8; }
size_t viterbi_ws_bytes(int n_jobs, int max_steps)
{
  const size_t stride = ((size_t)n_jobs + 31) & ~(size_t)31;
  return tpc_bytes_per_job(tpc_rows(max_steps)) * stride + 256;
}

static cudaError_t launch_viterbi_warp(cudaStream_t stream, const VitJob * jobs, const FrameDesc * fic_frames, int n_jobs, const VitProfile * profiles, int max_steps,
                                       const int16_t * soft, uint8_t * out_bits, const uint8_t * prbs, uint8_t * crc_ok, int * ber,
                                       unsigned long long * launch_counter)
{
  const int cap = (max_steps + 15) & ~15;
  const int per_warp = cap * VIT_SMEM_PER_STEP;
  int warps = 8;
  while (warps > 1 && per_warp * warps > 56 * 1024) warps >>= 1; // <= 56 KB per CTA -> 4 CTAs/SM when possible
  const int smem = per_warp * warps;
  if (smem > 227 * 1024) return cudaErrorInvalidValue;
  const LaunchProps lp = launch_props((const void *)k_viterbi, warps * 32, (size_t)smem, 227 * 1024); // opt-in once per device
  if (lp.err != cudaSuccess) return lp.err;
  const int ctas_needed = (n_jobs + warps - 1) / warps;
  const int per_sm = max(1, min(16, (227 * 1024) / max(smem, 1)));
  const int grid = min(ctas_needed, N_SM * per_sm);
  k_viterbi<<<grid, warps * 32, smem, stream>>>(jobs, fic_frames, n_jobs, profiles, soft, out_bits, prbs, crc_ok, ber, cap);
  if (launch_counter) (*launch_counter)++;
  return cudaGetLastError();
}

// Batches of at least VIT_TPC_MIN_JOBS code words take the thread-per-code-word path (in chunks that fit the workspace);
// small batches (single frames while a recording acquires lock, stage taps on a handful of code words) keep one warp
// per code word, which has the shorter latency. Both produce the reference's bits exactly.
constexpr int VIT_TPC_MIN_JOBS = 2048;

cudaError_t launch_viterbi(cudaStream_t stream, const VitJob * jobs, const FrameDesc * fic_frames, int n_jobs, const VitProfile * profiles, int max_steps,
                           const int16_t * soft, uint8_t * out_bits, const uint8_t * prbs, uint8_t * crc_ok, int * ber,
                           const unsigned * step_tab, void * ws, size_t ws_bytes, unsigned long long * launch_counter, const VitSpanHook * hook)
{
  if (n_jobs <= 0) return cudaSuccess;
  const int rows = tpc_rows(max_steps);
  const size_t per_job = tpc_bytes_per_job(rows);
  size_t fit = ws != nullptr && ws_bytes > 256 ? (ws_bytes - 256) / per_job : 0;
  fit &= ~(size_t)31;
  // DABSTAR_VITERBI_TPC_MIN overrides the batch size from which the thread-per-code-word path is taken (read per launch
  // so the parity tests can run every case through both kernels)
  int min_jobs = VIT_TPC_MIN_JOBS;
  if (const char * ev = getenv("DABSTAR_VITERBI_TPC_MIN")) min_jobs = atoi(ev);
  if (n_jobs < min_jobs || fit < 32 || step_tab == nullptr)
  {
    if (hook) hook->mark(hook->user, 3, stream);
    const cudaError_t e = launch_viterbi_warp(stream, jobs, fic_frames, n_jobs, profiles, max_steps, soft, out_bits, prbs, crc_ok, ber, launch_counter);
    if (hook) hook->mark(hook->user, 2, stream);
    return e;
  }
  const int chunk = (int)min((size_t)((n_jobs + 31) & ~31), fit);
  unsigned * sym = static_cast<unsigned *>(ws);
  unsigned long long * surv = reinterpret_cast<unsigned long long *>(static_cast<unsigned char *>(ws) + (((size_t)(rows + TPC_READ_AHEAD) * chunk * 4 + 255) & ~(size_t)255));
  for (int first = 0; first < n_jobs; first += chunk)
  {
    const int n = min(chunk, n_jobs - first);
    const int groups = (n + 31) / 32;
    const dim3 ggrid((unsigned)groups, (unsigned)((rows + GATHER_STEPS - 1) / GATHER_STEPS));
    if (hook) hook->mark(hook->user, 0, stream);
    k_vit_gather_kb<<<ggrid, 256, 0, stream>>>(jobs, fic_frames, first, n, profiles, step_tab, soft, sym, chunk, rows);
    if (hook) hook->mark(hook->user, 1, stream);
    k_vit_tpc<<<groups, 32, 0, stream>>>(jobs, fic_frames, first, n, profiles, sym, surv, chunk, out_bits, prbs);
    if (hook) hook->mark(hook->user, 2, stream);
    if (launch_counter) (*launch_counter) += 2;
    if (crc_ok != nullptr || ber != nullptr)
    {
      k_fic_post<<<(n + POST_WARPS - 1) / POST_WARPS, POST_WARPS * 32, 0, stream>>>(jobs, fic_frames, first, n, profiles, step_tab, soft, out_bits, prbs, crc_ok, ber);
      if (launch_counter) (*launch_counter)++;
    }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
} // namespace dab
