// pfec.cuh — packet-mode FEC of a DAB sub-channel: where the FEC frames lie in a packet stream, the code table of one frame and
// the RS(204,188) decoder of its rows, as functions the device pass (pfec_kernels.cu) and the host tests share.
//
// Source: ETSI EN 300 401 clause 5.3.5 (FEC for packet mode) and clause 6.2.2 (FIG 0/14). The layout below was written from the
// standard's text; it is not replayed against another implementation. Every layout fact lives in exactly one function here.
//   - An FEC frame is an Application Data Table (ADT) of 2256 bytes (94 slots of 24 bytes, whole packets, padding packets
//     included) followed by 9 FEC packets of 24 bytes: 103 slots. It starts and ends on a 24-byte slot boundary of the packet
//     stream, anywhere inside a logical frame, and usually spans several logical frames.
//   - An FEC packet has a 2-byte header (packet length 00, continuity index, first / last flags, address 1022) and 22 bytes of RS
//     data; the 9 packets carry the 192 RS bytes and 6 padding bytes. Their headers are not covered by the code. The first / last
//     flags of the nine mark them as one run: first (10), seven intermediate (00), last (01).
//   - The ADT and the RS data form a 12 x 204 table filled column by column: ADT byte k is row k mod 12, column k / 12; RS byte j
//     is row j mod 12, column 188 + j / 12. Each row is a code word of RS(204,188), shortened from RS(255,239) (51 leading zero
//     bytes, 188 information bytes, 16 parity bytes), field x^8 + x^4 + x^3 + x^2 + 1, generator roots alpha^0..alpha^15: up to 8
//     byte errors per row are corrected, and a burst of up to 96 stream bytes costs each row at most 8 bytes.
//
// Locating the FEC frames (one decision per slot, no walk). Slot s+k *fits* position k of a run when its first two bytes read
// packet length 00 and address 1022 and its first / last flags are those of position k (10 for k = 0, 01 for k = 8, 00 between).
// score(s) counts the positions k = 0..8 that slot s+k fits (slots outside the stream fit nothing). Slot s starts a run when
// score(s) >= 6, score(s) > score(s-1) and score(s) >= score(s+1). Headers alone cannot tell the two ends of a run apart when
// they differ only by the flags, so the flags take part: with the length and address alone, a run whose last header is damaged
// would be found one slot early. With up to two damaged headers per run, or three that are not the first, the last and one
// beside them, the start is found exactly. The FEC frame is the 94 slots before the run and the run. A frame is INCOMPLETE (it
// is listed but not corrected) when the stream starts fewer than 94 slots before its run, when its run is cut by the end of the
// stream, or when the previous run starts fewer than 103 slots before it (that run lies inside its ADT).
#pragma once
#include <cstdint>

namespace dab
{
constexpr int PFEC_SLOT = 24;          // bytes per slot
constexpr int PFEC_ADT_SLOTS = 94;     // slots of the Application Data Table (2256 bytes)
constexpr int PFEC_RUN = 9;            // FEC packets per frame
constexpr int PFEC_FRAME_SLOTS = PFEC_ADT_SLOTS + PFEC_RUN;
constexpr int PFEC_ROWS = 12, PFEC_K = 188, PFEC_N = 204, PFEC_ROOTS = 16, PFEC_T = 8, PFEC_PAD = 51;
constexpr int PFEC_ADDRESS = 1022;
constexpr int PFEC_MIN_SCORE = 6;
// status of an FEC frame
enum : int
{
  PFEC_CLEAN = 0,      // every row a code word
  PFEC_CORRECTED = 1,  // some rows corrected, none failed
  PFEC_PARTIAL = 2,    // some rows had more than 8 errors and were left as received
  PFEC_INCOMPLETE = 3, // cut by the stream's start or end or overlapped by the previous frame: not corrected
};

// The fit code of one slot: 0 when its header is not an FEC packet header, else 1 + its first / last flags
__host__ __device__ inline int pfec_slot_code(const uint8_t * p)
{
  if ((p[0] >> 6) != 0 || (((p[0] & 3u) << 8) | p[1]) != (unsigned)PFEC_ADDRESS) return 0;
  return 1 + ((p[0] >> 2) & 3);
}
// The first / last flags of position k of a run
__host__ __device__ inline int pfec_run_flags(int k) { return k == 0 ? 2 : k == PFEC_RUN - 1 ? 1 : 0; }
// score(s) over the fit codes of the n slots of a stream
__host__ __device__ inline int pfec_score(const uint8_t * code, long long n, long long s)
{
  int c = 0;
  for (int k = 0; k < PFEC_RUN; k++)
  {
    const long long i = s + k;
    if (i >= 0 && i < n && code[i] == 1 + pfec_run_flags(k)) c++;
  }
  return c;
}
__host__ __device__ inline bool pfec_run_start(const uint8_t * code, long long n, long long s)
{
  const int c = pfec_score(code, n, s);
  return c >= PFEC_MIN_SCORE && c > pfec_score(code, n, s - 1) && c >= pfec_score(code, n, s + 1);
}
// The frame of the run at slot `run`, prev: the previous run's slot (-1 none), n: slots of the stream
__host__ __device__ inline bool pfec_incomplete(long long run, long long prev, long long n)
{
  return run < PFEC_ADT_SLOTS || run + PFEC_RUN > n || (prev >= 0 && run - prev < PFEC_FRAME_SLOTS);
}
// Stream byte of column c of row r of the frame whose run is at slot `run` (ADT bytes for c < 188, RS bytes above)
__host__ __device__ inline long long pfec_byte(long long run, int r, int c)
{
  if (c < PFEC_K) return (run - PFEC_ADT_SLOTS) * PFEC_SLOT + 12LL * c + r;
  const int j = 12 * (c - PFEC_K) + r; // RS byte j: FEC packet j / 22, after its 2-byte header
  return (run + j / 22) * PFEC_SLOT + 2 + j % 22;
}

// GF(2^8) with x^8 + x^4 + x^3 + x^2 + 1; mulr[j][x] = x alpha^j (the syndrome Horner steps)
struct PfecTables
{
  uint8_t exp[512], log[256];
  uint8_t mulr[PFEC_ROOTS][256];
};
__host__ __device__ inline void pfec_tables(PfecTables & t)
{
  unsigned x = 1;
  for (int i = 0; i < 255; i++)
  {
    t.exp[i] = t.exp[i + 255] = (uint8_t)x;
    t.log[x] = (uint8_t)i;
    x <<= 1;
    if (x & 0x100) x ^= 0x11d;
  }
  t.exp[510] = t.exp[511] = 0;
  t.log[0] = 0;
  for (int j = 0; j < PFEC_ROOTS; j++)
    for (int v = 0; v < 256; v++) t.mulr[j][v] = v == 0 ? 0 : t.exp[t.log[v] + j];
}
__host__ __device__ inline unsigned pfec_mul(const PfecTables & t, unsigned a, unsigned b) { return (a && b) ? t.exp[t.log[a] + t.log[b]] : 0u; }

// One row: get(c) reads column c (0..203). Returns the number of corrected bytes (0..8) and their columns and values in col[] /
// val[] (the caller XORs them in), or -1 when the row has more than 8 errors (nothing to apply).
template <typename Get>
__host__ __device__ inline int pfec_row_decode(const PfecTables & t, Get get, int (&col)[PFEC_T], uint8_t (&val)[PFEC_T])
{
  unsigned syn[PFEC_ROOTS];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int j = 0; j < PFEC_ROOTS; j++) syn[j] = 0;
  for (int c = 0; c < PFEC_N; c++)
  {
    const unsigned d = get(c);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int j = 0; j < PFEC_ROOTS; j++) syn[j] = d ^ t.mulr[j][syn[j]];
  }
  uint8_t S[PFEC_ROOTS]; // the rest indexes the syndromes by value
  unsigned any = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int j = 0; j < PFEC_ROOTS; j++) { any |= syn[j]; S[j] = (uint8_t)syn[j]; }
  if (!any) return 0;
  // Berlekamp-Massey: the error locator lambda (lambda[0] = 1) of degree L
  uint8_t lambda[PFEC_ROOTS + 1] = { 1 }, prev[PFEC_ROOTS + 1] = { 1 };
  int L = 0, m = 1;
  unsigned b = 1;
  for (int n = 0; n < PFEC_ROOTS; n++)
  {
    unsigned d = S[n];
    for (int i = 1; i <= L; i++) d ^= pfec_mul(t, lambda[i], S[n - i]);
    if (d == 0) { m++; continue; }
    const unsigned coef = t.exp[t.log[d] + 255 - t.log[b]]; // d / b
    uint8_t keep[PFEC_ROOTS + 1];
    for (int i = 0; i <= PFEC_ROOTS; i++) keep[i] = lambda[i];
    for (int i = m; i <= PFEC_ROOTS; i++) lambda[i] ^= (uint8_t)pfec_mul(t, coef, prev[i - m]);
    if (2 * L <= n)
    {
      L = n + 1 - L;
      for (int i = 0; i <= PFEC_ROOTS; i++) prev[i] = keep[i];
      b = d;
      m = 1;
    }
    else m++;
  }
  if (L > PFEC_T) return -1;
  for (int i = L + 1; i <= PFEC_ROOTS; i++) if (lambda[i]) return -1;
  // omega = syn(x) lambda(x) mod x^16
  uint8_t omega[PFEC_ROOTS];
  for (int i = 0; i < PFEC_ROOTS; i++)
  {
    unsigned v = 0;
    for (int j = 0; j <= i && j <= L; j++) v ^= pfec_mul(t, lambda[j], S[i - j]);
    omega[i] = (uint8_t)v;
  }
  // Chien search over the 204 positions of the shortened code (column c has locator X = alpha^(203 - c)), Forney:
  // e = X omega(1/X) / lambda'(1/X) for roots alpha^0.. (fcr 0)
  int found = 0;
  for (int c = 0; c < PFEC_N; c++)
  {
    const int xinv = (255 - (PFEC_N - 1 - c)) % 255; // log of 1/X
    unsigned s = 0, dl = 0;
    for (int i = 0; i <= L; i++)
    {
      if (!lambda[i]) continue;
      const unsigned term = t.exp[(t.log[lambda[i]] + xinv * i) % 255];
      s ^= term;
      if (i & 1) dl ^= t.exp[(t.log[lambda[i]] + xinv * (i - 1)) % 255];
    }
    if (s) continue;
    if (found == PFEC_T || !dl) return -1;
    unsigned om = 0;
    for (int i = 0; i < PFEC_ROOTS; i++)
      if (omega[i]) om ^= t.exp[(t.log[omega[i]] + xinv * i) % 255];
    const int lx = PFEC_N - 1 - c;
    const unsigned e = om ? t.exp[(t.log[om] + lx + 255 - t.log[dl]) % 255] : 0u;
    if (!e) return -1;
    col[found] = c;
    val[found] = (uint8_t)e;
    found++;
  }
  return found == L ? found : -1;
}
} // namespace dab
