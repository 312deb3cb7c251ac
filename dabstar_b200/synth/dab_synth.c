/* dab_synth — bundled synthetic DAB Mode-I transmitter (test-signal generator, host C + OpenMP).
 *
 * Produces what BASELINE.json's configs ask for: random FIC/MSC payloads -> FIB CRC -> energy dispersal
 * -> K=7 rate-1/4 convolutional code -> puncturing (FIC / EEP / UEP) -> 16-CIF time interleaving ->
 * CIF multiplex -> frequency interleaving -> pi/4-DQPSK against the phase reference symbol -> 2048-pt
 * IFFT -> 504-sample cyclic prefix -> null symbol -> carrier offset + AWGN -> cf32 / u8 / i16 IQ at
 * 2.048 MS/s. It is the inverse of the receive chain described in SURVEY.md section 8(a) and follows
 * ETSI EN 300 401 (tables restated from the standard; the reference has no transmitter).
 *
 * This is a signal source for tests and benchmarks, not part of the decode path.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#ifdef _OPENMP
#include <omp.h>
#endif

enum { TU = 2048, TG = 504, TS = 2552, TNULL = 2656, TF = 196608, KC = 1536, SYM_BITS = 3072, CIF_BITS = 55296, FS = 2048000 };

typedef struct { float re, im; } cf;

typedef struct
{
  int32_t  n_frames;
  int32_t  format;        /* 0 = cf32, 1 = u8 (v*128+127.38), 2 = i16 (v*32768) */
  uint64_t seed;
  float    snr_db;        /* >= 100: no noise */
  float    cfo_hz;        /* carrier offset applied to the whole stream */
  float    rms;           /* RMS amplitude of the data symbols in full-scale units (e.g. 0.25) */
  int32_t  lead_samples;  /* noise-like filler before the first null symbol */
  int32_t  tail_samples;  /* filler after the last frame (lets the receiver finish the last frame) */
  int32_t  n_subch;
  const int32_t * subch;  /* n_subch x 7: subChId,startCU,sizeCU,shortForm,protLevel,bitRate,(unused) */
  int32_t  fig_mode;      /* 0: random FIB payloads; 1: MCI of the configured ensemble (FIG 0/0 with a running CIF counter,
                             FIG 0/1 per sub-channel, FIG 0/2 one audio service per sub-channel), EN 300 401 clauses 6.2-6.4 */
  int32_t  eid;           /* ensemble identifier for fig_mode 1 */
  int32_t  tii_main;      /* fig_mode 1: transmitter identification sent in the null symbol after every frame whose CIF counter has */
  int32_t  tii_sub;       /*   (count & 7) >= 4 (EN 300 401 clause 14.8): main id 0..69 (pattern), sub id 0..23 (comb); -1: no TII */
  const uint8_t * const * msc_payload; /* NULL, or n_subch pointers: the logical frames sub-channel s carries, n_frames*4*24*bitRate bits
                                          (one per byte, transmit order), or NULL for random bits (drawn as if no payload were given) */
  int32_t  n_packet;      /* fig_mode 1: packet-mode components (0: none, and the FIC is what it is without them) */
  const int32_t * packet; /*   n_packet x 5: subChId, SCId, packet address, DSCTy, DG flag. A listed sub-channel carries no programme
                               service; each entry becomes a data service with one TMId 3 component (FIG 0/2, P/D 1) and a FIG 0/3 entry */
  int32_t  n_fec;         /* fig_mode 1: sub-channels flagged with packet-mode FEC (0: none, and the FIC is what it is without them) */
  const int32_t * fec;    /*   n_fec subChIds, each sent as a FIG 0/14 entry with FEC scheme 1 (EN 300 401 clause 6.2.2) */
} dabsynth_cfg;

/* ---------------------------------------------------------------------------------------------- rng */
static inline uint64_t mix64(uint64_t z)
{
  z += 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}
typedef struct { uint64_t s; } rng_t;
static inline uint64_t rng_next(rng_t * r) { r->s += 0x9e3779b97f4a7c15ull; return mix64(r->s); }
static inline rng_t rng_make(uint64_t seed, uint64_t a, uint64_t b) { rng_t r = { mix64(seed ^ mix64(a * 0x100000001b3ull + b)) }; return r; }
static inline float rng_unit(rng_t * r) { return (float)((rng_next(r) >> 40) + 1) * (1.0f / 16777217.0f); } /* (0,1) */
static inline void rng_gauss2(rng_t * r, float * a, float * b)
{
  const float u = rng_unit(r), v = rng_unit(r);
  const float m = sqrtf(-2.0f * logf(u));
  *a = m * cosf(6.28318530718f * v);
  *b = m * sinf(6.28318530718f * v);
}

/* ---------------------------------------------------------------------------------------------- tables */
static const uint32_t PI_MASK[24] = {
  0x11111113u, 0x11131113u, 0x11131313u, 0x13131313u, 0x13131333u, 0x13331333u, 0x13333333u, 0x33333333u,
  0x33333337u, 0x33373337u, 0x33373737u, 0x37373737u, 0x37373777u, 0x37773777u, 0x37777777u, 0x77777777u,
  0x7777777fu, 0x777f777fu, 0x777f7f7fu, 0x7f7f7f7fu, 0x7f7f7fffu, 0x7fff7fffu, 0x7fffffffu, 0xffffffffu };

typedef struct { int16_t bitrate, level, L[4], PI[4]; } uep_row;
static const uep_row UEP_TABLE[] = {
  {32,5, {3,4,17,0}, {5,3,2,0}}, {32,4, {3,3,18,0}, {11,6,5,0}}, {32,3, {3,4,14,3}, {15,9,6,8}},
  {32,2, {3,4,14,3}, {22,13,8,13}}, {32,1, {3,5,13,3}, {24,17,12,17}}, {48,5, {4,3,26,3}, {5,4,2,3}},
  {48,4, {3,4,26,3}, {9,6,4,6}}, {48,3, {3,4,26,3}, {15,10,6,9}}, {48,2, {3,4,26,3}, {24,14,8,15}},
  {48,1, {3,5,25,3}, {24,18,13,18}}, {56,5, {6,10,23,3}, {5,4,2,3}}, {56,4, {6,10,23,3}, {9,6,4,5}},
  {56,3, {6,12,21,3}, {16,7,6,9}}, {56,2, {6,10,23,3}, {23,13,8,13}}, {64,5, {6,9,31,2}, {5,3,2,3}},
  {64,4, {6,9,33,0}, {11,6,5,0}}, {64,3, {6,12,27,3}, {16,8,6,9}}, {64,2, {6,10,29,3}, {23,13,8,13}},
  {64,1, {6,11,28,3}, {24,18,12,18}}, {80,5, {6,10,41,3}, {6,3,2,3}}, {80,4, {6,10,41,3}, {11,6,5,6}},
  {80,3, {6,11,40,3}, {16,8,6,7}}, {80,2, {6,10,41,3}, {23,13,8,13}}, {80,1, {6,10,41,3}, {24,7,12,18}},
  {96,5, {7,9,53,3}, {5,4,2,4}}, {96,4, {7,10,52,3}, {9,6,4,6}}, {96,3, {6,12,51,3}, {16,9,6,10}},
  {96,2, {6,10,53,3}, {22,12,9,12}}, {96,1, {6,13,50,3}, {24,18,13,19}}, {112,5, {14,17,50,3}, {5,4,2,5}},
  {112,4, {11,21,49,3}, {9,6,4,8}}, {112,3, {11,23,47,3}, {16,8,6,9}}, {112,2, {11,21,49,3}, {23,12,9,14}},
  {128,5, {12,19,62,3}, {5,3,2,4}}, {128,4, {11,21,61,3}, {11,6,5,7}}, {128,3, {11,22,60,3}, {16,9,6,10}},
  {128,2, {11,21,61,3}, {22,12,9,14}}, {128,1, {11,20,62,3}, {24,17,13,19}}, {160,5, {11,19,87,3}, {5,4,2,4}},
  {160,4, {11,23,83,3}, {11,6,5,9}}, {160,3, {11,24,82,3}, {16,8,6,11}}, {160,2, {11,21,85,3}, {22,11,9,13}},
  {160,1, {11,22,84,3}, {24,18,12,19}}, {192,5, {11,20,110,3}, {6,4,2,5}}, {192,4, {11,22,108,3}, {10,6,4,9}},
  {192,3, {11,24,106,3}, {16,10,6,11}}, {192,2, {11,20,110,3}, {22,13,9,13}}, {192,1, {11,21,109,3}, {24,20,13,24}},
  {224,5, {12,22,131,3}, {8,6,2,6}}, {224,4, {12,26,127,3}, {12,8,4,11}}, {224,3, {11,20,134,3}, {16,10,7,9}},
  {224,2, {11,22,132,3}, {24,16,10,15}}, {224,1, {11,24,130,3}, {24,20,12,20}}, {256,5, {11,24,154,3}, {6,5,2,5}},
  {256,4, {11,24,154,3}, {12,9,5,10}}, {256,3, {11,27,151,3}, {16,10,7,10}}, {256,2, {11,22,156,3}, {24,14,10,13}},
  {256,1, {11,26,152,3}, {24,19,14,18}}, {320,5, {11,26,200,3}, {8,5,2,6}}, {320,4, {11,25,201,3}, {13,9,5,10}},
  {320,2, {11,26,200,3}, {24,17,9,17}}, {384,5, {11,27,247,3}, {8,6,2,7}}, {384,3, {11,24,250,3}, {16,9,7,10}},
  {384,1, {12,28,245,3}, {24,20,14,23}} };
#define N_UEP ((int)(sizeof(UEP_TABLE) / sizeof(UEP_TABLE[0])))

static const uint8_t PRS_ROW[48] = { 0,1,2,3, 0,1,2,3, 0,1,2,3, 0,1,2,3, 0,1,2,3, 0,1,2,3,
                                     0,3,2,1, 0,3,2,1, 0,3,2,1, 0,3,2,1, 0,3,2,1, 0,3,2,1 };
static const uint8_t PRS_N[48] = { 1,2,0,1, 3,2,2,3, 2,1,2,3, 1,2,3,3, 2,2,2,1, 1,3,1,2,
                                   3,1,1,1, 2,2,1,0, 2,2,3,3, 0,2,1,3, 3,3,3,0, 3,0,1,1 };
static const uint8_t PRS_H[4][32] = {
  { 0,2,0,0,0,0,1,1,2,0,0,0,2,2,1,1, 0,2,0,0,0,0,1,1,2,0,0,0,2,2,1,1 },
  { 0,3,2,3,0,1,3,0,2,1,2,3,2,3,3,0, 0,3,2,3,0,1,3,0,2,1,2,3,2,3,3,0 },
  { 0,0,0,2,0,2,1,3,2,2,0,2,2,0,1,3, 0,0,0,2,0,2,1,3,2,2,0,2,2,0,1,3 },
  { 0,1,2,1,0,3,3,2,2,3,2,1,2,1,3,2, 0,1,2,1,0,3,3,2,2,3,2,1,2,1,3,2 } };
static const int TIME_MAP[16] = { 0, 8, 4, 12, 2, 10, 6, 14, 1, 9, 5, 13, 3, 11, 7, 15 };

static int16_t g_bin[KC];        /* interleaved carrier k -> fft bin in [-768,768]\{0} */
static uint8_t g_prs_q[TU];      /* quadrant of the PRS per fft index, 255 = unused bin */
static uint8_t g_prbs[9216];
static cf g_tw[TU / 2];
static uint16_t g_rev[TU];
static int g_ready = 0;

static void init_tables(void)
{
  if (g_ready) return;
  int n = 0, v = 0;
  for (int i = 0; i < TU; i++)
  {
    if (i > 0) v = (13 * v + 511) % TU;
    if (v == TU / 2 || v < 256 || v > 256 + KC) continue;
    g_bin[n++] = (int16_t)(v - TU / 2);
  }
  memset(g_prs_q, 255, sizeof(g_prs_q));
  for (int k = -768; k <= 768; k++)
  {
    if (k == 0) continue;
    const int blk = k < 0 ? (k + 768) / 32 : 24 + (k - 1) / 32;
    const int kmin = k < 0 ? -768 + 32 * blk : 1 + 32 * (blk - 24);
    g_prs_q[k < 0 ? k + TU : k] = (uint8_t)((PRS_H[PRS_ROW[blk]][k - kmin] + PRS_N[blk]) & 3);
  }
  unsigned reg = 0x1ff;
  for (int i = 0; i < 9216; i++)
  {
    const unsigned b = ((reg >> 8) ^ (reg >> 4)) & 1u;
    reg = ((reg << 1) | b) & 0x1ff;
    g_prbs[i] = (uint8_t)b;
  }
  for (int k = 0; k < TU / 2; k++)
  {
    g_tw[k].re = (float)cos(2.0 * M_PI * k / TU);
    g_tw[k].im = (float)sin(2.0 * M_PI * k / TU);
  }
  for (int i = 0; i < TU; i++)
  {
    int r = 0;
    for (int b = 0; b < 11; b++) if (i & (1 << b)) r |= 1 << (10 - b);
    g_rev[i] = (uint16_t)r;
  }
  g_ready = 1;
}

/* in-place inverse DFT (sign +), unnormalised */
static void ifft2048(cf * x)
{
  for (int i = 0; i < TU; i++)
  {
    const int r = g_rev[i];
    if (r > i) { const cf t = x[i]; x[i] = x[r]; x[r] = t; }
  }
  for (int len = 2; len <= TU; len <<= 1)
  {
    const int half = len / 2, step = TU / len;
    for (int s = 0; s < TU; s += len)
      for (int k = 0; k < half; k++)
      {
        const cf w = g_tw[k * step];
        const cf b = x[s + k + half];
        const cf t = { b.re * w.re - b.im * w.im, b.re * w.im + b.im * w.re };
        x[s + k + half].re = x[s + k].re - t.re; x[s + k + half].im = x[s + k].im - t.im;
        x[s + k].re += t.re; x[s + k].im += t.im;
      }
  }
}

/* ---------------------------------------------------------------------------------------------- coding */
static inline int parity8(unsigned x) { x ^= x >> 4; x ^= x >> 2; x ^= x >> 1; return (int)(x & 1u); }

/* Mother code: n info bits + 6 zero tail bits -> 4(n+6) coded bits, generators 133,171,145,133 octal
 * written here in the bit order the receiver re-encodes with (109,79,83,109 on a left-shifting register). */
static void conv_encode(const uint8_t * in, int n, uint8_t * out)
{
  static const unsigned poly[4] = { 109, 79, 83, 109 };
  unsigned sr = 0;
  for (int i = 0; i < n + 6; i++)
  {
    sr = ((sr << 1) | (i < n ? in[i] : 0u)) & 0xff;
    for (int j = 0; j < 4; j++) out[4 * i + j] = (uint8_t)parity8(sr & poly[j]);
  }
}

static int puncture_blocks(const uint8_t * mother, int * pos, uint8_t * out, int n, int blocks, int pi)
{
  for (int b = 0; b < blocks; b++)
    for (int j = 0; j < 128; j++)
    {
      if ((PI_MASK[pi - 1] >> (j & 31)) & 1u) out[n++] = mother[*pos];
      (*pos)++;
    }
  return n;
}
static int puncture_tail(const uint8_t * mother, int * pos, uint8_t * out, int n)
{
  for (int j = 0; j < 24; j++)
  {
    if ((PI_MASK[7] >> j) & 1u) out[n++] = mother[*pos];
    (*pos)++;
  }
  return n;
}

static int profile_segments(int short_form, int bit_rate, int prot_level, int L[4], int P[4])
{
  memset(L, 0, sizeof(int) * 4); memset(P, 0, sizeof(int) * 4);
  if (short_form)
  {
    int idx = -1;
    for (int i = 0; i < N_UEP; i++) if (UEP_TABLE[i].bitrate == bit_rate && UEP_TABLE[i].level == prot_level) { idx = i; break; }
    if (idx < 0) return -1;
    for (int s = 0; s < 4; s++) { L[s] = UEP_TABLE[idx].L[s]; P[s] = UEP_TABLE[idx].PI[s]; }
    return 0;
  }
  const int level = prot_level & 3;
  if ((prot_level & 4) == 0)
  {
    const int nn = bit_rate / 8;
    switch (level)
    {
    case 0: L[0] = 6 * nn - 3; L[1] = 3; P[0] = 24; P[1] = 23; break;
    case 1: if (nn == 1) { L[0] = 5; L[1] = 1; P[0] = 13; P[1] = 12; } else { L[0] = 2 * nn - 3; L[1] = 4 * nn + 3; P[0] = 14; P[1] = 13; } break;
    case 2: L[0] = 6 * nn - 3; L[1] = 3; P[0] = 8; P[1] = 7; break;
    default: L[0] = 4 * nn - 3; L[1] = 2 * nn + 3; P[0] = 3; P[1] = 2; break;
    }
  }
  else
  {
    static const int8_t pb[4][2] = { {10, 9}, {6, 5}, {4, 3}, {2, 1} };
    L[0] = 24 * (bit_rate / 32) - 3; L[1] = 3; P[0] = pb[level][0]; P[1] = pb[level][1];
  }
  return 0;
}

static uint16_t crc16(const uint8_t * bits, int n)
{
  unsigned reg = 0xffff;
  for (int i = 0; i < n; i++)
  {
    const unsigned fb = ((reg >> 15) & 1u) ^ bits[i];
    reg = (reg << 1) & 0xffff;
    if (fb) reg ^= 0x1021;
  }
  return (uint16_t)(~reg & 0xffff);
}

/* ---------------------------------------------------------------------------------------------- API */
int64_t dabsynth_num_samples(const dabsynth_cfg * c)
{
  return (int64_t)c->lead_samples + (int64_t)c->n_frames * TF + (int64_t)c->tail_samples;
}

/* ---- FIC content for fig_mode 1 (EN 300 401 clause 5.2.2 FIG structure, 6.4.1 FIG 0/0, 6.2.1 FIG 0/1, 6.3.1 FIG 0/2) ---- */
/* index into EN 300 401 table 8 (bit rate, protection level) -> short-form table index, -1 if the pair is not in the table */
static const int16_t T8_RATE[14] = { 32, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320, 384 };
static int table8_index(int bit_rate, int level)
{
  int idx = 0;
  for (int r = 0; r < 14; r++)
    for (int l = 5; l >= 1; l--)
    {
      /* pairs the table leaves out: 56/1, 112/1, 320/3, 320/1, 384/4, 384/2 */
      const int rate = T8_RATE[r];
      if ((rate == 56 && l == 1) || (rate == 112 && l == 1) || (rate == 320 && (l == 3 || l == 1)) || (rate == 384 && (l == 4 || l == 2))) continue;
      if (rate == bit_rate && l == level) return idx;
      idx++;
    }
  return -1;
}

typedef struct { uint8_t b[12][30]; int fib, used; } fic_writer;

static void ficw_init(fic_writer * w) { memset(w->b, 0, sizeof(w->b)); w->fib = 0; w->used = 0; }
/* room for a FIG of `bytes` bytes in the current FIB, else close it (end marker) and move on; NULL when the FIC is full */
static uint8_t * ficw_reserve(fic_writer * w, int bytes)
{
  if (w->used + bytes > 30)
  {
    if (w->used < 30) w->b[w->fib][w->used] = 0xFF;
    w->fib++;
    w->used = 0;
  }
  if (w->fib >= 12) return NULL;
  uint8_t * p = &w->b[w->fib][w->used];
  w->used += bytes;
  return p;
}
static void ficw_finish(fic_writer * w)
{
  if (w->fib < 12 && w->used < 30) w->b[w->fib][w->used] = 0xFF;
  for (int f = w->fib + 1; f < 12; f++) w->b[f][0] = 0xFF;
}

/* The 12 FIBs (30 bytes each, CRC not included) of frame f */
static int build_mci(const dabsynth_cfg * c, int f, fic_writer * w)
{
  ficw_init(w);
  const int cif = (4 * f) % 5000;
  uint8_t * p = ficw_reserve(w, 6);
  p[0] = (0 << 5) | 5;                                  /* FIG type 0, length 5 */
  p[1] = 0;                                             /* C/N 0, OE 0, P/D 0, extension 0 */
  p[2] = (uint8_t)(c->eid >> 8); p[3] = (uint8_t)c->eid;
  p[4] = (uint8_t)((0 << 6) | (0 << 5) | ((cif / 250) & 31)); /* change flags 0, alarm 0, CIF count high */
  p[5] = (uint8_t)(cif % 250);
  /* FIG 0/1: as many sub-channels per FIG as fit into the FIB */
  int i = 0;
  while (i < c->n_subch)
  {
    int room = 30 - w->used;
    if (room < 2 + 4) room = 30;
    int n = 0, bytes = 2;
    while (i + n < c->n_subch)
    {
      const int add = c->subch[7 * (i + n) + 3] ? 3 : 4;
      if (bytes + add > room) break;
      bytes += add; n++;
    }
    p = ficw_reserve(w, bytes);
    if (!p || n == 0) return -1;
    p[0] = (uint8_t)((0 << 5) | (bytes - 1));
    p[1] = 1;
    uint8_t * q = p + 2;
    for (int k = 0; k < n; k++, i++)
    {
      const int32_t * s = c->subch + 7 * i;
      q[0] = (uint8_t)((s[0] << 2) | ((s[1] >> 8) & 3));
      q[1] = (uint8_t)(s[1] & 0xff);
      if (s[3])
      {
        const int ti = table8_index(s[5], s[4]);
        if (ti < 0) return -1;
        q[2] = (uint8_t)((0 << 7) | (0 << 6) | ti);     /* short form, table switch 0 */
        q += 3;
      }
      else
      {
        const int option = (s[4] & 4) ? 1 : 0, level = s[4] & 3;
        q[2] = (uint8_t)((1 << 7) | (option << 4) | (level << 2) | ((s[2] >> 8) & 3));
        q[3] = (uint8_t)(s[2] & 0xff);
        q += 4;
      }
    }
  }
  /* FIG 0/2: one programme service with one stream-audio component per sub-channel that carries no packet-mode component */
  int prog[c->n_subch > 0 ? c->n_subch : 1], n_prog = 0;
  for (int j = 0; j < c->n_subch; j++)
  {
    int packet = 0;
    for (int e = 0; e < c->n_packet; e++) packet |= c->packet[5 * e] == c->subch[7 * j];
    if (!packet) prog[n_prog++] = j;
  }
  i = 0;
  while (i < n_prog)
  {
    int room = 30 - w->used;
    if (room < 2 + 5) room = 30;
    int n = (room - 2) / 5;
    if (n > n_prog - i) n = n_prog - i;
    p = ficw_reserve(w, 2 + 5 * n);
    if (!p || n == 0) return -1;
    p[0] = (uint8_t)((0 << 5) | (1 + 5 * n));
    p[1] = 2;
    uint8_t * q = p + 2;
    for (int k = 0; k < n; k++, i++, q += 5)
    {
      const int32_t * s = c->subch + 7 * prog[i];
      const int sid = 0xD000 + s[0];
      q[0] = (uint8_t)(sid >> 8); q[1] = (uint8_t)sid;
      q[2] = 1;                                         /* local flag 0, CAId 0, one component */
      const int ascty = s[3] ? 0 : 63;                  /* UEP: MPEG layer II, EEP: DAB+ */
      q[3] = (uint8_t)((0 << 6) | ascty);               /* TMId 0 (stream audio) */
      q[4] = (uint8_t)((s[0] << 2) | (1 << 1) | 0);     /* SubChId, primary, no CA */
    }
  }
  /* FIG 0/2 (P/D 1): one data service with one packet-mode component (TMId 3) per packet entry; then FIG 0/3 (clause 6.3.2)
     tells where each SCId is carried */
  for (int part = 0; part < 2; part++)
  {
    const int size = part == 0 ? 7 : 5;
    i = 0;
    while (i < c->n_packet)
    {
      int room = 30 - w->used;
      if (room < 2 + size) room = 30;
      int n = (room - 2) / size;
      if (n > c->n_packet - i) n = c->n_packet - i;
      p = ficw_reserve(w, 2 + size * n);
      if (!p || n == 0) return -1;
      p[0] = (uint8_t)((0 << 5) | (1 + size * n));
      p[1] = part == 0 ? (uint8_t)((1 << 5) | 2) : 3;   /* C/N 0, OE 0, P/D 1, extension 2 / P/D 0, extension 3 */
      uint8_t * q = p + 2;
      for (int k = 0; k < n; k++, i++, q += size)
      {
        const int32_t * e = c->packet + 5 * i;          /* subChId, SCId, address, DSCTy, DG flag */
        if (part == 0)
        {
          const uint32_t sid = 0xE1D00000u | (uint32_t)(e[1] & 0xfff);
          q[0] = (uint8_t)(sid >> 24); q[1] = (uint8_t)(sid >> 16); q[2] = (uint8_t)(sid >> 8); q[3] = (uint8_t)sid;
          q[4] = 1;                                     /* local flag 0, CAId 0, one component */
          q[5] = (uint8_t)((3 << 6) | ((e[1] >> 6) & 63)); /* TMId 3, SCId */
          q[6] = (uint8_t)(((e[1] & 63) << 2) | (1 << 1) | 0); /* primary, no CA */
        }
        else
        {
          q[0] = (uint8_t)(e[1] >> 4);
          q[1] = (uint8_t)((e[1] & 15) << 4);           /* Rfa 0, CAOrg flag 0 */
          q[2] = (uint8_t)(((e[4] & 1) << 7) | (e[3] & 63)); /* DG flag, Rfu 0, DSCTy */
          q[3] = (uint8_t)((e[0] << 2) | ((e[2] >> 8) & 3));
          q[4] = (uint8_t)(e[2] & 0xff);
        }
      }
    }
  }
  /* FIG 0/14: SubChId (6 bits), FEC scheme (2 bits) */
  i = 0;
  while (i < c->n_fec)
  {
    int room = 30 - w->used;
    if (room < 2 + 1) room = 30;
    int n = room - 2;
    if (n > c->n_fec - i) n = c->n_fec - i;
    p = ficw_reserve(w, 2 + n);
    if (!p || n == 0) return -1;
    p[0] = (uint8_t)((0 << 5) | (1 + n));
    p[1] = 14;                                          /* C/N 0, OE 0, P/D 0, extension 14 */
    for (int k = 0; k < n; k++, i++) p[2 + k] = (uint8_t)(((c->fec[i] & 63) << 2) | 1);
  }
  ficw_finish(w);
  return 0;
}

/* fib_truth: n_frames*3072 bytes (one bit per byte, FIBs incl. CRC, as the receiver delivers them).
 * msc_truth[s]: n_frames*4*24*bitRate bytes for sub-channel s (logical frames in transmit order); may be NULL. */
int dabsynth_generate(const dabsynth_cfg * c, void * out_iq, uint8_t * fib_truth, uint8_t ** msc_truth)
{
  init_tables();
  const int nf = c->n_frames, ncif = 4 * nf;
  const int64_t total = dabsynth_num_samples(c);
  if (nf < 0 || c->n_subch < 0 || c->n_subch > 64) return -1;

  /* coded + punctured logical frames of every sub-channel, then time-interleaved CIF payloads */
  uint8_t ** coded = (uint8_t **)calloc((size_t)(c->n_subch > 0 ? c->n_subch : 1), sizeof(uint8_t *));
  for (int s = 0; s < c->n_subch; s++)
  {
    const int32_t * d = c->subch + 7 * s;
    const int frag = d[2] * 64, nbits = 24 * d[5];
    int L[4], P[4];
    if (d[1] < 0 || d[1] + d[2] > 864 || profile_segments(d[3], d[5], d[4], L, P) != 0) { free(coded); return -2; }
    coded[s] = (uint8_t *)calloc((size_t)ncif * (size_t)frag, 1);
#pragma omp parallel for schedule(static)
    for (int q = 0; q < ncif; q++)
    {
      uint8_t * info = (uint8_t *)malloc((size_t)nbits);
      uint8_t * mother = (uint8_t *)malloc((size_t)(4 * (nbits + 6)));
      const uint8_t * given = c->msc_payload ? c->msc_payload[s] : NULL;
      if (given)
        for (int i = 0; i < nbits; i++) info[i] = given[(size_t)q * nbits + i] & 1u;
      else
      {
        rng_t r = rng_make(c->seed, 0x1000 + (uint64_t)s, (uint64_t)q);
        for (int i = 0; i < nbits; i += 64)
        {
          uint64_t w = rng_next(&r);
          for (int b = 0; b < 64 && i + b < nbits; b++) info[i + b] = (uint8_t)((w >> b) & 1u);
        }
      }
      if (msc_truth && msc_truth[s]) memcpy(msc_truth[s] + (size_t)q * nbits, info, (size_t)nbits);
      for (int i = 0; i < nbits; i++) info[i] ^= g_prbs[i];
      conv_encode(info, nbits, mother);
      int pos = 0, n = 0;
      uint8_t * dst = coded[s] + (size_t)q * frag;
      for (int seg = 0; seg < 4; seg++) if (L[seg] > 0) n = puncture_blocks(mother, &pos, dst, n, L[seg], P[seg]);
      n = puncture_tail(mother, &pos, dst, n);
      (void)n; /* UEP leaves frag - n padding bits at 0 */
      free(info); free(mother);
    }
  }

  const float amp = c->rms / sqrtf((float)KC);            /* per-carrier amplitude for unnormalised IFFT */
  const float noise_sigma = c->snr_db >= 100.0f ? 0.0f : c->rms * powf(10.0f, -c->snr_db / 20.0f) * 0.70710678f;
  const double dphi = 2.0 * M_PI * (double)c->cfo_hz / (double)FS;

#pragma omp parallel
  {
    int64_t cap = TF;
    if (c->lead_samples > cap) cap = c->lead_samples;
    if (c->tail_samples > cap) cap = c->tail_samples;
    cf * frame = (cf *)malloc(sizeof(cf) * (size_t)cap);
    cf * sym = (cf *)malloc(sizeof(cf) * TU);
    cf * prev = (cf *)malloc(sizeof(cf) * TU);
    uint8_t * bits = (uint8_t *)malloc((size_t)75 * SYM_BITS);
    uint8_t * mother = (uint8_t *)malloc(3096);
    uint8_t fic[768];

#pragma omp for schedule(dynamic, 1)
    for (int f = -1; f <= nf; f++)
    {
      int64_t base, count;
      if (f == -1) { base = 0; count = c->lead_samples; }
      else if (f == nf) { base = (int64_t)c->lead_samples + (int64_t)nf * TF; count = c->tail_samples; }
      else { base = (int64_t)c->lead_samples + (int64_t)f * TF; count = TF; }
      if (count <= 0) continue;

      if (f >= 0 && f < nf)
      {
        /* FIC: 4 blocks of 3 FIBs */
        rng_t r = rng_make(c->seed, 0x10, (uint64_t)f);
        fic_writer mci;
        if (c->fig_mode == 1) build_mci(c, f, &mci);
        for (int blk = 0; blk < 4; blk++)
        {
          for (int fib = 0; fib < 3; fib++)
          {
            uint8_t * p = &fic[fib * 256];
            if (c->fig_mode == 1) { for (int i = 0; i < 240; i++) p[i] = (uint8_t)((mci.b[3 * blk + fib][i >> 3] >> (7 - (i & 7))) & 1u); }
            else
            for (int i = 0; i < 240; i += 60) { uint64_t w = rng_next(&r); for (int b = 0; b < 60; b++) p[i + b] = (uint8_t)((w >> b) & 1u); }
            const uint16_t crc = crc16(p, 240);
            for (int b = 0; b < 16; b++) p[240 + b] = (uint8_t)((crc >> (15 - b)) & 1u);
          }
          if (fib_truth) memcpy(fib_truth + (size_t)f * 3072 + (size_t)blk * 768, fic, 768);
          for (int i = 0; i < 768; i++) fic[i] ^= g_prbs[i];
          conv_encode(fic, 768, mother);
          int pos = 0, n = 0;
          uint8_t * dst = bits + blk * 2304;
          n = puncture_blocks(mother, &pos, dst, n, 21, 16);
          n = puncture_blocks(mother, &pos, dst, n, 3, 15);
          n = puncture_tail(mother, &pos, dst, n);
        }
        /* MSC: 4 CIFs; unused capacity carries random bits */
        for (int cc = 0; cc < 4; cc++)
        {
          const int cif = 4 * f + cc;
          uint8_t * dst = bits + 9216 + cc * CIF_BITS;
          rng_t rp = rng_make(c->seed, 0x20, (uint64_t)cif);
          for (int i = 0; i < CIF_BITS; i += 64) { uint64_t w = rng_next(&rp); for (int b = 0; b < 64; b++) dst[i + b] = (uint8_t)((w >> b) & 1u); }
          for (int s = 0; s < c->n_subch; s++)
          {
            const int32_t * d = c->subch + 7 * s;
            const int frag = d[2] * 64;
            uint8_t * o = dst + d[1] * 64;
            for (int i = 0; i < frag; i++)
            {
              const int q = cif - TIME_MAP[i & 15];
              o[i] = q >= 0 ? coded[s][(size_t)q * frag + i] : 0;
            }
          }
        }
        /* OFDM: null, PRS, 75 differentially modulated symbols */
        memset(frame, 0, sizeof(cf) * TNULL);
        if (c->fig_mode == 1 && c->tii_main >= 0 && c->tii_main < 70 && c->tii_sub >= 0 && c->tii_sub < 24 && f >= 1 && ((((4 * (f - 1)) % 5000) & 7) >= 4))
        {
          /* TII: in each of the 4 blocks of 384 carriers, the groups of the main id's pattern carry the comb's carrier pair */
          int pat = 0, np = 0;
          for (int b = 0; b < 256 && np <= c->tii_main; b++) if (__builtin_popcount((unsigned)b) == 4) { pat = b; np++; }
          memset(sym, 0, sizeof(cf) * TU);
          for (int blk = 0; blk < 4; blk++)
            for (int grp = 0; grp < 8; grp++)
            {
              if (!(pat & (0x80 >> grp))) continue;
              const int k = -KC / 2 + 2 * (blk * 192 + grp * 24 + c->tii_sub), bin = k < 0 ? k + TU : k + 1;
              sym[bin].re = amp; sym[bin + 1].re = amp;
            }
          ifft2048(sym);
          for (int i = 0; i < TNULL; i++) frame[i] = sym[(i - TG + 4 * TU) % TU]; /* the receiver transforms samples TG .. TG + TU - 1 */
        }
        for (int i = 0; i < TU; i++)
        {
          static const float qre[4] = { 1, 0, -1, 0 }, qim[4] = { 0, 1, 0, -1 };
          const int q = g_prs_q[i];
          prev[i].re = q == 255 ? 0.0f : qre[q] * amp;
          prev[i].im = q == 255 ? 0.0f : qim[q] * amp;
        }
        for (int l = 0; l < 76; l++)
        {
          if (l > 0)
          {
            const uint8_t * b = bits + (size_t)(l - 1) * SYM_BITS;
            for (int k = 0; k < KC; k++)
            {
              const int bin = g_bin[k] < 0 ? g_bin[k] + TU : g_bin[k];
              const float dr = b[k] ? -0.70710678f : 0.70710678f, di = b[KC + k] ? -0.70710678f : 0.70710678f;
              const cf p = prev[bin];
              prev[bin].re = p.re * dr - p.im * di;
              prev[bin].im = p.re * di + p.im * dr;
            }
          }
          memcpy(sym, prev, sizeof(cf) * TU);
          ifft2048(sym);
          cf * dst = frame + TNULL + (size_t)l * TS;
          memcpy(dst, sym + TU - TG, sizeof(cf) * TG);
          memcpy(dst + TG, sym, sizeof(cf) * TU);
        }
      }
      else
      {
        /* filler: noise-like signal at data-symbol power */
        rng_t r = rng_make(c->seed, 0x30, (uint64_t)(f + 1));
        for (int64_t i = 0; i < count; i++)
        {
          float a, b;
          rng_gauss2(&r, &a, &b);
          frame[i].re = a * c->rms * 0.70710678f;
          frame[i].im = b * c->rms * 0.70710678f;
        }
      }

      /* channel + quantisation */
      rng_t rn = rng_make(c->seed, 0x40, (uint64_t)(f + 1));
      for (int64_t i = 0; i < count; i++)
      {
        cf v = frame[i];
        if (c->cfo_hz != 0.0f)
        {
          const double ph = fmod(dphi * (double)(base + i), 2.0 * M_PI);
          const float cr = (float)cos(ph), sr = (float)sin(ph);
          const cf t = { v.re * cr - v.im * sr, v.re * sr + v.im * cr };
          v = t;
        }
        if (noise_sigma > 0.0f)
        {
          float a, b;
          rng_gauss2(&rn, &a, &b);
          v.re += a * noise_sigma; v.im += b * noise_sigma;
        }
        if (c->format == 0) ((cf *)out_iq)[base + i] = v;
        else if (c->format == 1)
        {
          float a = roundf(v.re * 128.0f + 127.38f), b = roundf(v.im * 128.0f + 127.38f);
          a = a < 0 ? 0 : (a > 255 ? 255 : a); b = b < 0 ? 0 : (b > 255 ? 255 : b);
          ((uint8_t *)out_iq)[2 * (base + i)] = (uint8_t)a; ((uint8_t *)out_iq)[2 * (base + i) + 1] = (uint8_t)b;
        }
        else
        {
          float a = roundf(v.re * 32768.0f), b = roundf(v.im * 32768.0f);
          a = a < -32768 ? -32768 : (a > 32767 ? 32767 : a); b = b < -32768 ? -32768 : (b > 32767 ? 32767 : b);
          ((int16_t *)out_iq)[2 * (base + i)] = (int16_t)a; ((int16_t *)out_iq)[2 * (base + i) + 1] = (int16_t)b;
        }
      }
    }
    free(frame); free(sym); free(prev); free(bits); free(mother);
  }
  for (int s = 0; s < c->n_subch; s++) free(coded[s]);
  free(coded);
  (void)total;
  return 0;
}
