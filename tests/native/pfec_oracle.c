/* Plain-C restatement of packet-mode FEC (ETSI EN 300 401 clause 5.3.5), written apart from dabstar_b200/csrc/pfec.cuh and sharing
 * no code with it: the FEC-packet runs located by the same per-slot rule, each row decoded by the Euclidean (Sugiyama) algorithm
 * instead of Berlekamp-Massey, and the corrections applied to a copy. Built as a shared library for tests/pfec_support.py.
 *   dabo_pfec_decode(cw)        one RS(204,188) code word, corrected in place -> corrected bytes or -1
 *   dabo_pfec_run(bytes, bit_rate, n_frames, corrected, mask, rec, cap) -> frames; bytes / corrected: n_frames * 3 * bit_rate
 *                               packed bytes; mask: one byte per 24-byte slot; rec: cap x 10 int32 (dabstar_fec_frame) */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static int gexp[512], glog[256], ready;

static void init(void)
{
  if (ready) return;
  int x = 1;
  for (int i = 0; i < 255; i++)
  {
    gexp[i] = gexp[i + 255] = x;
    glog[x] = i;
    x <<= 1;
    if (x & 256) x ^= 0x11d;
  }
  ready = 1;
}
static int mul(int a, int b) { return a && b ? gexp[glog[a] + glog[b]] : 0; }
static int inv(int a) { return gexp[255 - glog[a]]; }
static int pw(int e) { e %= 255; if (e < 0) e += 255; return gexp[e]; } /* alpha^e */
static int deg(const int * p, int n) { int d = -1; for (int i = 0; i < n; i++) if (p[i]) d = i; return d; }
static int eval(const int * p, int n, int x) { int v = 0; for (int i = n - 1; i >= 0; i--) v = mul(v, x) ^ p[i]; return v; }

#define NP 40 /* polynomial room: coefficient i of x^i */

int dabo_pfec_decode(uint8_t * cw)
{
  init();
  int S[16], any = 0;
  for (int j = 0; j < 16; j++)
  {
    int v = 0; /* cw[0] is the coefficient of x^203 */
    for (int i = 0; i < 204; i++) v = mul(v, pw(j)) ^ cw[i];
    S[j] = v;
    any |= v;
  }
  if (!any) return 0;
  /* Sugiyama: a = x^16, b = S(x); t_prev = 0, t = 1; divide until deg(b) < 8 */
  int a[NP] = { 0 }, b[NP] = { 0 }, tp[NP] = { 0 }, t[NP] = { 0 };
  a[16] = 1;
  for (int j = 0; j < 16; j++) b[j] = S[j];
  t[0] = 1;
  while (deg(b, NP) >= 8)
  {
    int q[NP] = { 0 }, r[NP];
    memcpy(r, a, sizeof r);
    const int db = deg(b, NP), lb = inv(b[db]);
    for (int d = deg(r, NP); d >= db; d = deg(r, NP))
    {
      const int c = mul(r[d], lb);
      q[d - db] ^= c;
      for (int i = 0; i <= db; i++) r[d - db + i] ^= mul(c, b[i]);
    }
    int tn[NP] = { 0 };
    for (int i = 0; i < NP; i++)
      for (int k = 0; k < NP && i + k < NP; k++) tn[i + k] ^= mul(q[i], t[k]);
    for (int i = 0; i < NP; i++) tn[i] ^= tp[i];
    memcpy(a, b, sizeof a);
    memcpy(b, r, sizeof b);
    memcpy(tp, t, sizeof tp);
    memcpy(t, tn, sizeof t);
  }
  if (!t[0]) return -1;
  const int n0 = inv(t[0]);
  int lam[NP], om[NP];
  for (int i = 0; i < NP; i++) { lam[i] = mul(t[i], n0); om[i] = mul(b[i], n0); }
  const int L = deg(lam, NP);
  if (L < 1 || L > 8) return -1;
  int dl[NP] = { 0 }; /* formal derivative */
  for (int i = 1; i < NP; i++) if (i & 1) dl[i - 1] = lam[i];
  int pos[8], val[8], n = 0;
  for (int i = 0; i < 204; i++)
  {
    const int e = 203 - i, xi = pw(-e); /* locator alpha^e of byte i; xi its inverse */
    if (eval(lam, NP, xi)) continue;
    const int den = eval(dl, NP, xi);
    if (n == 8 || !den) return -1;
    const int v = mul(mul(pw(e), eval(om, NP, xi)), inv(den));
    if (!v) return -1;
    pos[n] = i;
    val[n] = v;
    n++;
  }
  if (n != L) return -1;
  for (int k = 0; k < n; k++) cw[pos[k]] ^= (uint8_t)val[k];
  return n;
}

/* first two header bytes of an FEC packet: length 00, address 1022; the first / last flags expected at position k of a run */
static int fits(const uint8_t * p, int k)
{
  const int fl = k == 0 ? 2 : (k == 8 ? 1 : 0);
  return (p[0] >> 6) == 0 && ((p[0] & 3) << 8 | p[1]) == 1022 && ((p[0] >> 2) & 3) == fl;
}
static int score(const uint8_t * b, long n, long s)
{
  int c = 0;
  for (int k = 0; k < 9; k++)
    if (s + k >= 0 && s + k < n && fits(b + (s + k) * 24, k)) c++;
  return c;
}

int dabo_pfec_run(const uint8_t * bytes, int bit_rate, int n_frames, uint8_t * corrected, uint8_t * mask, int32_t * rec, int cap)
{
  init();
  const long n = (long)n_frames * (bit_rate / 8), spf = bit_rate / 8;
  memcpy(corrected, bytes, (size_t)n * 24);
  memset(mask, 0, (size_t)n);
  long prev = -1;
  int out = 0;
  for (long s = 0; s < n; s++)
  {
    const int c = score(bytes, n, s);
    if (c < 6 || c <= score(bytes, n, s - 1) || c < score(bytes, n, s + 1)) continue;
    for (long j = s; j < s + 9 && j < n; j++) mask[j] = 1;
    const int cut = s < 94 || s + 9 > n || (prev >= 0 && s - prev < 103);
    int fixed = 0, failed = 0, nb = 0;
    if (!cut)
    {
      const long adt = (s - 94) * 24;
      for (int r = 0; r < 12; r++)
      {
        uint8_t cw[204];
        long at[204];
        for (int col = 0; col < 188; col++) at[col] = adt + 12L * col + r;
        for (int p = 0; p < 16; p++)
        {
          const int j = 12 * p + r; /* RS byte j of the frame */
          at[188 + p] = (s + j / 22) * 24 + 2 + j % 22;
        }
        for (int col = 0; col < 204; col++) cw[col] = bytes[at[col]];
        const int m = dabo_pfec_decode(cw);
        if (m < 0) { failed++; continue; }
        if (m > 0) fixed++;
        nb += m;
        for (int col = 0; col < 204; col++) corrected[at[col]] = cw[col];
      }
    }
    if (out < cap)
    {
      int32_t * o = rec + 10L * out;
      const long last = (s + 9 < n ? s + 9 : n) - 1;
      o[0] = (int32_t)(s - 94); o[1] = (int32_t)s; o[2] = (int32_t)((s - 94 > 0 ? s - 94 : 0) / spf); o[3] = (int32_t)(last / spf);
      o[4] = cut ? 3 : failed ? 2 : fixed ? 1 : 0;
      o[5] = fixed; o[6] = failed; o[7] = nb; o[8] = c; o[9] = 0;
    }
    out++;
    prev = s;
  }
  return out;
}
