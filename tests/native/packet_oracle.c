/* packet_oracle.c — a plain-C restatement of the packet-mode pass (ETSI EN 300 401 clauses 5.3.2 and 5.3.3), written from the
 * standard and sharing no code with dabstar_b200/csrc/packet.cuh: the packets of every logical frame, the data groups of one
 * address assembled in stream order, and their MSC data group headers and CRCs.
 *
 * dabo_pkt_run(bits, bit_rate, n_frames, address, dg_flag, rec, cap, payload, stats): bits one per byte, n_frames x 24 * bit_rate.
 * rec: cap x 23 int64 per group (the fields of dabstar_data_group in order, offset last); payload: the groups' bytes; stats: 15
 * int64 (the fields of dabstar_packet_stats). Returns the number of groups. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

unsigned dabo_pkt_crc(const uint8_t * d, int n)
{
  unsigned r = 0xFFFF;
  for (int i = 0; i < n; i++)
    for (int b = 7; b >= 0; b--)
    {
      const unsigned in = (d[i] >> b) & 1, top = (r >> 15) & 1;
      r = (r << 1) & 0xFFFF;
      if (in != top) r ^= 0x1021;
    }
  return r ^ 0xFFFF;
}

enum { G_OK, G_NOCRC, G_CRC, G_BAD, G_RAW };
enum { F_FIRST = 0, F_LAST, F_NP, F_STATUS, F_EXTF, F_CRCF, F_SEGF, F_UAF, F_TYPE, F_CONT, F_REP, F_EXT, F_SEGL, F_SEGN, F_TID, F_LI, F_CRCS, F_CRCC,
       F_LEN, F_DS, F_DL, F_RES, F_OFF, N_F };

static void parse_group(const uint8_t * g, int len, int raw, int64_t * r)
{
  for (int i = F_STATUS; i < F_LEN; i++) r[i] = -1;
  r[F_LEN] = len;
  r[F_RES] = 0;
  if (raw) { r[F_STATUS] = G_RAW; r[F_DS] = 0; r[F_DL] = len; return; }
  r[F_STATUS] = G_BAD; r[F_DS] = 0; r[F_DL] = 0;
  if (len < 2) return;
  const int extf = g[0] >> 7 & 1, crcf = g[0] >> 6 & 1, segf = g[0] >> 5 & 1, uaf = g[0] >> 4 & 1;
  r[F_EXTF] = extf; r[F_CRCF] = crcf; r[F_SEGF] = segf; r[F_UAF] = uaf; r[F_TYPE] = g[0] & 15; r[F_CONT] = g[1] >> 4; r[F_REP] = g[1] & 15;
  const int end = len - (crcf ? 2 : 0); /* first byte of the CRC */
  int at = 2;
  if (extf) { if (at + 2 > end) return; r[F_EXT] = g[at] * 256 + g[at + 1]; at += 2; }
  if (segf) { if (at + 2 > end) return; r[F_SEGL] = g[at] >> 7; r[F_SEGN] = (g[at] & 0x7F) * 256 + g[at + 1]; at += 2; }
  if (uaf)
  {
    if (at + 1 > end) return;
    const int tidf = g[at] >> 4 & 1, li = g[at] & 15;
    r[F_LI] = li;
    if (at + 1 + li > end) return;
    if (tidf) { if (li < 2) return; r[F_TID] = g[at + 1] * 256 + g[at + 2]; }
    at += 1 + li;
  }
  if (at > end) return;
  r[F_DS] = at;
  r[F_DL] = end - at;
  if (!crcf) { r[F_STATUS] = G_NOCRC; return; }
  r[F_CRCS] = g[len - 2] * 256 + g[len - 1];
  r[F_CRCC] = dabo_pkt_crc(g, len - 2);
  r[F_STATUS] = r[F_CRCS] == r[F_CRCC] ? G_OK : G_CRC;
}

int dabo_pkt_run(const uint8_t * bits, int bit_rate, int n_frames, int address, int dg_flag, int64_t * rec, int cap, uint8_t * payload, int64_t * stats)
{
  const int fb = 3 * bit_rate;
  uint8_t * frame = (uint8_t *)malloc((size_t)fb);
  uint8_t * grp = (uint8_t *)malloc((size_t)fb * (size_t)(n_frames > 0 ? n_frames : 1));
  memset(stats, 0, 15 * sizeof(int64_t));
  int open = 0, have_prev = 0, prev_ci = 0, n_out = 0, g_first = 0, g_np = 0, g_len = 0;
  int64_t pay = 0;
  for (int f = 0; f < n_frames; f++)
  {
    for (int i = 0; i < fb; i++)
    {
      unsigned v = 0;
      for (int b = 0; b < 8; b++) v = v << 1 | (bits[(size_t)f * 24 * bit_rate + 8 * i + b] & 1);
      frame[i] = (uint8_t)v;
    }
    int pos = 0;
    while (pos < fb)
    {
      const uint8_t * p = frame + pos;
      const int plen = 24 * (1 + (p[0] >> 6)), room = fb - pos;
      if (plen > room) { stats[3]++; break; }
      pos += plen;
      const unsigned stored = p[plen - 2] * 256u + p[plen - 1];
      if (dabo_pkt_crc(p, plen - 2) != stored) { stats[1]++; continue; }
      const int ci = p[0] >> 4 & 3, first = p[0] >> 3 & 1, last = p[0] >> 2 & 1, addr = (p[0] & 3) * 256 + p[1], cmd = p[2] >> 7, ul = p[2] & 0x7F;
      if (ul > plen - 5) { stats[2]++; continue; }
      if (addr == 0) { stats[4]++; continue; }
      if (addr != address) { stats[6]++; continue; }
      if (cmd) { stats[5]++; continue; }
      stats[0]++;
      const int cont = have_prev && ci == ((prev_ci + 1) & 3);
      if (have_prev && !cont) stats[7]++;
      have_prev = 1;
      prev_ci = ci;
      if (first) /* first, or single */
      {
        if (open) stats[8]++;
        open = 1; g_first = f; g_np = 0; g_len = 0;
      }
      else if (!open || !cont)
      {
        if (open) stats[8]++; else stats[9]++;
        open = 0;
        continue;
      }
      memcpy(grp + g_len, p + 3, (size_t)ul);
      g_len += ul;
      g_np++;
      if (last)
      {
        int64_t r[N_F];
        r[F_FIRST] = g_first; r[F_LAST] = f; r[F_NP] = g_np;
        parse_group(grp, g_len, dg_flag, r);
        r[F_OFF] = pay;
        if (n_out < cap)
        {
          memcpy(rec + (size_t)n_out * N_F, r, sizeof r);
          if (payload) memcpy(payload + pay, grp, (size_t)g_len);
        }
        stats[10 + r[F_STATUS]]++;
        pay += g_len;
        n_out++;
        open = 0;
      }
    }
  }
  free(frame);
  free(grp);
  return n_out;
}
