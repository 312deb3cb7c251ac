// Host build of pfec.cuh as the FEC pass uses it (k_pfec_code / k_pfec_start: pfec_slot_code, pfec_run_start; k_pfec_list:
// pfec_incomplete; k_pfec_correct: pfec_byte, pfec_row_decode), here as one sequential replay, and the packet walk of packet.cuh
// over the corrected bytes with the FEC mask (packet_frame's PKT_FEC path). Built as a shared library for tests/pfec_support.py.
//   pfck_decode(cw)                                   one RS(204,188) code word, corrected in place -> corrected bytes or -1
//   pfck_run(bytes, bit_rate, n_frames, corrected, mask, rec, cap) -> frames (as dabo_pfec_run in pfec_oracle.c)
//   pfck_groups(bits, bit_rate, n_frames, address, dg_flag, rec, cap, payload, stats) -> groups, from the corrected bytes (rec: cap
//                                                      x 23 int64, stats: 15 int64, as pchk_run in packet_check.cu)
#include "packet.cuh"
#include "pfec.cuh"

#include <cstring>
#include <vector>

using namespace dab;

static const PfecTables & tables()
{
  static PfecTables t;
  static bool ready = false;
  if (!ready) { memset(&t, 0, sizeof t); pfec_tables(t); ready = true; }
  return t;
}

extern "C" int pfck_decode(uint8_t * cw)
{
  int col[PFEC_T];
  uint8_t val[PFEC_T];
  const int m = pfec_row_decode(tables(), [&](int c) { return (unsigned)cw[c]; }, col, val);
  for (int i = 0; i < m; i++) cw[col[i]] ^= val[i];
  return m;
}

extern "C" int pfck_run(const uint8_t * bytes, int bit_rate, int n_frames, uint8_t * corrected, uint8_t * mask, int32_t * rec, int cap)
{
  const long long n = (long long)n_frames * (bit_rate / 8), spf = bit_rate / 8;
  std::vector<uint8_t> code((size_t)n);
  for (long long i = 0; i < n; i++) code[(size_t)i] = (uint8_t)pfec_slot_code(bytes + i * PFEC_SLOT);
  memcpy(corrected, bytes, (size_t)n * PFEC_SLOT);
  memset(mask, 0, (size_t)n);
  long long prev = -1;
  int out = 0;
  for (long long s = 0; s < n; s++)
  {
    if (!pfec_run_start(code.data(), n, s)) continue;
    for (long long j = s; j < s + PFEC_RUN && j < n; j++) mask[j] = 1;
    const bool cut = pfec_incomplete(s, prev, n);
    int fixed = 0, failed = 0, nb = 0;
    for (int r = 0; r < PFEC_ROWS && !cut; r++)
    {
      int col[PFEC_T];
      uint8_t val[PFEC_T];
      const int m = pfec_row_decode(tables(), [&](int c) { return (unsigned)bytes[pfec_byte(s, r, c)]; }, col, val);
      if (m < 0) { failed++; continue; }
      fixed += m > 0;
      nb += m;
      for (int i = 0; i < m; i++) corrected[pfec_byte(s, r, col[i])] ^= val[i];
    }
    if (out < cap)
    {
      int32_t * o = rec + 10 * (size_t)out;
      const long long last = (s + PFEC_RUN < n ? s + PFEC_RUN : n) - 1;
      o[0] = (int32_t)(s - PFEC_ADT_SLOTS); o[1] = (int32_t)s; o[2] = (int32_t)((s > PFEC_ADT_SLOTS ? s - PFEC_ADT_SLOTS : 0) / spf); o[3] = (int32_t)(last / spf);
      o[4] = cut ? PFEC_INCOMPLETE : failed ? PFEC_PARTIAL : fixed ? PFEC_CORRECTED : PFEC_CLEAN;
      o[5] = fixed; o[6] = failed; o[7] = nb; o[8] = pfec_score(code.data(), n, s); o[9] = 0;
    }
    out++;
    prev = s;
  }
  return out;
}

extern "C" int pfck_groups(const uint8_t * bits, int bit_rate, int n_frames, int address, int dg_flag, int64_t * rec, int cap, uint8_t * payload, int64_t * stats)
{
  const int fb = 3 * bit_rate, spf = bit_rate / 8;
  std::vector<uint8_t> raw((size_t)n_frames * fb), packed(raw.size()), mask((size_t)n_frames * spf);
  for (size_t i = 0; i < raw.size(); i++)
  {
    unsigned v = 0;
    for (int b = 0; b < 8; b++) v = (v << 1) | (bits[8 * i + b] & 1u);
    raw[i] = (uint8_t)v;
  }
  std::vector<int32_t> frec((size_t)n_frames * spf / 2 + 1);
  pfck_run(raw.data(), bit_rate, n_frames, packed.data(), mask.data(), frec.data(), (int)(frec.size() / 10));
  std::vector<PacketSlot> slots((size_t)n_frames * spf);
  for (int f = 0; f < n_frames; f++) packet_frame(packed.data() + (size_t)f * fb, fb, slots.data() + (size_t)f * spf, mask.data() + (size_t)f * spf);
  memset(stats, 0, 15 * sizeof(int64_t));
  unsigned prev = 0;
  int state = 0, n_out = 0, start = 0;
  std::vector<uint8_t> g;
  int64_t off = 0;
  for (size_t i = 0; i < slots.size(); i++)
  {
    const PacketSlot & s = slots[i];
    if (s.cls == PKT_CRC_ERROR) stats[1]++;
    else if (s.cls == PKT_BAD_LENGTH) stats[2]++;
    else if (s.cls == PKT_CUT) stats[3]++;
    if (s.cls != PKT_OK) continue;
    if (pkt_addr(s.hdr) == 0) { stats[4]++; continue; }
    if (pkt_addr(s.hdr) != address) { stats[6]++; continue; }
    if (!packet_mine(s, address)) { stats[5]++; continue; }
    stats[0]++;
    const bool cont = packet_continues(prev, s.hdr);
    if ((prev & 4u) && !cont) stats[7]++;
    int emit, abandon, drop;
    const int fl = pkt_fl(s.hdr);
    state = packet_walk_step(state, fl, cont, &emit, &abandon, &drop);
    stats[8] += abandon;
    stats[9] += drop;
    prev = 4u | (unsigned)pkt_ci(s.hdr);
    if (fl >= 2) { start = (int)i; g.clear(); }
    if (fl < 2 && !state && !emit) continue;
    const uint8_t * src = packed.data() + (i / spf) * fb + s.pos + 3;
    g.insert(g.end(), src, src + pkt_useful(s.hdr));
    if (!emit) continue;
    const DgInfo d = dg_parse(g.data(), (int)g.size(), dg_flag != 0);
    int64_t r[23] = { start / spf, (int64_t)(i / spf), 0, d.status, d.ext_flag, d.crc_flag, d.seg_flag, d.ua_flag, d.type, d.cont, d.rep, d.extension,
                      d.seg_last, d.seg_num, d.tid, d.li, d.crc_stored, d.crc_computed, (int64_t)g.size(), d.data_start, d.data_len, 0, off };
    int np = 0;
    for (size_t j = (size_t)start; j <= i; j++) np += packet_mine(slots[j], address);
    r[2] = np;
    if (n_out < cap)
    {
      memcpy(rec + (size_t)n_out * 23, r, sizeof r);
      if (payload) memcpy(payload + off, g.data(), g.size());
    }
    stats[10 + d.status]++;
    off += (int64_t)g.size();
    n_out++;
  }
  return n_out;
}
