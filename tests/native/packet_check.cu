// Host build of packet.cuh as the packet pass uses it: every logical frame's packets (k_packet_scan: packet_frame), the walk over
// one address's packets in stream order (k_packet_walk: packet_mine, packet_continues, packet_walk_step, here as one sequential
// replay) and the data groups' headers (k_packet_compact: dg_parse). Built as a shared library for tests/packet_support.py.
//   pchk_crc(bytes, n)                              -> pkt_crc
//   pchk_run(bits, bit_rate, n_frames, address, dg_flag, rec, cap, payload, stats) -> groups; rec: cap x 23 int64 (the fields of
//                                                      dabstar_data_group in order), stats: 15 int64 (dabstar_packet_stats)
#include "packet.cuh"

#include <cstring>
#include <vector>

using namespace dab;

extern "C" unsigned pchk_crc(const uint8_t * p, int n) { return pkt_crc(p, n); }

extern "C" int pchk_run(const uint8_t * bits, int bit_rate, int n_frames, int address, int dg_flag, int64_t * rec, int cap, uint8_t * payload, int64_t * stats)
{
  const int fb = 3 * bit_rate, spf = bit_rate / 8;
  std::vector<uint8_t> packed((size_t)n_frames * fb);
  for (size_t i = 0; i < packed.size(); i++)
  {
    unsigned v = 0;
    for (int b = 0; b < 8; b++) v = (v << 1) | (bits[8 * i + b] & 1u);
    packed[i] = (uint8_t)v;
  }
  std::vector<PacketSlot> slots((size_t)n_frames * spf);
  for (int f = 0; f < n_frames; f++) packet_frame(packed.data() + (size_t)f * fb, fb, slots.data() + (size_t)f * spf);
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
