// packet.cuh — packet-mode data of a DAB sub-channel: the parse of one packet, the walk over one frame's packets, the group
// assembly step over one address's packets and the parse of an MSC data group, as functions the device pass
// (packet_kernels.cu) and the host tests share.
//
// Source: ETSI EN 300 401 clause 5.3.2 (packet structure: 24 / 48 / 72 / 96-byte packets, 24-bit header, CRC-16) and clause
// 5.3.3 (MSC data group: header, session header, data field, CRC-16). Both CRCs are the FIB CRC of clause 5.2.1:
// x^16 + x^12 + x^5 + 1, preset 0xFFFF, complemented, transmitted most significant bit first. On a sub-channel with packet-mode
// FEC (FIG 0/14, the RS(204,188) outer code of clause 5.3.5, pfec.cuh) the frames are walked after correction, and a packet that
// starts on a slot of an FEC-packet run is skipped (PKT_FEC).
#pragma once
#include <cstdint>

namespace dab
{
// class of one packet slot
enum : int
{
  PKT_OK = 0,         // CRC good, useful data length <= packet length - 5
  PKT_CRC_ERROR = 1,  // CRC mismatch (the header cannot be trusted)
  PKT_BAD_LENGTH = 2, // CRC good, useful data length > packet length - 5
  PKT_CUT = 3,        // the packet would run past the end of the logical frame; the frame's walk ends there
  PKT_EMPTY = 4,      // no packet starts in this slot (the frame's packets ended before it)
  PKT_FEC = 5,        // an FEC packet (24 bytes) of packet-mode FEC: skipped, counted in the FEC frame records only
};
// status of a data group
enum : int
{
  DG_OK = 0,        // MSC data group, CRC flag 1, CRC good
  DG_NO_CRC = 1,    // MSC data group without CRC (CRC flag 0)
  DG_CRC_ERROR = 2, // MSC data group, CRC mismatch
  DG_MALFORMED = 3, // the data group's headers (and CRC) do not fit into the group
  DG_RAW = 4,       // DG flag 1: the useful data are not an MSC data group and are not parsed
};

// one packet slot of a frame: its 24-bit header, its byte offset inside the logical frame, its class
struct PacketSlot
{
  uint32_t hdr;
  uint16_t pos;
  uint8_t cls, pad;
};
__host__ __device__ inline int pkt_len(uint32_t h) { return 24 * (1 + (int)((h >> 22) & 3u)); }
__host__ __device__ inline int pkt_ci(uint32_t h) { return (int)((h >> 20) & 3u); }
__host__ __device__ inline int pkt_fl(uint32_t h) { return (int)((h >> 18) & 3u); } // first flag, last flag
__host__ __device__ inline int pkt_addr(uint32_t h) { return (int)((h >> 8) & 1023u); }
__host__ __device__ inline int pkt_cmd(uint32_t h) { return (int)((h >> 7) & 1u); }
__host__ __device__ inline int pkt_useful(uint32_t h) { return (int)(h & 127u); }

// CRC-16 x^16 + x^12 + x^5 + 1 over n bytes, most significant bit first, from crc (preset 0xFFFF); the caller complements
__host__ __device__ inline unsigned pkt_crc_update(unsigned crc, const uint8_t * p, int n)
{
  for (int i = 0; i < n; i++)
  {
    crc ^= (unsigned)p[i] << 8;
    for (int b = 0; b < 8; b++) crc = (crc & 0x8000u) ? ((crc << 1) ^ 0x1021u) & 0xffffu : (crc << 1) & 0xffffu;
  }
  return crc;
}
__host__ __device__ inline unsigned pkt_crc(const uint8_t * p, int n) { return ~pkt_crc_update(0xffffu, p, n) & 0xffffu; }

// The packet that starts at p, avail bytes before the end of its logical frame (>= 1)
__host__ __device__ inline int packet_classify(const uint8_t * p, int avail, uint32_t * hdr)
{
  *hdr = 0;
  if (avail < 3) return PKT_CUT;
  const uint32_t h = ((uint32_t)p[0] << 16) | ((uint32_t)p[1] << 8) | p[2];
  *hdr = h;
  const int len = pkt_len(h);
  if (len > avail) return PKT_CUT;
  if (pkt_crc(p, len - 2) != (((unsigned)p[len - 2] << 8) | p[len - 1])) return PKT_CRC_ERROR;
  return pkt_useful(h) > len - 5 ? PKT_BAD_LENGTH : PKT_OK;
}

// The packets of one logical frame of fb bytes: slot k gets the k-th packet (fb / 24 slots; the rest PKT_EMPTY). Returns the
// number of packets found (a PKT_CUT one included). fec (packet-mode FEC only): one byte per 24-byte slot of the frame, non-zero
// where an FEC packet lies.
__host__ __device__ inline int packet_frame(const uint8_t * f, int fb, PacketSlot * slots, const uint8_t * fec = nullptr)
{
  const int n_slots = fb / 24;
  int pos = 0, k = 0;
  while (pos < fb && k < n_slots)
  {
    uint32_t h;
    if (fec && fec[pos / 24])
    {
      slots[k++] = PacketSlot{ ((uint32_t)f[pos] << 16) | ((uint32_t)f[pos + 1] << 8) | f[pos + 2], (uint16_t)pos, (uint8_t)PKT_FEC, 0 };
      pos += 24;
      continue;
    }
    const int c = packet_classify(f + pos, fb - pos, &h);
    slots[k++] = PacketSlot{ h, (uint16_t)pos, (uint8_t)c, 0 };
    if (c == PKT_CUT) break;
    pos += pkt_len(h);
  }
  const int found = k;
  for (; k < n_slots; k++) slots[k] = PacketSlot{ 0u, 0, (uint8_t)PKT_EMPTY, 0 };
  return found;
}

// A packet of the data-group assembly of address a: CRC good, well formed, a data (not a command) packet with that address
__host__ __device__ inline bool packet_mine(const PacketSlot & s, int a) { return s.cls == PKT_OK && pkt_addr(s.hdr) == a && !pkt_cmd(s.hdr); }
// CI of the previous packet as a walk carries it: 0 none, 4 | CI
__host__ __device__ inline bool packet_continues(unsigned prev, uint32_t h) { return (prev & 4u) && (int)(((prev & 3u) + 1u) & 3u) == pkt_ci(h); }

// Group assembly step: state 0 idle, 1 open; fl: the packet's first / last flags; cont: it continues the previous packet.
// Returns the next state; *emit: the packet closes a group (single or last); *abandon: an open group is given up; *drop: an
// orphan packet (intermediate or last without an open group) is dropped.
__host__ __device__ inline int packet_walk_step(int state, int fl, bool cont, int * emit, int * abandon, int * drop)
{
  *emit = 0; *abandon = 0; *drop = 0;
  if (fl == 2) { *abandon = state; return 1; }                 // first
  if (fl == 3) { *abandon = state; *emit = 1; return 0; }      // single
  if (state == 1 && cont) { if (fl == 1) *emit = 1; return fl == 1 ? 0 : 1; } // intermediate / last that continue the group
  *abandon = state;
  *drop = !state;
  return 0;
}

// The MSC data group (clause 5.3.3) of len bytes at g. Fields that are absent are -1.
struct DgInfo
{
  int status;
  int ext_flag, crc_flag, seg_flag, ua_flag, type, cont, rep;
  int extension, seg_last, seg_num, tid, li;
  int crc_stored, crc_computed;
  int data_start, data_len;
};
__host__ __device__ inline DgInfo dg_parse(const uint8_t * g, int len, bool raw)
{
  DgInfo d{ DG_RAW, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, 0, len };
  if (raw) return d;
  d.status = DG_MALFORMED;
  d.data_start = 0;
  d.data_len = 0;
  if (len < 2) return d;
  d.ext_flag = g[0] >> 7; d.crc_flag = (g[0] >> 6) & 1; d.seg_flag = (g[0] >> 5) & 1; d.ua_flag = (g[0] >> 4) & 1; d.type = g[0] & 15;
  d.cont = g[1] >> 4; d.rep = g[1] & 15;
  int o = 2;
  const int tail = d.crc_flag ? 2 : 0;
  if (d.ext_flag)
  {
    if (o + 2 + tail > len) return d;
    d.extension = (g[o] << 8) | g[o + 1];
    o += 2;
  }
  if (d.seg_flag)
  {
    if (o + 2 + tail > len) return d;
    d.seg_last = g[o] >> 7;
    d.seg_num = ((g[o] & 127) << 8) | g[o + 1];
    o += 2;
  }
  if (d.ua_flag)
  {
    if (o + 1 + tail > len) return d;
    const int tid_flag = (g[o] >> 4) & 1;
    d.li = g[o] & 15;
    if (o + 1 + d.li + tail > len || (tid_flag && d.li < 2)) return d;
    if (tid_flag) d.tid = (g[o + 1] << 8) | g[o + 2];
    o += 1 + d.li;
  }
  if (o + tail > len) return d;
  d.data_start = o;
  d.data_len = len - tail - o;
  if (!d.crc_flag) { d.status = DG_NO_CRC; return d; }
  d.crc_stored = (g[len - 2] << 8) | g[len - 1];
  d.crc_computed = (int)pkt_crc(g, len - 2);
  d.status = d.crc_stored == d.crc_computed ? DG_OK : DG_CRC_ERROR;
  return d;
}
} // namespace dab
