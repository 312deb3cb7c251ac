// mp2.cuh — MPEG-1 / MPEG-2 LSF audio layer II frames of a DAB (MP2) sub-channel: the classification of one audio-frame slot and
// the walk step over a stream's slots, as functions the device pass (mp2_kernels.cu) and the host tests share.
//
// Sources: ISO/IEC 11172-3 2.4.1.3 (header), 2.4.3.1 (CRC-16), Annex B Table B.2 (layer II allocation); ISO/IEC 13818-3
// Table B.1 (layer II allocation at the LSF sampling rates); ETSI EN 300 401 clause 7 (an audio frame fills one 24 ms logical
// frame at 48 kHz, two at 24 kHz, and always carries the CRC).
#pragma once
#include <cstdint>

namespace dab
{
enum : int
{
  MP2_OK = 0,        // valid header and matching CRC
  MP2_NO_HEADER = 1, // syncword != 0xFFF, layer != II, or protection_bit = 1 (no CRC)
  MP2_MISMATCH = 2,  // sampling_frequency != 01, bitrate_index 0 / 15, or the header's bit rate != the sub-channel's
  MP2_CRC_ERROR = 3, // valid header, CRC mismatch
  MP2_CUT = 4,       // a 24 kHz frame whose second logical frame lies past the end of the stream
};
constexpr int MP2_LSF = 8; // class byte: the slot holds a valid 24 kHz (ID 0) header

// one audio-frame slot of a stream (layout of dabstar_mp2_frame)
struct Mp2Rec
{
  int32_t first_frame, n_frames, status;
  uint32_t header;                 // the slot's first 32 bits, as read
  int32_t crc_stored, crc_computed; // -1 where not reached
};

// layer II bit rate (kbit/s) of bitrate_index 1..14: MPEG-1 (id 1) or LSF (id 0); 0 for indices 0 and 15
__host__ __device__ inline int mp2_bit_rate(int id, int index)
{
  if (index <= 0 || index >= 15) return 0;
  if (!id) return index <= 8 ? 8 * index : 64 + 16 * (index - 8);
  if (index <= 4) return index == 1 ? 32 : 32 + 8 * index;           // 32 48 56 64
  if (index <= 8) return 80 + 16 * (index - 5);                       // 80 96 112 128
  return index <= 12 ? 160 + 32 * (index - 9) : 320 + 64 * (index - 13); // 160 192 224 256, 320 384
}
// a rate some layer II frame can have: a sub-channel the MP2 pass can take
__host__ __device__ inline bool mp2_rate_ok(int bit_rate)
{
  for (int i = 1; i < 15; i++)
    if (mp2_bit_rate(0, i) == bit_rate || mp2_bit_rate(1, i) == bit_rate) return true;
  return false;
}

// allocation bits per sub-band: table 0 = 11172-3 B.2a (48 kHz, >= 56 kbit/s per channel), 1 = B.2c (48 kHz, <= 48 kbit/s per
// channel), 2 = 13818-3 B.1 (24 kHz)
__host__ __device__ inline int mp2_sblimit(int table) { return table == 0 ? 27 : table == 1 ? 8 : 30; }
__host__ __device__ inline int mp2_nbal(int table, int sb)
{
  if (table == 0) return sb < 11 ? 4 : sb < 23 ? 3 : 2;
  if (table == 1) return sb < 2 ? 4 : 3;
  return sb < 4 ? 4 : sb < 11 ? 3 : 2;
}

// `n` bits (n <= 16) at bit `pos` of p, most significant first
__host__ __device__ inline unsigned mp2_bits(const uint8_t * p, long long pos, int n)
{
  const uint8_t * b = p + (pos >> 3);
  const int sh = (int)(pos & 7);
  unsigned v = ((unsigned)b[0] << 16) | (sh + n > 8 ? (unsigned)b[1] << 8 : 0u) | (sh + n > 16 ? (unsigned)b[2] : 0u);
  return (v >> (24 - sh - n)) & ((1u << n) - 1u);
}
// CRC-16 x^16 + x^15 + x^2 + 1 over the n low bits of v, most significant first (11172-3 2.4.3.1; preset 0xFFFF, no inversion)
__host__ __device__ inline unsigned mp2_crc_bits(unsigned crc, unsigned v, int n)
{
  for (int i = n - 1; i >= 0; i--)
  {
    const unsigned fb = ((v >> i) ^ (crc >> 15)) & 1u;
    crc = (crc << 1) & 0xffffu;
    if (fb) crc ^= 0x8005u;
  }
  return crc;
}

struct Mp2Slot
{
  int status, lsf;
  uint32_t header;
  int crc_stored, crc_computed;
};

// The slot starting at p of a sub-channel of bit_rate kbit/s; avail: bytes from p to the end of the stream (>= 6). Reads stay
// inside the frame (3 x bit_rate bytes, 6 x at 24 kHz) and the stream; a 24 kHz frame whose allocation or SCFSI would leave the
// stream is MP2_CUT here already.
__host__ __device__ inline Mp2Slot mp2_classify(const uint8_t * p, long long avail, int bit_rate)
{
  Mp2Slot s{ MP2_NO_HEADER, 0, (mp2_bits(p, 0, 16) << 16) | mp2_bits(p, 16, 16), -1, -1 };
  const unsigned h = s.header;
  if ((h >> 20) != 0xfffu || ((h >> 17) & 3u) != 2u || ((h >> 16) & 1u) != 0u) return s;
  const int id = (h >> 19) & 1, bri = (h >> 12) & 15, sfreq = (h >> 10) & 3, mode = (h >> 6) & 3, ext = (h >> 4) & 3;
  s.status = MP2_MISMATCH;
  if (sfreq != 1 || mp2_bit_rate(id, bri) != bit_rate) return s;
  s.lsf = !id;
  s.crc_stored = (int)mp2_bits(p, 32, 16);
  const long long frame = (id ? 3LL : 6LL) * bit_rate, limit = 8 * (avail < frame ? avail : frame); // bits that may be read
  const int nch = mode == 3 ? 1 : 2;
  const int table = !id ? 2 : (bit_rate / nch >= 56 ? 0 : 1);
  const int sblimit = mp2_sblimit(table);
  const int bound = mode == 1 ? (4 * (ext + 1) < sblimit ? 4 * (ext + 1) : sblimit) : sblimit;
  unsigned crc = mp2_crc_bits(0xffffu, h & 0xffffu, 16);
  long long pos = 48; // allocation: per channel below the bound, shared from there to sblimit
  for (int sb = 0; sb < sblimit; sb++)
  {
    const int nb = mp2_nbal(table, sb);
    for (int c = 0; c < (sb < bound ? nch : 1); c++)
    {
      if (pos + nb > limit) { s.status = MP2_CUT; return s; }
      crc = mp2_crc_bits(crc, mp2_bits(p, pos, nb), nb);
      pos += nb;
    }
  }
  long long apos = 48; // SCFSI: 2 bits per channel of every sub-band with a non-zero allocation (the allocation read again)
  for (int sb = 0; sb < sblimit; sb++)
  {
    const int nb = mp2_nbal(table, sb);
    for (int c = 0; c < nch; c++)
    {
      const unsigned a = mp2_bits(p, apos, nb);
      if (sb < bound || c == nch - 1) apos += nb;
      if (!a) continue;
      if (pos + 2 > limit) { s.status = MP2_CUT; return s; }
      crc = mp2_crc_bits(crc, mp2_bits(p, pos, 2), 2);
      pos += 2;
    }
  }
  s.crc_computed = (int)crc;
  s.status = s.crc_computed == s.crc_stored ? MP2_OK : MP2_CRC_ERROR;
  return s;
}
__host__ __device__ inline uint8_t mp2_class_byte(const Mp2Slot & s) { return (uint8_t)(s.status | (s.lsf ? MP2_LSF : 0)); }

// Walk step: the record of the slot that starts at logical frame i of n, from the slot's class byte. Returns the logical frames
// it covers (the next slot starts there) and its status: an OK 24 kHz frame takes frames i and i + 1, or is CUT at the end.
__host__ __device__ inline int mp2_walk_step(uint8_t cls, int i, int n, int * status)
{
  const int st = cls & 7;
  if (st == MP2_OK && (cls & MP2_LSF))
  {
    *status = i + 1 < n ? MP2_OK : MP2_CUT;
    return i + 1 < n ? 2 : 1;
  }
  *status = st;
  return 1;
}
} // namespace dab
