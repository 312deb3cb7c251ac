/* mp2_oracle.c — plain-C restatement of the MPEG layer II audio-frame check of a DAB (MP2) sub-channel, written from the
 * standards and sharing no code with dabstar_b200/csrc/mp2.cuh: it works on one-bit-per-byte frames and walks each stream in
 * order, classifying only the slots the walk reaches.
 *   ISO/IEC 11172-3 2.4.1.3 header, 2.4.1.6 / 2.4.2.3 audio_data (allocation, SCFSI), 2.4.3.1 CRC-16, Annex B Table B.2a / B.2c;
 *   ISO/IEC 13818-3 Table B.1 (LSF, 24 kHz); ETSI EN 300 401 clause 7 (one audio frame per logical frame at 48 kHz, per two at
 *   24 kHz, always with CRC).
 * Build: gcc -O2 -shared -fPIC -o libmp2_oracle.so mp2_oracle.c */
#include <stdint.h>
#include <string.h>

typedef struct
{
  int32_t first_frame, n_frames, status;
  uint32_t header;
  int32_t crc_stored, crc_computed;
} dabo_mp2_rec;

static const int RATE_MPEG1[16] = { 0, 32, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320, 384, 0 };
static const int RATE_LSF[16] = { 0, 8, 16, 24, 32, 40, 48, 56, 64, 80, 96, 112, 128, 144, 160, 0 };
/* nbal per sub-band */
static const int NBAL_B2A[27] = { 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 3, 3, 3, 3, 3, 3, 3, 3, 3, 3, 3, 3, 2, 2, 2, 2 };
static const int NBAL_B2C[8] = { 4, 4, 3, 3, 3, 3, 3, 3 };
static const int NBAL_LSF[30] = { 4, 4, 4, 4, 3, 3, 3, 3, 3, 3, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2 };

/* CRC-16, generator 0x8005, preset 0xFFFF, over n bits (one per byte) */
static unsigned crc_over_bits(unsigned crc, const uint8_t * bits, long n)
{
  for (long i = 0; i < n; i++)
  {
    const unsigned top = (crc >> 15) & 1u;
    crc = (crc << 1) & 0xffffu;
    if (top ^ (bits[i] & 1u)) crc ^= 0x8005u;
  }
  return crc;
}

static unsigned field(const uint8_t * bits, long pos, int n)
{
  unsigned v = 0;
  for (int i = 0; i < n; i++) v = (v << 1) | (bits[pos + i] & 1u);
  return v;
}

unsigned dabo_mp2_crc16(const uint8_t * bytes, int n_bytes)
{
  unsigned crc = 0xffffu;
  for (int i = 0; i < n_bytes; i++)
  {
    uint8_t b[8];
    for (int k = 0; k < 8; k++) b[k] = (uint8_t)((bytes[i] >> (7 - k)) & 1);
    crc = crc_over_bits(crc, b, 8);
  }
  return crc;
}

/* the allocation table of a header: sets *nbal and *sblimit */
static void alloc_table(int id, int bit_rate, int nch, const int ** nbal, int * sblimit)
{
  if (!id) { *nbal = NBAL_LSF; *sblimit = 30; }
  else if (bit_rate / nch >= 56) { *nbal = NBAL_B2A; *sblimit = 27; }
  else { *nbal = NBAL_B2C; *sblimit = 8; }
}

/* allocation bits of one frame: (sample rate 48 / 24 kHz, total bit rate, mode, mode_extension) */
int dabo_mp2_alloc_bits(int khz, int bit_rate, int mode, int mode_ext)
{
  const int nch = mode == 3 ? 1 : 2;
  const int * nbal;
  int sblimit, bound, n = 0;
  alloc_table(khz == 48, bit_rate, nch, &nbal, &sblimit);
  bound = mode == 1 ? 4 * (mode_ext + 1) : sblimit;
  if (bound > sblimit) bound = sblimit;
  for (int sb = 0; sb < sblimit; sb++) n += nbal[sb] * (sb < bound ? nch : 1);
  return n;
}

/* slot at logical frame i; avail_bits: bits from there to the end of the stream. Returns the status, fills r. */
static int classify(const uint8_t * b, long avail_bits, int bit_rate, dabo_mp2_rec * r, int * lsf)
{
  int alloc[2][32];
  r->header = field(b, 0, 32);
  r->crc_stored = r->crc_computed = -1;
  *lsf = 0;
  if (field(b, 0, 12) != 0xfff || field(b, 13, 2) != 2 || b[15]) return 1;
  const int id = b[12], idx = (int)field(b, 16, 4), sfreq = (int)field(b, 20, 2), mode = (int)field(b, 24, 2), ext = (int)field(b, 26, 2);
  const int rate = id ? RATE_MPEG1[idx] : RATE_LSF[idx];
  if (sfreq != 1 || rate == 0 || rate != bit_rate) return 2;
  *lsf = !id;
  r->crc_stored = (int)field(b, 32, 16);
  long limit = (id ? 24L : 48L) * bit_rate;
  if (limit > avail_bits) limit = avail_bits;
  const int nch = mode == 3 ? 1 : 2;
  const int * nbal;
  int sblimit, bound;
  alloc_table(id, bit_rate, nch, &nbal, &sblimit);
  bound = mode == 1 ? 4 * (ext + 1) : sblimit;
  if (bound > sblimit) bound = sblimit;
  long pos = 48;
  for (int sb = 0; sb < sblimit; sb++)
  {
    if (sb < bound)
      for (int ch = 0; ch < nch; ch++)
      {
        if (pos + nbal[sb] > limit) return 4;
        alloc[ch][sb] = (int)field(b, pos, nbal[sb]);
        pos += nbal[sb];
      }
    else
    {
      if (pos + nbal[sb] > limit) return 4;
      alloc[0][sb] = alloc[1][sb] = (int)field(b, pos, nbal[sb]);
      pos += nbal[sb];
    }
  }
  for (int sb = 0; sb < sblimit; sb++)
    for (int ch = 0; ch < nch; ch++)
      if (alloc[ch][sb])
      {
        if (pos + 2 > limit) return 4;
        pos += 2;
      }
  /* protected: header bits 16..31, then everything from the end of crc_check to the end of the SCFSI */
  unsigned crc = crc_over_bits(0xffffu, b + 16, 16);
  crc = crc_over_bits(crc, b + 48, pos - 48);
  r->crc_computed = (int)crc;
  return r->crc_computed == r->crc_stored ? 0 : 3;
}

/* frame_bits: n_frames x 24*bit_rate bits. Writes up to cap records and, if payload is not NULL, the OK frames' bytes (packed
 * MSB first) in record order. Returns the number of records. */
int dabo_mp2_run(const uint8_t * frame_bits, int bit_rate, int n_frames, dabo_mp2_rec * out, int cap, uint8_t * payload)
{
  const long fbits = 24L * bit_rate;
  long n_rec = 0, o = 0;
  for (int i = 0; i < n_frames;)
  {
    dabo_mp2_rec r;
    int lsf;
    const uint8_t * b = frame_bits + (long)i * fbits;
    r.first_frame = i;
    r.n_frames = 1;
    r.status = classify(b, (long)(n_frames - i) * fbits, bit_rate, &r, &lsf);
    if (r.status == 0 && lsf)
    {
      if (i + 1 < n_frames) r.n_frames = 2;
      else r.status = 4;
    }
    if (r.status == 0 && payload)
      for (long k = 0; k < r.n_frames * fbits; k += 8)
      {
        payload[o] = (uint8_t)field(b, k, 8);
        o++;
      }
    if (n_rec < cap) out[n_rec] = r;
    n_rec++;
    i += r.n_frames;
  }
  return (int)n_rec;
}
