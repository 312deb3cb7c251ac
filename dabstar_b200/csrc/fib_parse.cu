// fib_parse.cu — host-side multiplex configuration parser: FIG 0/0, 0/1, 0/2, 0/3 out of CRC-good FIBs.
//
// The minimal part of the reference's FibDecoder the decode path itself depends on (SURVEY.md section 8f.1):
//   FibDecoder::process_FIB            decoder/fib_decoder.cpp:59-106       FIG walk inside one FIB
//   FibDecoder::_process_Fig0s0        decoder/fib_decoder_fig0.cpp:89-113  ensemble id, change flags, CIF counter
//   FibDecoder::_subprocess_Fig0s1     decoder/fib_decoder_fig0.cpp:142-227 sub-channel organisation (short / long form)
//   FibDecoder::_subprocess_Fig0s2     decoder/fib_decoder_fig0.cpp:229-290 service -> sub-channel binding
//   cProtLevelTable                    decoder/fib_table.h:51               EN 300 401 table 8 (short-form index)
// It feeds MscHandler::set_channel (which sub-channels exist, where, how protected) and EtiGenerator (CIF counter,
// sub-channel list). FIG 0/3 (EN 300 401 clause 6.3.2: where a packet-mode component is carried) and FIG 0/14 (clause 6.2.2: the
// FEC scheme of a packet-mode sub-channel) are read from the standard; they feed the packet pass's self-configuration only and
// never restart the parser. Labels, announcements, the "next
// configuration" database and the GUI timers of the reference's decoder are not part of it. Only the current configuration
// (C/N = 0) is collected.
// Plain host C++ (no device code); lives in a .cu file so that the one nvcc command of build.py picks it up.
#include "dabstar_b200.h"

#include <cstring>
#include <vector>

namespace
{
// EN 300 401 table 8: sub-channel size in CU for the short-form table index. Index order: bit rates 32..384 kbit/s,
// within a rate protection level 5 down to 1, without the six pairs the table leaves out.
struct Table8Row { int16_t cu; int8_t level; int16_t rate; };
const Table8Row * table8()
{
  static Table8Row rows[64];
  static bool ready = false;
  if (!ready)
  {
    static const int16_t rates[14] = { 32, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320, 384 };
    // CU sizes per rate for levels 5,4,3,2,1 (0 = pair not in the table)
    static const int16_t cu[14][5] = { { 16, 21, 24, 29, 35 }, { 24, 29, 35, 42, 52 }, { 29, 35, 42, 52, 0 }, { 32, 42, 48, 58, 70 },
                                       { 40, 52, 58, 70, 84 }, { 48, 58, 70, 84, 104 }, { 58, 70, 84, 104, 0 }, { 64, 84, 96, 116, 140 },
                                       { 80, 104, 116, 140, 168 }, { 96, 116, 140, 168, 208 }, { 116, 140, 168, 208, 232 },
                                       { 128, 168, 192, 232, 280 }, { 160, 208, 0, 280, 0 }, { 192, 0, 280, 0, 416 } };
    int n = 0;
    for (int r = 0; r < 14; r++)
      for (int l = 0; l < 5; l++)
        if (cu[r][l] != 0) rows[n++] = { cu[r][l], (int8_t)(5 - l), rates[r] };
    ready = true;
  }
  return rows;
}

inline unsigned bits(const uint8_t * d, int off, int n) // d: one bit per byte, most significant first
{
  unsigned v = 0;
  for (int i = 0; i < n; i++) v = (v << 1) | (d[off + i] & 1u);
  return v;
}
} // namespace

struct dabstar_fib_parser
{
  dabstar_ensemble_info ens{};
  bool have_ens = false;
  std::vector<dabstar_subch> subch;          // in order of first appearance (FibConfigFig0::Fig0s1_BasicSubChannelOrganizationVec)
  std::vector<dabstar_service_comp> comps;   // (SId, component index) in order of first appearance
  std::vector<dabstar_packet_comp> pcomps;   // FIG 0/3, by SCId in order of first appearance
  std::vector<dabstar_fec_scheme> fec;       // FIG 0/14, by SubChId in order of first appearance
  int prev_change = 0;
  int restarts = 0;

  void restart() { subch.clear(); comps.clear(); pcomps.clear(); fec.clear(); restarts++; }   // FibDecoder::_restart_fib_decoding: collected content is untrustworthy

  // returns bytes used, -1 to abandon the FIB, or -2 to abandon this FIG: an entry that would cross the end of the FIG
  // (fig_bits = its length in bits) is not read - a CRC-good but malformed FIG must not make the parser read past the FIB
  int fig0s1(const uint8_t * d, int off_bytes, int fig_bits)
  {
    int o = off_bytes * 8;
    if (o + 24 > fig_bits) return -2;
    dabstar_subch s{};
    s.sub_ch_id = (int)bits(d, o, 6);
    bool known = false;
    bool known_short = false;
    for (const dabstar_subch & e : subch) if (e.sub_ch_id == s.sub_ch_id) { known = true; known_short = e.short_form != 0; }
    if (known) return (o + (known_short ? 24 : 32)) / 8; // the stored form decides the length, as the reference does
    s.start_cu = (int)bits(d, o + 6, 10);
    s.short_form = bits(d, o + 16, 1) == 0 ? 1 : 0;
    if (!s.short_form && o + 32 > fig_bits) return -2;
    if (s.short_form)
    {
      const Table8Row & row = table8()[bits(d, o + 18, 6)];
      s.size_cu = row.cu;
      s.prot_level = row.level;
      s.bit_rate = row.rate;
      o += 24;
    }
    else
    {
      const int option = (int)bits(d, o + 17, 3), level = (int)bits(d, o + 20, 2);
      s.size_cu = (int)bits(d, o + 22, 10);
      static const int per8[4] = { 12, 8, 6, 4 }, per32[4] = { 27, 21, 18, 15 };
      if (option == 0) { s.bit_rate = s.size_cu / per8[level] * 8; s.prot_level = level; }
      else if (option == 1) { s.bit_rate = s.size_cu / per32[level] * 32; s.prot_level = level + 4; }
      else { s.bit_rate = 0; s.prot_level = level; }
      o += 32;
    }
    // a sub-channel must fit into the 864 CU of a CIF and must not overlap a known one; else everything collected is dropped
    bool bad = s.start_cu + s.size_cu > 864;
    for (const dabstar_subch & e : subch)
      if (e.size_cu > 0 && s.start_cu < e.start_cu + e.size_cu && e.start_cu < s.start_cu + s.size_cu) bad = true;
    if (bad) { restart(); return -1; }
    subch.push_back(s);
    return o / 8;
  }

  int fig0s2(const uint8_t * d, int off_bytes, int pd, int fig_bits)
  {
    int o = off_bytes * 8;
    if (o + (pd ? 40 : 24) > fig_bits) return -2;
    const uint32_t sid = pd ? bits(d, o, 32) : bits(d, o, 16);
    o += pd ? 32 : 16;
    const int n = (int)bits(d, o + 4, 4);
    o += 8;
    if (o + 16 * n > fig_bits) return -2;
    for (int c = 0; c < n; c++, o += 16)
    {
      bool known = false;
      for (const dabstar_service_comp & e : comps) if (e.sid == sid && e.comp_index == c) known = true;
      if (known) continue;
      dabstar_service_comp sc{};
      sc.sid = sid;
      sc.comp_index = c;
      sc.tmid = (int)bits(d, o, 2);
      sc.sub_ch_id = -1;
      if (sc.tmid == 0 || sc.tmid == 1) { sc.type = (int)bits(d, o + 2, 6); sc.sub_ch_id = (int)bits(d, o + 8, 6); }
      else if (sc.tmid == 3) sc.type = (int)bits(d, o + 2, 12); // SCId of a packet-mode component
      sc.primary = (int)bits(d, o + 14, 1);
      sc.ca_flag = (int)bits(d, o + 15, 1);
      comps.push_back(sc);
    }
    return o / 8;
  }

  // FIG 0/3: SCId (12), Rfa (3), CAOrg flag, DG flag, Rfu, DSCTy (6), SubChId (6), packet address (10), CAOrg (16) if flagged
  int fig0s3(const uint8_t * d, int off_bytes, int fig_bits)
  {
    const int o = off_bytes * 8;
    if (o + 40 > fig_bits) return -2;
    const int ca = (int)bits(d, o + 15, 1), len = ca ? 56 : 40;
    if (o + len > fig_bits) return -2;
    dabstar_packet_comp pc{};
    pc.scid = (int)bits(d, o, 12);
    pc.dg_flag = (int)bits(d, o + 16, 1);
    pc.dscty = (int)bits(d, o + 18, 6);
    pc.sub_ch_id = (int)bits(d, o + 24, 6);
    pc.packet_address = (int)bits(d, o + 30, 10);
    pc.ca_org = ca ? (int)bits(d, o + 40, 16) : -1;
    bool known = false;
    for (const dabstar_packet_comp & e : pcomps) if (e.scid == pc.scid) known = true;
    if (!known) pcomps.push_back(pc);
    return (o + len) / 8;
  }

  // FIG 0/14: SubChId (6), FEC scheme (2)
  int fig0s14(const uint8_t * d, int off_bytes, int fig_bits)
  {
    const int o = off_bytes * 8;
    if (o + 8 > fig_bits) return -2;
    const dabstar_fec_scheme e{ (int)bits(d, o, 6), (int)bits(d, o + 6, 2) };
    bool known = false;
    for (const dabstar_fec_scheme & x : fec) if (x.sub_ch_id == e.sub_ch_id) known = true;
    if (!known) fec.push_back(e);
    return (o + 8) / 8;
  }

  void push(const uint8_t * fib) // 256 bits, one per byte; the caller has checked the CRC
  {
    int processed = 0;
    while (processed < 30)
    {
      const uint8_t * d = fib + processed * 8;
      const int type = (int)bits(d, 0, 3), len = (int)bits(d, 3, 5);
      if (type == 7 && len == 31) break;                 // end marker
      if (processed + len + 1 > 30) break;               // FIG package length error
      if (type == 0 && len >= 1)
      {
        const int cn = (int)bits(d, 8, 1), pd = (int)bits(d, 10, 1), ext = (int)bits(d, 11, 5);
        if (ext == 0 && len >= 5)
        {
          ens.eid = (int)bits(d, 16, 16);
          ens.change_flags = (int)bits(d, 32, 2);
          ens.alarm = (int)bits(d, 34, 1);
          ens.cif_count_hi = (int)bits(d, 35, 5);
          ens.cif_count_lo = (int)bits(d, 40, 8);
          have_ens = true;
          prev_change = ens.change_flags;
        }
        else if (cn == 0 && ext == 3)
        {
          int used = 2;
          while (used < len + 1 && (used = fig0s3(d, used, 8 * (len + 1))) >= 0) {}
        }
        else if (cn == 0 && ext == 14)
        {
          int used = 2;
          while (used < len + 1 && (used = fig0s14(d, used, 8 * (len + 1))) >= 0) {}
        }
        else if (cn == 0 && (ext == 1 || ext == 2))
        {
          int used = 2; // FIG header + type-0 header
          bool abandon = false;
          while (used < len + 1)
          {
            used = ext == 1 ? fig0s1(d, used, 8 * (len + 1)) : fig0s2(d, used, pd, 8 * (len + 1));
            if (used == -2) break;                       // truncated entry: the rest of this FIG is not evaluated
            if (used < 0) { abandon = true; break; }
          }
          if (abandon) break; // the rest of this FIB is not evaluated
        }
      }
      processed += len + 1;
    }
  }
};

extern "C" int dabstar_fib_parser_create(dabstar_fib_parser ** out)
{
  if (!out) return DABSTAR_E_INVALID;
  *out = new dabstar_fib_parser;
  return 0;
}
extern "C" void dabstar_fib_parser_destroy(dabstar_fib_parser * p) { delete p; }
extern "C" int dabstar_fib_parser_push(dabstar_fib_parser * p, const uint8_t * fib_bits, int n_fibs)
{
  if (!p || (!fib_bits && n_fibs > 0) || n_fibs < 0) return DABSTAR_E_INVALID;
  for (int i = 0; i < n_fibs; i++) p->push(fib_bits + (size_t)i * 256);
  return 0;
}
extern "C" int dabstar_fib_parser_ensemble(const dabstar_fib_parser * p, dabstar_ensemble_info * out)
{
  if (!p || !out) return DABSTAR_E_INVALID;
  *out = p->ens;
  out->n_subch = (int)p->subch.size();
  out->n_components = (int)p->comps.size();
  out->restarts = p->restarts;
  return p->have_ens ? 1 : 0;
}
extern "C" int dabstar_fib_parser_subchannels(const dabstar_fib_parser * p, dabstar_subch * out, int cap)
{
  if (!p || (!out && cap > 0)) return DABSTAR_E_INVALID;
  const int n = (int)p->subch.size() < cap ? (int)p->subch.size() : cap;
  for (int i = 0; i < n; i++) out[i] = p->subch[i];
  return (int)p->subch.size();
}
extern "C" int dabstar_fib_parser_components(const dabstar_fib_parser * p, dabstar_service_comp * out, int cap)
{
  if (!p || (!out && cap > 0)) return DABSTAR_E_INVALID;
  const int n = (int)p->comps.size() < cap ? (int)p->comps.size() : cap;
  for (int i = 0; i < n; i++) out[i] = p->comps[i];
  return (int)p->comps.size();
}
extern "C" int dabstar_fib_parser_packet_components(const dabstar_fib_parser * p, dabstar_packet_comp * out, int cap)
{
  if (!p || (!out && cap > 0)) return DABSTAR_E_INVALID;
  const int n = (int)p->pcomps.size() < cap ? (int)p->pcomps.size() : cap;
  for (int i = 0; i < n; i++) out[i] = p->pcomps[i];
  return (int)p->pcomps.size();
}
extern "C" int dabstar_fib_parser_fec_schemes(const dabstar_fib_parser * p, dabstar_fec_scheme * out, int cap)
{
  if (!p || (!out && cap > 0)) return DABSTAR_E_INVALID;
  const int n = (int)p->fec.size() < cap ? (int)p->fec.size() : cap;
  for (int i = 0; i < n; i++) out[i] = p->fec[i];
  return (int)p->fec.size();
}
