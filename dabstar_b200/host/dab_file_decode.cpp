// dab_file_decode — headless file-input harness: raw interleaved IQ file(s) -> decoded FIC / MSC bits on the GPU.
//
//   dab_file_decode [-f u8|i16|cf32] [-x container,bits,LSB|MSB,IQ|QI|I_Only|Q_Only] [-a] [-e] [-q quality.csv]
//                   [-s subChId,startCU,sizeCU,shortForm,protLevel,bitRate]... [-o prefix] file.iq [file2.iq ...]
//     -x  XML/UFF sample description (container int8|uint8|int16|int24|int32|float32) for layouts other than the three native ones
//     -c  containers: every file's header is inspected (RIFF/WAVE .wav / .sdr, XML .uff, else raw u8); samples are converted and
//         resampled to 2.048 MS/s as the reference's file readers do
//     -a  self-configuration: sub-channels from the recording's FIG 0/1 (no -s needed)
//     -t  with -a: TII detection on the null symbols the recording's CIF counter selects (5 per search, threshold 8 dB), and those
//         null symbols leave the demapper's null power alone, as in the reference with its FIB decoder running
//     -e  also write the ETI(NI) stream, <prefix><n>.eti (what DABstar's ETI generator writes)
//     -d  all|id[,id...]: DAB+ super-frames of those sub-channels (all: what the recording's FIG 0/2 lists as DAB+, needs -a),
//         found, repaired and cut into access units on the GPU; prints per sub-channel super-frames attempted / ok, RS corrections /
//         failures and access units good / bad; with -o, <prefix><n>.subch<id>.aus holds every CRC-good AU after its 2-byte
//         big-endian length
//     -m  all|id[,id...]: MPEG layer II audio frames of those sub-channels (all: what the recording's FIG 0/2 lists as MPEG layer
//         II, needs -a), header- and CRC-checked on the GPU; prints per sub-channel the audio-frame slots per status; with -o,
//         <prefix><n>.subch<id>.mp2 holds the OK frames (an MPEG audio elementary stream)
//     -p  all|id:address[,id:address...]: packet-mode data groups of those (sub-channel, address) streams (all: every packet-mode
//         component of the recording's FIG 0/2 and 0/3, needs -a), packets and groups checked on the GPU; prints per stream the
//         packet and group counters; with -o, <prefix><n>.subch<id>.addr<address>.dg holds the groups' bytes in order
//     -F  all|id[,id...]: packet-mode FEC (RS(204,188) FEC frames located and corrected on the GPU) in front of -p on those
//         sub-channels (all: every sub-channel the recording's FIG 0/14 gives FEC scheme 1, needs -a); prints per FEC sub-channel
//         its FEC frames per status and the rows corrected / failed
//     -q  signal quality of every frame as CSV: frame,sym0_pos,mer_db,snr_db,noise_power,fbb_hz (fbb_hz: the baseband frequency
//         correction of the frame's data symbols); with several files, file n's lines go to <path>.<n>
//
// The reference can only play files through its GUI, paced to real time (raw_reader.cpp:153-165); this harness feeds
// whole files to dabstar::DabProcessor (one reference DabProcessor per file, all files in lock step) and writes
//   <prefix><n>.fic      CRC-good FIBs packed to 32 bytes, the reference's FIC dump format (fic_decoder.cpp:291-308)
//   <prefix><n>.sub<id>  the sub-channel's logical frames packed 8 bits per byte (as eti_generator.cpp:403-411 packs them)
// Build: g++ -std=c++17 -O2 dab_file_decode.cpp -I../../include -L.. -ldabstar_b200 -o dab_file_decode
#include "dabstar_facade.hpp"

#include <cstdio>
#include <cstdlib>
#include <string>

static std::vector<unsigned char> read_file(const char * path)
{
  FILE * f = fopen(path, "rb");
  if (!f) throw std::runtime_error(std::string("cannot open ") + path);
  fseek(f, 0, SEEK_END);
  const long n = ftell(f);
  fseek(f, 0, SEEK_SET);
  std::vector<unsigned char> v((size_t)n);
  if (n > 0 && fread(v.data(), 1, (size_t)n, f) != (size_t)n) { fclose(f); throw std::runtime_error("short read"); }
  fclose(f);
  return v;
}

int main(int argc, char ** argv)
{
  int fmt = DABSTAR_FMT_U8;
  bool autoCfg = false, eti = false, xml = false, containers = false, tii = false;
  dabstar_sample_format sf{};
  std::string prefix = "dab_out_", qualPath, dabplus, mp2, packet, fec;
  bool prefixSet = false;
  std::vector<dabstar_subch> subch;
  std::vector<const char *> files;
  for (int i = 1; i < argc; i++)
  {
    const std::string a = argv[i];
    if (a == "-f" && i + 1 < argc) { const std::string v = argv[++i]; fmt = v == "i16" ? DABSTAR_FMT_I16 : (v == "cf32" ? DABSTAR_FMT_CF32 : DABSTAR_FMT_U8); }
    else if (a == "-o" && i + 1 < argc) { prefix = argv[++i]; prefixSet = true; }
    else if (a == "-d" && i + 1 < argc) dabplus = argv[++i];
    else if (a == "-m" && i + 1 < argc) mp2 = argv[++i];
    else if (a == "-p" && i + 1 < argc) packet = argv[++i];
    else if (a == "-F" && i + 1 < argc) fec = argv[++i];
    else if (a == "-a") autoCfg = true;
    else if (a == "-t") tii = true;
    else if (a == "-c") { containers = true; fmt = DABSTAR_FMT_CF32; }
    else if (a == "-e") eti = true;
    else if (a == "-q" && i + 1 < argc) qualPath = argv[++i];
    else if (a == "-x" && i + 1 < argc)
    {
      char cont[16] = { 0 }, order[8] = { 0 }, iq[16] = { 0 };
      int bitsPer = 0;
      if (sscanf(argv[++i], "%15[^,],%d,%7[^,],%15s", cont, &bitsPer, order, iq) != 4) { fprintf(stderr, "bad -x\n"); return 2; }
      static const char * const conts[6] = { "int8", "uint8", "int16", "int24", "int32", "float32" };
      static const char * const orders[4] = { "IQ", "QI", "I_Only", "Q_Only" };
      sf.container = -1; sf.iq_order = -1;
      for (int k = 0; k < 6; k++) if (std::string(cont) == conts[k]) sf.container = k;
      for (int k = 0; k < 4; k++) if (std::string(iq) == orders[k]) sf.iq_order = k;
      sf.bits_per_channel = bitsPer;
      sf.msb_first = std::string(order) == "MSB";
      xml = true;
      fmt = DABSTAR_FMT_CF32;
    }
    else if (a == "-s" && i + 1 < argc)
    {
      dabstar_subch s{};
      if (sscanf(argv[++i], "%d,%d,%d,%d,%d,%d", &s.sub_ch_id, &s.start_cu, &s.size_cu, &s.short_form, &s.prot_level, &s.bit_rate) != 6) { fprintf(stderr, "bad -s\n"); return 2; }
      subch.push_back(s);
    }
    else files.push_back(argv[i]);
  }
  if (files.empty()) { fprintf(stderr, "usage: dab_file_decode [-f u8|i16|cf32] [-s id,startCU,sizeCU,shortForm,protLevel,bitRate]... [-o prefix] file.iq ...\n"); return 2; }
  try
  {
    dabstar::Context ctx(0);
    const int elem = xml ? dabstar_sample_format_bytes(&sf) : 0;
    if (xml && elem == 0) { fprintf(stderr, "unknown sample format in -x\n"); return 2; }
    const size_t bps = xml ? (size_t)elem : (fmt == DABSTAR_FMT_U8 ? 2 : (fmt == DABSTAR_FMT_I16 ? 4 : 8));
    std::vector<std::vector<unsigned char>> data;
    std::vector<const void *> ptrs;
    std::vector<int64_t> ns;
    std::vector<std::vector<float>> conv;
    for (const char * f : files) { data.push_back(read_file(f)); }
    if (containers)
    {
      for (size_t r = 0; r < data.size(); r++)
      {
        dabstar_file_info fi{};
        conv.push_back(dabstar::read_recording(ctx, data[r].data(), data[r].size(), &fi));
        static const char * const kinds[3] = { "raw", "xml", "wav" };
        printf("%s: %s container, %d S/s, %lld samples from byte %lld\n", files[r], kinds[fi.kind], fi.sample_rate, (long long)fi.n_samples, (long long)fi.data_offset);
      }
      for (auto & v : conv) { ptrs.push_back(v.data()); ns.push_back((int64_t)(v.size() / 2)); }
    }
    else
      for (auto & d : data) { ptrs.push_back(d.data()); ns.push_back((int64_t)(d.size() / bps)); }
    dabstar::DabProcessor proc(ctx, (int)files.size(), fmt, subch.empty() && !autoCfg);
    for (size_t r = 0; r < files.size(); r++)
    {
      if (autoCfg) proc.set_auto_config((int)r, true, tii);
      if (autoCfg && tii) proc.set_tii_processing((int)r, true);
      else proc.set_audio_channel((int)r, subch);
      if (eti) proc.start_eti_generator((int)r);
      for (const bool isMp2 : { false, true })
      {
        const std::string & sel = isMp2 ? mp2 : dabplus;
        auto set = [&](int id) { if (isMp2) proc.set_mp2((int)r, id); else proc.set_dabplus((int)r, id); };
        if (sel == "all") set(-1);
        else if (!sel.empty())
          for (size_t p = 0; p <= sel.size();)
          {
            const size_t q = std::min(sel.find(',', p), sel.size());
            set(atoi(sel.substr(p, q - p).c_str()));
            p = q + 1;
          }
      }
    }
    std::vector<std::pair<int, int>> streams; // -p id:address list
    for (size_t p = 0; packet != "all" && p < packet.size();)
    {
      const size_t q = std::min(packet.find(',', p), packet.size());
      const std::string item = packet.substr(p, q - p);
      const size_t c = item.find(':');
      if (c == std::string::npos) throw std::runtime_error("-p: expected id:address, got " + item);
      streams.push_back({ atoi(item.substr(0, c).c_str()), atoi(item.substr(c + 1).c_str()) });
      p = q + 1;
    }
    std::vector<int> fecIds; // -F id list
    for (size_t p = 0; fec != "all" && p < fec.size();)
    {
      const size_t q = std::min(fec.find(',', p), fec.size());
      fecIds.push_back(atoi(fec.substr(p, q - p).c_str()));
      p = q + 1;
    }
    for (size_t r = 0; r < files.size(); r++)
    {
      if (packet == "all") proc.set_packet((int)r, -1);
      for (const auto & x : streams) proc.set_packet((int)r, x.first, x.second);
      if (fec == "all") proc.set_packet_fec((int)r, -1);
      for (int id : fecIds) proc.set_packet_fec((int)r, id);
    }
    if (!qualPath.empty()) proc.set_frame_quality(true);
    if (xml && !containers) proc.run_files(ptrs, ns, sf);
    else proc.run(ptrs, ns);
    for (size_t r = 0; r < files.size(); r++)
    {
      if (autoCfg)
      {
        subch = proc.sub_channels((int)r);
        for (auto & s : subch) printf("%s: sub-channel %d: CU %d+%d, %s level %d, %d kbit/s\n", files[r], s.sub_ch_id, s.start_cu, s.size_cu, s.short_form ? "UEP" : "EEP", s.prot_level, s.bit_rate);
      }
      if (eti)
      {
        const std::vector<dabstar::u8> e = proc.eti((int)r);
        FILE * ef = fopen((prefix + std::to_string(r) + ".eti").c_str(), "wb");
        if (ef) { fwrite(e.data(), 1, e.size(), ef); fclose(ef); }
        printf("%s: %zu ETI(NI) frames\n", files[r], e.size() / 6144);
      }
      long fibs = 0;
      FILE * fic = fopen((prefix + std::to_string(r) + ".fic").c_str(), "wb");
      std::vector<FILE *> outs;
      for (auto & s : subch) outs.push_back(fopen((prefix + std::to_string(r) + ".sub" + std::to_string(s.sub_ch_id)).c_str(), "wb"));
      proc.deliver((int)r,
        [&](const std::array<dabstar::u8, 256> & fib, dabstar::u16) {
          unsigned char b[32];
          for (int j = 0; j < 32; j++) { b[j] = 0; for (int k = 0; k < 8; k++) b[j] = (unsigned char)((b[j] << 1) | (fib[8 * j + k] & 1)); }
          if (fic) fwrite(b, 1, 32, fic);
          fibs++;
        },
        [&](int id, const std::vector<dabstar::u8> & bits) {
          for (size_t c = 0; c < subch.size(); c++)
          {
            if (subch[c].sub_ch_id != id || !outs[c]) continue;
            for (size_t j = 0; j + 8 <= bits.size(); j += 8) { unsigned char b = 0; for (int k = 0; k < 8; k++) b = (unsigned char)((b << 1) | (bits[j + k] & 1)); fputc(b, outs[c]); }
          }
        }, subch);
      if (fic) fclose(fic);
      for (FILE * o : outs) if (o) fclose(o);
      printf("%s: %d frames, %ld good FIBs, %.2f ms device time\n", files[r], proc.n_frames((int)r), fibs, proc.last_ms());
      for (const auto & s : proc.sub_channels((int)r))
      {
        if (dabplus.empty() || !proc.dabplus_decoded((int)r, s.sub_ch_id)) continue;
        long good = 0, bad = 0;
        FILE * af = prefixSet ? fopen((prefix + std::to_string(r) + ".subch" + std::to_string(s.sub_ch_id) + ".aus").c_str(), "wb") : nullptr;
        const std::vector<dabstar_superframe> sfs = proc.superframes((int)r, s.sub_ch_id, [&](const dabstar::u8 * au, int len, const dabstar_superframe &) {
          good++;
          if (af) { fputc((len >> 8) & 0xff, af); fputc(len & 0xff, af); fwrite(au, 1, (size_t)len, af); }
        });
        if (af) fclose(af);
        long ok = 0, corr = 0, fail = 0;
        for (const auto & x : sfs)
        {
          ok += x.ok ? 1 : 0;
          corr += x.rs_corrections;
          fail += x.rs_errors;
          for (int u = 0; x.ok && u < x.num_aus; u++) bad += x.au_state[u] != 1 ? 1 : 0;
        }
        printf("%s: DAB+ sub-channel %d: %zu super-frames attempted, %ld ok, %ld RS corrections, %ld RS failures, %ld AUs good, %ld bad\n", files[r], s.sub_ch_id,
               sfs.size(), ok, corr, fail, good, bad);
      }
      for (const auto & s : proc.sub_channels((int)r))
      {
        if (mp2.empty() || !proc.mp2_decoded((int)r, s.sub_ch_id)) continue;
        FILE * mf = prefixSet ? fopen((prefix + std::to_string(r) + ".subch" + std::to_string(s.sub_ch_id) + ".mp2").c_str(), "wb") : nullptr;
        const std::vector<dabstar_mp2_frame> fr = proc.mp2_frames((int)r, s.sub_ch_id, [&](const dabstar::u8 * f, int len, const dabstar_mp2_frame &) {
          if (mf) fwrite(f, 1, (size_t)len, mf);
        });
        if (mf) fclose(mf);
        long cnt[5] = { 0 };
        for (const auto & x : fr) if (x.status >= 0 && x.status < 5) cnt[x.status]++;
        printf("%s: MP2 sub-channel %d: %zu slots, %ld ok, %ld no header, %ld mismatch, %ld CRC errors, %ld cut\n", files[r], s.sub_ch_id, fr.size(), cnt[0], cnt[1],
               cnt[2], cnt[3], cnt[4]);
      }
      std::vector<std::pair<int, int>> decoded = streams;
      if (packet == "all")
        for (const auto & c : proc.packet_components((int)r)) decoded.push_back({ c.sub_ch_id, c.packet_address });
      for (size_t k = 0; k < decoded.size(); k++)
      {
        const int id = decoded[k].first, addr = decoded[k].second;
        bool seen = false;
        for (size_t j = 0; j < k; j++) seen = seen || decoded[j] == decoded[k];
        if (seen || !proc.packet_decoded((int)r, id, addr)) continue;
        FILE * df = prefixSet ? fopen((prefix + std::to_string(r) + ".subch" + std::to_string(id) + ".addr" + std::to_string(addr) + ".dg").c_str(), "wb") : nullptr;
        const std::vector<dabstar_data_group> gr = proc.data_groups((int)r, id, addr, [&](const dabstar::u8 * g, int len, const dabstar_data_group &) {
          if (df) fwrite(g, 1, (size_t)len, df);
        });
        if (df) fclose(df);
        const dabstar_packet_stats st = proc.packet_stats((int)r, id, addr);
        printf("%s: packet sub-channel %d address %d: %zu groups, %lld ok, %lld no CRC, %lld CRC errors, %lld malformed, %lld raw; %lld packets, %lld CRC errors, "
               "%lld bad length, %lld cut, %lld padding, %lld command, %lld other address, %lld continuity breaks, %lld abandoned, %lld dropped\n",
               files[r], id, addr, gr.size(), (long long)st.groups[0], (long long)st.groups[1], (long long)st.groups[2], (long long)st.groups[3], (long long)st.groups[4],
               (long long)st.packets, (long long)st.crc_errors, (long long)st.bad_length, (long long)st.cut, (long long)st.padding, (long long)st.command,
               (long long)st.other_address, (long long)st.continuity_breaks, (long long)st.abandoned, (long long)st.dropped);
      }
      for (int id = 0; !fec.empty() && id < 64; id++)
      {
        if (!proc.fec_decoded((int)r, id)) continue;
        long cnt[4] = { 0 }, fixed = 0, failed = 0, bytes = 0;
        const std::vector<dabstar_fec_frame> fr = proc.fec_frames((int)r, id);
        for (const auto & x : fr)
        {
          if (x.status >= 0 && x.status < 4) cnt[x.status]++;
          fixed += x.rows_corrected; failed += x.rows_failed; bytes += x.bytes_corrected;
        }
        printf("%s: FEC sub-channel %d: %zu FEC frames, %ld clean, %ld corrected, %ld partial, %ld incomplete; %ld rows corrected (%ld bytes), %ld rows failed\n",
               files[r], id, fr.size(), cnt[0], cnt[1], cnt[2], cnt[3], fixed, bytes, failed);
      }
      if (autoCfg && tii)
        for (const auto & ev : proc.tii_events((int)r))
          for (const auto & id : ev.transmitterIds)
            printf("%s: frame %d: TII main id %d sub id %d strength %.2f phase %.0f deg%s\n", files[r], ev.frame, id.main_id, id.sub_id, id.strength, id.phase_deg,
                   id.non_etsi ? " (non-ETSI phases)" : "");
      if (proc.n_frames((int)r) > 0)
      {
        const dabstar::SLcdData q = proc.lcd_data((int)r);
        printf("%s: MER %.1f dB, SNR %.1f dB\n", files[r], q.MER, q.SNR);
      }
      if (!qualPath.empty())
      {
        const std::string path = files.size() > 1 ? qualPath + "." + std::to_string(r) : qualPath;
        FILE * qf = fopen(path.c_str(), "w");
        if (!qf) throw std::runtime_error("cannot write " + path);
        const std::vector<dabstar::SLcdData> lcd = proc.frame_lcd_data((int)r);
        const std::vector<dabstar_frame_info> info = proc.frame_info((int)r);
        fprintf(qf, "frame,sym0_pos,mer_db,snr_db,noise_power,fbb_hz\n");
        for (size_t f = 0; f < lcd.size() && f < info.size(); f++)
          fprintf(qf, "%zu,%lld,%.4f,%.4f,%.9g,%.3f\n", f, (long long)info[f].sym0_pos, lcd[f].MER, lcd[f].SNR, lcd[f].NoisePower, info[f].fbb_data);
        fclose(qf);
      }
    }
  }
  catch (const std::exception & e) { fprintf(stderr, "error: %s\n", e.what()); return 1; }
  return 0;
}
