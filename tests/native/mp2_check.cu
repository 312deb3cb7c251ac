// Host driver of mp2.cuh as the MP2 pass runs it: classify every logical frame of a stream (k_mp2_scan), then walk the slots
// (k_mp2_walk) and collect the OK frames' bytes (k_mp2_compact).
// stdin, one command per line:
//   crc <hex bytes>                  -> CRC-16 (mp2_crc_bits, preset 0xFFFF) of the bytes
//   alloc <table> <nch> <bound>      -> allocation bits of a frame (mp2_sblimit / mp2_nbal)
//   run <bit_rate> <n_frames> <hex>  -> "<n_records>", one line "first n status header crc_stored crc_computed" per record, then
//                                       the payload as hex ("-" if empty)
#include "mp2.cuh"

#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

static std::vector<uint8_t> read_hex()
{
  std::vector<uint8_t> v;
  int c;
  while ((c = getchar()) == ' ') {}
  int hi = -1;
  while (c != EOF && c != '\n')
  {
    const int d = c <= '9' ? c - '0' : (c | 32) - 'a' + 10;
    if (hi < 0) hi = d;
    else { v.push_back((uint8_t)(hi * 16 + d)); hi = -1; }
    c = getchar();
  }
  return v;
}

int main()
{
  char cmd[16];
  while (scanf("%15s", cmd) == 1)
  {
    if (!strcmp(cmd, "crc"))
    {
      const std::vector<uint8_t> b = read_hex();
      unsigned crc = 0xffffu;
      for (uint8_t x : b) crc = dab::mp2_crc_bits(crc, x, 8);
      printf("%u\n", crc);
    }
    else if (!strcmp(cmd, "alloc"))
    {
      int table, nch, bound, n = 0;
      if (scanf("%d %d %d", &table, &nch, &bound) != 3) return 1;
      for (int sb = 0; sb < dab::mp2_sblimit(table); sb++) n += dab::mp2_nbal(table, sb) * (sb < bound ? nch : 1);
      printf("%d\n", n);
    }
    else if (!strcmp(cmd, "run"))
    {
      int bit_rate, n;
      if (scanf("%d %d", &bit_rate, &n) != 2) return 1;
      const std::vector<uint8_t> p = read_hex();
      const long long fb = 3LL * bit_rate;
      if ((long long)p.size() != n * fb) return 2;
      std::vector<uint8_t> cls((size_t)n);
      std::vector<dab::Mp2Slot> slot((size_t)n);
      for (int i = 0; i < n; i++)
      {
        slot[i] = dab::mp2_classify(p.data() + i * fb, (n - i) * fb, bit_rate);
        cls[i] = dab::mp2_class_byte(slot[i]);
      }
      std::vector<dab::Mp2Rec> rec;
      std::string pay;
      for (int i = 0; i < n;)
      {
        int status;
        const int span = dab::mp2_walk_step(cls[i], i, n, &status);
        rec.push_back(dab::Mp2Rec{ i, span, status, slot[i].header, slot[i].crc_stored, slot[i].crc_computed });
        if (status == dab::MP2_OK)
          for (long long b = i * fb; b < (i + span) * fb; b++)
          {
            char h[3];
            snprintf(h, sizeof h, "%02x", p[b]);
            pay += h;
          }
        i += span;
      }
      printf("%zu\n", rec.size());
      for (const auto & r : rec) printf("%d %d %d %u %d %d\n", r.first_frame, r.n_frames, r.status, r.header, r.crc_stored, r.crc_computed);
      printf("%s\n", pay.empty() ? "-" : pay.c_str());
    }
    else return 1;
    fflush(stdout);
  }
  return 0;
}
