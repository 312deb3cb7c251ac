// packet_kernels.cu — packet-mode data of DAB sub-channels on the GPU: the packets of every logical frame, the data-group
// assembly of each (sub-channel, address) stream, and the compaction of the groups with their MSC data group headers checked.
//
// A packet's length is in its own first two bits and packets tile the logical frame (ETSI EN 300 401 clause 5.3.2), so every
// logical frame is walked on its own (k_packet_scan, packet.cuh: packet_frame), once per sub-channel however many addresses are
// selected. Data groups span packets and logical frames; their assembly per address (k_packet_walk, built on packet_walk_step)
// is a scan: every thread of a stream's block takes a contiguous chunk of slots and block-wide scans give each chunk, in turn,
// the previous packet's continuity index and the useful bytes before it, its entry state (2-state maps, block_scan.cuh), where
// the group open at its entry started, and where its groups go. The groups' useful data are then concatenated in stream order
// and the MSC data group headers parsed and CRC-checked (k_packet_compact) for one copy to the host (engine.cu: run_packet).
#include "kernels.h"
#include "stream_search.cuh"
#include "block_scan.cuh"

namespace dab
{
namespace
{
// thread = logical frame of any sub-channel: its packets into the frame's slots (with packet-mode FEC: of its corrected bytes, the
// FEC packets skipped)
__global__ void __launch_bounds__(128) k_packet_scan(const PacketSub * __restrict__ sub, int n_subs, long long n_frames, PacketSlot * __restrict__ slots)
{
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_frames) return;
  const PacketSub & s = sub[find_stream(sub, n_subs, g, [](const PacketSub & x) { return x.frame0; })];
  const long long f = g - s.frame0;
  const int fb = 3 * s.bit_rate, spf = s.bit_rate / 8;
  packet_frame(s.src + f * fb, fb, slots + s.slot0 + f * spf, s.fec ? s.fec + f * spf : nullptr);
}

// What the walk carries from chunk to chunk. Scan 1: the CI of the last packet of the address (0 none, 4 | CI), and the count
// and useful bytes of those packets.
struct PktCarry
{
  unsigned ci;
  int pk;
  long long bytes;
};
__device__ inline PktCarry carry_then(PktCarry a, PktCarry b) { return PktCarry{ b.ci ? b.ci : a.ci, a.pk + b.pk, a.bytes + b.bytes }; }
// Scan 3: the group open at a chunk's end: tag 0 as at its entry (the chunk opened or closed nothing), 1 none, 2 + s opened at
// slot s with pk packets and bytes useful bytes of the address before it
struct PktOpen
{
  int tag, pk;
  long long bytes;
};
__device__ inline PktOpen open_then(PktOpen a, PktOpen b) { return b.tag ? b : a; }
// Scan 4: groups emitted and their useful bytes
struct PktOut
{
  long long groups, bytes;
};

// The walk over slots [i0, i1) of one address from (prev, state, open, pk, bytes); f(i, slot, cont, emit, abandon, drop) for
// every packet of the address; on an emit, open describes the group's first packet and pk / bytes count up to its end.
template <typename F>
__device__ inline void walk_chunk(const PacketSlot * __restrict__ sl, int i0, int i1, int a, unsigned & prev, int & state, PktOpen & open, int & pk,
                                  long long & bytes, F f)
{
  for (int i = i0; i < i1; i++)
  {
    const PacketSlot s = sl[i];
    if (!packet_mine(s, a)) continue;
    const bool cont = packet_continues(prev, s.hdr);
    const int fl = pkt_fl(s.hdr);
    int emit, abandon, drop;
    state = packet_walk_step(state, fl, cont, &emit, &abandon, &drop);
    if (fl >= 2) open = PktOpen{ 2 + i, pk, bytes };
    pk++;
    bytes += pkt_useful(s.hdr);
    prev = 4u | (unsigned)pkt_ci(s.hdr);
    f(i, s, cont, emit, abandon, drop);
    if (!state) open.tag = 1;
  }
}

constexpr int PACKET_WALK_THREADS = 256;
// block = stream
__global__ void __launch_bounds__(PACKET_WALK_THREADS) k_packet_walk(const PacketSub * __restrict__ subs, const PacketStream * __restrict__ st,
                                                                     const PacketSlot * __restrict__ slots, PacketStage * __restrict__ stage,
                                                                     PacketCount * __restrict__ cnt)
{
  __shared__ PktCarry sh_carry[32];
  __shared__ unsigned sh_map[32];
  __shared__ PktOpen sh_open[32];
  __shared__ PktOut sh_out[32];
  __shared__ unsigned long long sh_stat[10];
  const PacketStream & s = st[blockIdx.x];
  const PacketSub & sub = subs[s.sub];
  const int a = s.address;
  const int n = sub.n_frames * (sub.bit_rate / 8), per = (n + (int)blockDim.x - 1) / (int)blockDim.x;
  const int i0 = min(n, (int)threadIdx.x * per), i1 = min(n, i0 + per);
  const PacketSlot * sl = slots + sub.slot0;
  if (threadIdx.x < 10) sh_stat[threadIdx.x] = 0;
  auto none = [](int, const PacketSlot &, bool, int, int, int) {};

  // 1: previous CI, packets and bytes before the chunk
  PktCarry mine{ 0u, 0, 0 };
  for (int i = i0; i < i1; i++)
    if (packet_mine(sl[i], a)) { mine.ci = 4u | (unsigned)pkt_ci(sl[i].hdr); mine.pk++; mine.bytes += pkt_useful(sl[i].hdr); }
  const PktCarry in = block_exclusive_scan(mine, PktCarry{ 0u, 0, 0 }, carry_then, sh_carry, (PktCarry *)nullptr);
  // 2: entry state
  unsigned m = 0;
  for (int e = 0; e < 2; e++)
  {
    unsigned prev = in.ci;
    int state = e, pk = in.pk;
    long long bytes = in.bytes;
    PktOpen open{ 0, 0, 0 };
    walk_chunk(sl, i0, i1, a, prev, state, open, pk, bytes, none);
    m |= (unsigned)state << e;
  }
  const int entry = (int)(block_exclusive_scan(m, MAP_IDENTITY, map_then, sh_map, (unsigned *)nullptr) & 1u);
  // 3: the group open at the entry
  PktOpen tag{ 0, 0, 0 };
  {
    unsigned prev = in.ci;
    int state = entry, pk = in.pk;
    long long bytes = in.bytes;
    walk_chunk(sl, i0, i1, a, prev, state, tag, pk, bytes, none);
  }
  const PktOpen open_in = block_exclusive_scan(tag, PktOpen{ 0, 0, 0 }, open_then, sh_open, (PktOpen *)nullptr);
  // 4: groups, bytes and counters
  PktOut out{ 0, 0 };
  unsigned long long c[10] = { 0 };
  {
    unsigned prev = in.ci;
    int state = entry, pk = in.pk;
    long long bytes = in.bytes;
    PktOpen open = open_in;
    walk_chunk(sl, i0, i1, a, prev, state, open, pk, bytes, [&](int, const PacketSlot &, bool, int emit, int abandon, int drop) {
      c[0]++;
      if (emit) { out.groups++; out.bytes += bytes - open.bytes; }
      c[8] += abandon;
      c[9] += drop;
    });
  }
  { // the packets of the chunk by class; continuity breaks of the address
    unsigned prev = in.ci;
    for (int i = i0; i < i1; i++)
    {
      const PacketSlot x = sl[i];
      if (x.cls == PKT_CRC_ERROR) c[1]++;
      else if (x.cls == PKT_BAD_LENGTH) c[2]++;
      else if (x.cls == PKT_CUT) c[3]++;
      else if (x.cls == PKT_OK)
      {
        const int xa = pkt_addr(x.hdr);
        if (xa == 0) c[4]++;
        else if (xa != a) c[6]++;
        else if (pkt_cmd(x.hdr)) c[5]++;
        else
        {
          if ((prev & 4u) && !packet_continues(prev, x.hdr)) c[7]++;
          prev = 4u | (unsigned)pkt_ci(x.hdr);
        }
      }
    }
  }
  PktOut total;
  const PktOut off = block_exclusive_scan(out, PktOut{ 0, 0 }, [](PktOut x, PktOut y) { return PktOut{ x.groups + y.groups, x.bytes + y.bytes }; }, sh_out, &total);
  for (int k = 0; k < 10; k++)
    if (c[k]) atomicAdd(&sh_stat[k], c[k]);
  // 5: the groups
  {
    unsigned prev = in.ci;
    int state = entry, pk = in.pk;
    long long bytes = in.bytes;
    PktOpen open = open_in;
    long long k = s.stage0 + off.groups, o = off.bytes;
    walk_chunk(sl, i0, i1, a, prev, state, open, pk, bytes, [&](int i, const PacketSlot &, bool, int emit, int, int) {
      if (!emit) return;
      const int b = (int)(bytes - open.bytes);
      stage[k++] = PacketStage{ open.tag - 2, i, pk - open.pk, b, o };
      o += b;
    });
  }
  __syncthreads();
  if (threadIdx.x == 0)
  {
    PacketCount r;
    r.groups = total.groups; r.bytes = total.bytes;
    r.packets = (long long)sh_stat[0]; r.crc_errors = (long long)sh_stat[1]; r.bad_length = (long long)sh_stat[2]; r.cut = (long long)sh_stat[3];
    r.padding = (long long)sh_stat[4]; r.command = (long long)sh_stat[5]; r.other_address = (long long)sh_stat[6];
    r.continuity_breaks = (long long)sh_stat[7]; r.abandoned = (long long)sh_stat[8]; r.dropped = (long long)sh_stat[9];
    cnt[blockIdx.x] = r;
  }
}

// warp = output group: the useful data of its packets in order, then (lane 0) its MSC data group header and CRC
constexpr int PACKET_COMPACT_WARPS = 4;
__global__ void __launch_bounds__(32 * PACKET_COMPACT_WARPS, 1) k_packet_compact(const PacketSub * __restrict__ subs, const PacketStream * __restrict__ st, int n_streams,
                                                                              long long n_out, const PacketSlot * __restrict__ slots,
                                                                              const PacketStage * __restrict__ stage, DgRec * __restrict__ out_rec,
                                                                              uint8_t * __restrict__ out_pay)
{
  const long long k = (long long)blockIdx.x * PACKET_COMPACT_WARPS + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (k >= n_out) return;
  const PacketStream & s = st[find_stream(st, n_streams, k, [](const PacketStream & x) { return x.out_rec0; })];
  const PacketSub & sub = subs[s.sub];
  const PacketStage g = stage[s.stage0 + (k - s.out_rec0)];
  const int fb = 3 * sub.bit_rate, spf = sub.bit_rate / 8;
  const PacketSlot * sl = slots + sub.slot0;
  uint8_t * dst = out_pay + s.out_pay0 + g.off;
  int at = 0;
  for (int i = g.start; i <= g.end; i += 32)
  {
    const bool in = i + lane <= g.end && packet_mine(sl[i + lane], s.address);
    unsigned mask = __ballot_sync(0xffffffffu, in);
    while (mask)
    {
      const int b = __ffs(mask) - 1;
      mask &= mask - 1;
      const PacketSlot x = sl[i + b];
      const int f = (i + b) / spf, u = pkt_useful(x.hdr);
      const uint8_t * src = sub.src + (long long)f * fb + x.pos + 3;
      for (int j = lane; j < u; j += 32) dst[at + j] = src[j];
      at += u;
    }
  }
  __syncwarp();
  if (lane) return;
  const DgInfo d = dg_parse(dst, g.bytes, s.dg_flag != 0);
  DgRec & r = out_rec[k];
  r.first_frame = g.start / spf; r.last_frame = g.end / spf; r.n_packets = g.n_packets; r.status = d.status;
  r.extension_flag = d.ext_flag; r.crc_flag = d.crc_flag; r.segment_flag = d.seg_flag; r.user_access_flag = d.ua_flag;
  r.type = d.type; r.continuity = d.cont; r.repetition = d.rep; r.extension = d.extension;
  r.segment_last = d.seg_last; r.segment_number = d.seg_num; r.transport_id = d.tid; r.length_indicator = d.li;
  r.crc_stored = d.crc_stored; r.crc_computed = d.crc_computed; r.length = g.bytes; r.data_start = d.data_start; r.data_length = d.data_len; r.reserved = 0;
  r.offset = g.off;
}
} // namespace

cudaError_t launch_packet_scan(cudaStream_t s, const PacketSub * sub, int n_subs, long long n_frames, PacketSlot * slots, unsigned long long * lc)
{
  if (n_frames <= 0) return cudaSuccess;
  k_packet_scan<<<(unsigned)((n_frames + 127) / 128), 128, 0, s>>>(sub, n_subs, n_frames, slots);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

cudaError_t launch_packet_walk(cudaStream_t s, const PacketSub * sub, const PacketStream * st, int n_streams, const PacketSlot * slots, PacketStage * stage,
                               PacketCount * cnt, unsigned long long * lc)
{
  if (n_streams <= 0) return cudaSuccess;
  k_packet_walk<<<n_streams, PACKET_WALK_THREADS, 0, s>>>(sub, st, slots, stage, cnt);
  if (lc) (*lc)++;
  return cudaGetLastError();
}

cudaError_t launch_packet_compact(cudaStream_t s, const PacketSub * sub, const PacketStream * st, int n_streams, long long n_out, const PacketSlot * slots,
                                  const PacketStage * stage, DgRec * out_rec, uint8_t * out_pay, unsigned long long * lc)
{
  if (n_out <= 0) return cudaSuccess;
  k_packet_compact<<<(unsigned)((n_out + PACKET_COMPACT_WARPS - 1) / PACKET_COMPACT_WARPS), 32 * PACKET_COMPACT_WARPS, 0, s>>>(sub, st, n_streams, n_out, slots, stage,
                                                                                                                               out_rec, out_pay);
  if (lc) (*lc)++;
  return cudaGetLastError();
}
} // namespace dab
