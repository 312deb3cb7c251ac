// dabstar_facade.hpp — C++ host facades over the C ABI (include/dabstar_b200.h) that keep the reference's class
// names and call shapes, so DABstar's headless callers can switch the GPU path in for the CPU one.
//
//   reference class (file:line under /root/reference/src)            facade here
//   FreqInterleaver::map_k_to_fft_bin   ofdm/freq_interleaver.h:50    dabstar::FreqInterleaver
//   PhaseReference                       ofdm/phasereference.h:53-58   dabstar::PhaseReference
//   ViterbiSpiral::deconvolve            viterbi_spiral.h:20           dabstar::ViterbiSpiral      (same signature)
//   Protection::deconvolve               protection/protection.h:44    dabstar::Protection         (same signature)
//   FicDecoder (mFicHandler)             decoder/fic_decoder.h:49-58   dabstar::FicDecoder         (same signature)
//   Backend::process                     backend/backend.h:60          dabstar::Backend            (same signature)
//   OfdmDecoder                          ofdm/ofdm_decoder.h:63-73     dabstar::OfdmDecoder        (frame granular)
//   DabProcessor                         main/dab_processor.h:71       dabstar::DabProcessor       (whole recordings)
//
// The per-call facades (ViterbiSpiral, Protection, FicDecoder, Backend) launch a batch of one: they exist for drop-in
// compatibility and for tests; throughput comes from the batch entry points (DabProcessor, *_batch methods).
// Errors: the ABI's negative codes are turned into std::runtime_error carrying dabstar_last_error().
#pragma once
#include "../../include/dabstar_b200.h"

#include <array>
#include <complex>
#include <cstdint>
#include <cstring>
#include <functional>
#include <stdexcept>
#include <string>
#include <vector>

namespace dabstar
{
using i16 = int16_t;
using i32 = int32_t;
using u8 = uint8_t;
using u16 = uint16_t;
using f32 = float;
using cf32 = std::complex<float>;

class Context
{
public:
  explicit Context(int device = 0, void * cudaStream = nullptr)
  {
    if (dabstar_create(&mCtx, device, cudaStream) != DABSTAR_OK) throw std::runtime_error("dabstar_create: no usable CUDA device (no CPU fallback)");
  }
  ~Context() { dabstar_destroy(mCtx); }
  Context(const Context &) = delete;
  Context & operator=(const Context &) = delete;
  dabstar_ctx * get() const { return mCtx; }
  int check(int rc, const char * what) const
  {
    if (rc < 0) throw std::runtime_error(std::string(what) + ": " + dabstar_last_error(mCtx));
    return rc;
  }

private:
  dabstar_ctx * mCtx = nullptr;
};

class FreqInterleaver
{
public:
  explicit FreqInterleaver(Context & c) { c.check(dabstar_freq_interleaver(c.get(), mTable.data()), "dabstar_freq_interleaver"); }
  i16 map_k_to_fft_bin(const i16 k) const { return mTable[k]; }

private:
  std::array<i16, DABSTAR_K> mTable{};
};

class PhaseReference
{
public:
  static constexpr i32 IDX_NOT_FOUND = 100000;
  explicit PhaseReference(Context & c) : mC(c) { c.check(dabstar_phase_table(c.get(), reinterpret_cast<float *>(mRefTable.data())), "dabstar_phase_table"); }
  void set_sync_on_strongest_peak(bool s) { mStrongest = s; }
  // iV: at least 2048 samples (TArrayTn in the reference)
  i32 correlate_with_phase_ref_and_find_max_peak(const cf32 * iV, const f32 iThreshold)
  {
    i32 r = -1;
    mC.check(dabstar_prs_correlate(mC.get(), reinterpret_cast<const float *>(iV), 1, iThreshold, mStrongest ? 1 : 0, &r, DABSTAR_MEM_HOST), "dabstar_prs_correlate");
    return r;
  }
  i32 estimate_carrier_offset_from_sync_symbol_0(const cf32 * iFft)
  {
    i32 r = IDX_NOT_FOUND;
    mC.check(dabstar_estimate_carrier_offset(mC.get(), reinterpret_cast<const float *>(iFft), 1, &r, DABSTAR_MEM_HOST), "dabstar_estimate_carrier_offset");
    return r;
  }
  std::array<cf32, DABSTAR_TU> mRefTable{};

private:
  Context & mC;
  bool mStrongest = false;
};

class ViterbiSpiral
{
public:
  ViterbiSpiral(Context & c, const i16 iWordlength) : mC(c), mFrameBits(iWordlength) {}
  // input: 4 * (wordlength + 6) soft bits, output: wordlength bits, one per byte
  void deconvolve(const i16 * input, u8 * output)
  {
    const int64_t zero = 0;
    const int32_t n = mFrameBits;
    mC.check(dabstar_viterbi(mC.get(), input, &zero, &n, 1, output, &zero, DABSTAR_MEM_HOST), "dabstar_viterbi");
  }

private:
  Context & mC;
  const i16 mFrameBits;
};

// EepProtection / UepProtection: shortForm selects the table as BackendDeconvolver does (backend_deconvolver.cpp:32-42)
class Protection
{
public:
  Protection(Context & c, bool iShortForm, i16 iBitRate, i16 iProtLevel, i16 iCuSize) : mC(c), mShort(iShortForm), mBitRate(iBitRate), mLevel(iProtLevel), mCuSize(iCuSize) {}
  bool deconvolve(const i16 * iV, i32 /*iSize*/, u8 * oOut)
  {
    mC.check(dabstar_protection_deconvolve(mC.get(), mShort ? 1 : 0, mBitRate, mLevel, mCuSize, iV, 1, oOut, DABSTAR_MEM_HOST), "dabstar_protection_deconvolve");
    return true;
  }

private:
  Context & mC;
  bool mShort;
  i16 mBitRate, mLevel, mCuSize;
};

// Consumer of CRC-good FIBs: IFibDecoder::process_FIB (decoder/fib_decoder_if.h:81)
using FibSink = std::function<void(const std::array<u8, 256> &, u16 ficIdx)>;

class FicDecoder
{
public:
  explicit FicDecoder(Context & c, FibSink sink = nullptr) : mC(c), mSink(std::move(sink)) { mSoft.resize(3 * DABSTAR_SYM_BITS); }
  void restart() { mRatio = 0; mRunning = true; }
  void stop() { mRunning = false; }
  // symbols 1..3 of a frame; the four FICs are decoded when the third symbol has arrived
  void process_block(const std::vector<i16> & iOfdmSoftBits, const i32 iOfdmSymbIdx)
  {
    if (iOfdmSymbIdx < 1 || iOfdmSymbIdx > 3 || iOfdmSoftBits.size() != DABSTAR_SYM_BITS) throw std::invalid_argument("FicDecoder::process_block");
    memcpy(&mSoft[(size_t)(iOfdmSymbIdx - 1) * DABSTAR_SYM_BITS], iOfdmSoftBits.data(), sizeof(i16) * DABSTAR_SYM_BITS);
    if (iOfdmSymbIdx != 3 || !mRunning) return;
    u8 crc[12];
    i32 ber[8];
    mC.check(dabstar_fic_decode(mC.get(), mSoft.data(), 3 * DABSTAR_SYM_BITS, 1, mFibBits.data(), crc, ber, DABSTAR_MEM_HOST), "dabstar_fic_decode");
    for (int fic = 0; fic < 4; fic++)
    {
      mFicValid[fic] = true;
      for (int fib = 0; fib < 3; fib++)
      {
        if (crc[3 * fic + fib])
        {
          if (mSink)
          {
            std::array<u8, 256> one;
            memcpy(one.data(), &mFibBits[fic * 768 + fib * 256], 256);
            mSink(one, (u16)fic);
          }
          if (mRatio < 10) mRatio++;
        }
        else
        {
          mFicValid[fic] = false;
          if (mRatio > 0) mRatio--;
        }
      }
    }
  }
  void get_fib_bits(u8 * v, bool * b) const
  {
    memcpy(v, mFibBits.data(), mFibBits.size());
    for (int i = 0; i < 4; i++) b[i] = mFicValid[i];
  }
  i32 get_fic_decode_ratio_percent() const { return mRatio * 10; }

private:
  Context & mC;
  FibSink mSink;
  std::vector<i16> mSoft;
  std::array<u8, 4 * 768> mFibBits{};
  std::array<bool, 4> mFicValid{};
  i32 mRatio = 0;
  bool mRunning = true;
};

// FrameProcessor::add_to_frame (backend/frame_processor.h:43)
using FrameSink = std::function<void(const std::vector<u8> &)>;

class Backend
{
public:
  Backend(Context & c, const dabstar_subch & d, FrameSink sink) : mC(c), mD(d), mSink(std::move(sink)), mOut((size_t)24 * d.bit_rate) {}
  // one CIF fragment (CuSize * 64 soft bits). Keeps the last 17 fragments on the host and runs them as one batch
  // per emitted logical frame; use DabProcessor for throughput.
  i32 process(const i16 * iV, const i32 cnt)
  {
    if (cnt != mD.size_cu * 64) throw std::invalid_argument("Backend::process");
    mHist.emplace_back(iV, iV + cnt);
    if (mHist.size() > 17) mHist.erase(mHist.begin());
    mSeen++;
    if (mSeen < 17) return 1;
    std::vector<i16> cifs((size_t)17 * DABSTAR_CIF_BITS, 0);
    for (size_t g = 0; g < 17; g++) memcpy(&cifs[g * DABSTAR_CIF_BITS + (size_t)mD.start_cu * 64], mHist[g].data(), sizeof(i16) * (size_t)cnt);
    mC.check(dabstar_backend_process(mC.get(), &mD, cifs.data(), 17, mOut.data(), DABSTAR_MEM_HOST), "dabstar_backend_process");
    if (mSink) mSink(mOut);
    return 1;
  }

private:
  Context & mC;
  dabstar_subch mD;
  FrameSink mSink;
  std::vector<u8> mOut;
  std::vector<std::vector<i16>> mHist;
  long mSeen = 0;
};

// Packet-mode data groups of one address of one packet-mode sub-channel: packets CRC-checked, groups assembled and (DG flag 0)
// their MSC data group headers and CRCs checked on the device (dabstar_packet_groups). Batch granular; MOT, EPG and the other
// data-service decoders stay CPU consumers of the groups handed to the sink.
class PacketProcessor
{
public:
  using GroupSink = std::function<void(const u8 * group, int len, const dabstar_data_group & rec)>;
  PacketProcessor(Context & c, int bitRate, int address, int dgFlag = 0, GroupSink sink = nullptr)
    : mC(c), mBitRate(bitRate), mAddress(address), mDgFlag(dgFlag), mSink(std::move(sink)) {}
  // iBits: nFrames x 24*bitRate bytes (one bit each). Returns one record per data group.
  std::vector<dabstar_data_group> add_frames(const u8 * iBits, int nFrames)
  {
    std::vector<dabstar_data_group> rec((size_t)std::max(nFrames * (mBitRate / 8), 1));
    std::vector<u8> pay((size_t)std::max(nFrames, 1) * 3 * (size_t)mBitRate);
    const int n = mC.check(dabstar_packet_groups(mC.get(), iBits, mBitRate, nFrames, mAddress, mDgFlag, rec.data(), (int)rec.size(), pay.data(), DABSTAR_MEM_HOST),
                           "dabstar_packet_groups");
    rec.resize((size_t)n);
    if (mSink) deliver(rec, pay.data(), mSink);
    return rec;
  }
  static void deliver(const std::vector<dabstar_data_group> & rec, const u8 * payload, const GroupSink & sink)
  {
    for (const auto & r : rec) sink(payload + r.offset, r.length, r);
  }

private:
  Context & mC;
  int mBitRate, mAddress, mDgFlag;
  GroupSink mSink;
};

// MPEG layer II audio frames of one DAB (MP2) sub-channel: header and CRC-16 of every audio-frame slot, on the device
// (dabstar_mp2_frames). Batch granular; an MP2 decoder stays a CPU consumer of the OK frames handed to the sink.
class Mp2Processor
{
public:
  using FrameSink = std::function<void(const u8 * frame, int len, const dabstar_mp2_frame & rec)>;
  Mp2Processor(Context & c, int bitRate, FrameSink sink = nullptr) : mC(c), mBitRate(bitRate), mSink(std::move(sink)) {}
  // iBits: nFrames x 24*bitRate bytes (one bit each). Returns one record per audio-frame slot.
  std::vector<dabstar_mp2_frame> add_frames(const u8 * iBits, int nFrames)
  {
    std::vector<dabstar_mp2_frame> rec((size_t)std::max(nFrames, 1));
    std::vector<u8> pay(rec.size() * 3 * (size_t)mBitRate);
    const int n = mC.check(dabstar_mp2_frames(mC.get(), iBits, mBitRate, nFrames, rec.data(), (int)rec.size(), pay.data(), DABSTAR_MEM_HOST), "dabstar_mp2_frames");
    rec.resize((size_t)n);
    if (mSink) deliver(rec, pay.data(), mBitRate, mSink);
    return rec;
  }
  // the OK frames of records, whose bytes follow one another in payload
  static void deliver(const std::vector<dabstar_mp2_frame> & rec, const u8 * payload, int bitRate, const FrameSink & sink)
  {
    size_t o = 0;
    for (const auto & r : rec)
      if (r.status == 0)
      {
        const int len = 3 * bitRate * r.n_frames;
        sink(payload + o, len, r);
        o += (size_t)len;
      }
  }

private:
  Context & mC;
  int mBitRate;
  FrameSink mSink;
};

// backend/audio/mp4processor.h: the DAB+ outer code of one sub-channel (super-frame sync, RS(120,110), Fire code, AU CRCs).
// Batch granular: add_frames takes a run of FrameProcessor::add_to_frame payloads; the AAC decoder stays a CPU consumer.
class Mp4Processor
{
public:
  using AuSink = std::function<void(const u8 * au, int len, const dabstar_superframe & sf)>;
  Mp4Processor(Context & c, int bitRate, AuSink sink = nullptr) : mC(c), mBitRate(bitRate), mSink(std::move(sink)) {}
  // iBits: nFrames x 24*bitRate bytes (one bit each). Returns the super-frames the processor attempted.
  std::vector<dabstar_superframe> add_frames(const u8 * iBits, int nFrames)
  {
    std::vector<dabstar_superframe> rec((size_t)std::max(nFrames, 1));
    const size_t sf = (size_t)110 * (mBitRate / 8);
    std::vector<u8> pay(rec.size() * sf);
    const int n = mC.check(dabstar_dabplus_decode(mC.get(), iBits, mBitRate, nFrames, rec.data(), (int)rec.size(), pay.data(), DABSTAR_MEM_HOST), "dabstar_dabplus_decode");
    rec.resize((size_t)n);
    if (mSink)
      for (int i = 0; i < n; i++)
        if (rec[i].ok)
          for (int u = 0; u < rec[i].num_aus; u++)
            if (rec[i].au_state[u] == 1) mSink(&pay[(size_t)i * sf + rec[i].au_start[u]], rec[i].au_start[u + 1] - rec[i].au_start[u] - 2, rec[i]);
    return rec;
  }

private:
  Context & mC;
  int mBitRate;
  AuSink mSink;
};

enum class ESoftBitType { SOFTDEC1 = 0, SOFTDEC2 = 1, SOFTDEC3 = 2 };

// What XmlFileReader / WavFileHandler / RawFileHandler + their reader threads produce from a recording file: the header
// is inspected on the host (dabstar_file_probe), the samples are converted and brought to 2.048 MS/s on the GPU.
// Returns interleaved re / im floats.
inline std::vector<float> read_recording(Context & c, const u8 * file, size_t fileBytes, dabstar_file_info * oInfo = nullptr)
{
  dabstar_file_info fi{};
  if (dabstar_file_probe(file, (int64_t)fileBytes, (int64_t)fileBytes, &fi) != DABSTAR_OK) throw std::runtime_error("dabstar_file_probe: unsupported recording header");
  if (oInfo) *oInfo = fi;
  std::vector<float> x((size_t)std::max<int64_t>(fi.n_samples, 1) * 2);
  c.check(dabstar_ingest_convert(c.get(), file + fi.data_offset, &fi.fmt, fi.n_samples, x.data(), DABSTAR_MEM_HOST), "dabstar_ingest_convert");
  x.resize((size_t)fi.n_samples * 2);
  if (fi.sample_rate == 2048000) return x;
  const int64_t n = dabstar_resample_count(fi.n_samples, fi.sample_rate, fi.reader);
  if (n < 0) throw std::runtime_error("dabstar_resample_count: unsupported sample rate");
  std::vector<float> y((size_t)std::max<int64_t>(n, 1) * 2);
  const int64_t got = dabstar_resample_linear(c.get(), x.data(), fi.n_samples, fi.sample_rate, fi.reader, y.data(), n, DABSTAR_MEM_HOST);
  c.check((int)std::min<int64_t>(got, 0), "dabstar_resample_linear");
  y.resize((size_t)got * 2);
  return y;
}

// OfdmDecoder::SLcdData (ofdm/ofdm_decoder.h:53-61) plus the two state scalars it is computed from
struct SLcdData
{
  f32 MER, SNR, MeanValue, MeanPowerOvrAll, NoisePower, MeanSigmaSqFreqCorr;
};

// ofdm/tii_detector.h:30-45 for nDetectors recordings at once (STiiResult = dabstar_tii_result).
class TiiDetector
{
public:
  explicit TiiDetector(Context & c, int nDetectors = 1) : mC(c), mN(nDetectors) { c.check(dabstar_tii_create(c.get(), nDetectors, &mT), "dabstar_tii_create"); }
  ~TiiDetector() { dabstar_tii_destroy(mT); }
  TiiDetector(const TiiDetector &) = delete;
  TiiDetector & operator=(const TiiDetector &) = delete;
  void reset() { mC.check(dabstar_tii_reset(mT), "dabstar_tii_reset"); }
  void set_detect_collisions(bool b) { mColl = b; mC.check(dabstar_tii_set_collisions(mT, mColl ? 1 : 0, mSubId), "dabstar_tii_set_collisions"); }
  void set_subid_for_collision_search(u8 subId) { mSubId = subId; mC.check(dabstar_tii_set_collisions(mT, mColl ? 1 : 0, mSubId), "dabstar_tii_set_collisions"); }
  // iV: nDetectors x nSymbols x 2048 null-symbol spectra in fft order (the reference adds one spectrum per call)
  void add_to_tii_buffer(const cf32 * iV, int nSymbols = 1) { mC.check(dabstar_tii_add(mT, reinterpret_cast<const float *>(iV), nSymbols, DABSTAR_MEM_HOST), "dabstar_tii_add"); }
  // per detector: the transmitters found, strongest first
  std::vector<std::vector<dabstar_tii_result>> process_tii_data(i16 iThreshold_db)
  {
    constexpr int cap = 128;
    std::vector<dabstar_tii_result> buf((size_t)mN * cap);
    std::vector<int32_t> cnt((size_t)mN);
    mC.check(dabstar_tii_process(mT, iThreshold_db, buf.data(), cap, cnt.data()), "dabstar_tii_process");
    std::vector<std::vector<dabstar_tii_result>> out((size_t)mN);
    for (int d = 0; d < mN; d++) out[d].assign(buf.begin() + (size_t)d * cap, buf.begin() + (size_t)d * cap + std::min(cnt[d], cap));
    return out;
  }

private:
  Context & mC;
  int mN;
  dabstar_tii * mT = nullptr;
  bool mColl = false;
  u8 mSubId = 0;
};

// Frame granular: one call = store_reference_symbol_0 + 75 x decode_symbol + store_null_symbol_without_tii.
class OfdmDecoder
{
public:
  explicit OfdmDecoder(Context & c) : mC(c) { c.check(dabstar_ofdm_state_create(c.get(), &mSt), "dabstar_ofdm_state_create"); }
  ~OfdmDecoder() { dabstar_ofdm_state_destroy(mC.get(), mSt); }
  void reset() { mC.check(dabstar_ofdm_state_reset(mC.get(), mSt), "dabstar_ofdm_state_reset"); }
  void set_soft_bit_gen_type(ESoftBitType t) { mType = t; }
  // iFft: nFrames x 77 x 2048 spectra; oBits: nFrames x 75 x 3072; oQuality (optional): nFrames x SLcdData, lcd_data() after
  // each frame's null symbol
  void decode_frames(const cf32 * iFft, int nFrames, const f32 * iClockErr, const u8 * iNullIsTii, i16 * oBits, SLcdData * oQuality = nullptr)
  {
    static_assert(sizeof(SLcdData) == 6 * sizeof(float), "SLcdData is the 6-float record of the C ABI");
    if (oQuality)
      mC.check(dabstar_ofdm_decode_frames_quality(mC.get(), mSt, reinterpret_cast<const float *>(iFft), nFrames, iClockErr, iNullIsTii, (int)mType, oBits,
                                                  DABSTAR_MEM_HOST, reinterpret_cast<float *>(oQuality)),
               "dabstar_ofdm_decode_frames_quality");
    else
      mC.check(dabstar_ofdm_decode_frames(mC.get(), mSt, reinterpret_cast<const float *>(iFft), nFrames, iClockErr, iNullIsTii, (int)mType, oBits, DABSTAR_MEM_HOST),
               "dabstar_ofdm_decode_frames");
  }
  SLcdData lcd_data() const // what signal_show_lcd_data would carry now
  {
    float q[6];
    mC.check(dabstar_ofdm_state_quality(mC.get(), mSt, q), "dabstar_ofdm_state_quality");
    return SLcdData{ q[0], q[1], q[2], q[3], q[4], q[5] };
  }

private:
  Context & mC;
  dabstar_ofdm_state * mSt = nullptr;
  ESoftBitType mType = ESoftBitType::SOFTDEC1;
};

// Whole recordings: DabProcessor::run() for n recordings in lock step.
class DabProcessor
{
public:
  DabProcessor(Context & c, int nRecordings, int inputFormat = DABSTAR_FMT_U8, bool scanMode = false, ESoftBitType t = ESoftBitType::SOFTDEC1)
    : mC(c), mN(nRecordings)
  {
    dabstar_decoder_cfg cfg{};
    cfg.input_format = inputFormat;
    cfg.soft_bit_type = (int)t;
    cfg.sync_threshold = 3.0f; // dabradio.cpp:92
    cfg.scan_mode = scanMode ? 1 : 0;
    c.check(dabstar_decoder_create(c.get(), &cfg, nRecordings, &mDec), "dabstar_decoder_create");
  }
  ~DabProcessor() { dabstar_decoder_destroy(mDec); }
  void set_audio_channel(int recording, const std::vector<dabstar_subch> & sc)
  {
    mC.check(dabstar_decoder_set_subchannels(mDec, recording, sc.data(), (int)sc.size()), "dabstar_decoder_set_subchannels");
  }
  // iq[r]: nSamples[r] interleaved IQ pairs in the configured format, host memory
  void run(const std::vector<const void *> & iq, const std::vector<int64_t> & nSamples)
  {
    mC.check(dabstar_decoder_run(mDec, iq.data(), nSamples.data(), DABSTAR_MEM_HOST), "dabstar_decoder_run");
  }
  // Recordings in any file sample format (XmlReader::readElements_*, xml_reader.cpp:254-800): layouts the FFT kernel does not read
  // natively are converted to complex float on the device first; the processor must have been created with DABSTAR_FMT_CF32.
  void run_files(const std::vector<const void *> & raw, const std::vector<int64_t> & nSamples, const dabstar_sample_format & fmt)
  {
    std::vector<std::vector<float>> conv(raw.size());
    std::vector<const void *> ptrs(raw.size());
    for (size_t r = 0; r < raw.size(); r++)
    {
      conv[r].resize((size_t)2 * (size_t)nSamples[r]);
      mC.check(dabstar_ingest_convert(mC.get(), raw[r], &fmt, nSamples[r], conv[r].data(), DABSTAR_MEM_HOST), "dabstar_ingest_convert");
      ptrs[r] = conv[r].data();
    }
    run(ptrs, nSamples);
  }
  // Sub-channels and CIF counter from the recording's own FIG 0/0 and 0/1 instead of set_audio_channel.
  // tiiNullSymbols: null symbols whose CIF counter has (count & 7) >= 4 leave the null power alone, as with a real FIB decoder (second pass)
  void set_auto_config(int recording, bool on = true, bool tiiNullSymbols = false)
  {
    mC.check(dabstar_decoder_set_auto_config(mDec, recording, on ? (tiiNullSymbols ? 2 : 1) : 0), "dabstar_decoder_set_auto_config");
  }
  std::vector<dabstar_subch> sub_channels(int recording) const
  {
    std::vector<dabstar_subch> v((size_t)std::max(0, dabstar_decoder_subchannels(mDec, recording, nullptr, 0)));
    if (!v.empty()) dabstar_decoder_subchannels(mDec, recording, v.data(), (int)v.size());
    return v;
  }
  // DabProcessor::start_eti_generator / stop_eti_generator (dab_processor.cpp:529-558): the next run also frames ETI(NI)
  void start_eti_generator(int recording, int cifCountHi = 0, int cifCountLo = 0)
  {
    mC.check(dabstar_decoder_enable_eti(mDec, recording, 1, cifCountHi, cifCountLo), "dabstar_decoder_enable_eti");
  }
  void stop_eti_generator(int recording) { mC.check(dabstar_decoder_enable_eti(mDec, recording, 0, 0, 0), "dabstar_decoder_enable_eti"); }
  // Mp4Processor behind the sub-channel's Backend (backend_driver.cpp:38-59) in the next runs, on the device; subChId -1: every
  // sub-channel the recording's own FIG 0/2 lists as DAB+ (needs set_auto_config)
  void set_dabplus(int recording, int subChId = -1, bool on = true)
  {
    mC.check(dabstar_decoder_set_dabplus(mDec, recording, subChId, on ? 1 : 0), "dabstar_decoder_set_dabplus");
  }
  bool dabplus_decoded(int recording, int subChId) const { return dabstar_decoder_superframes(mDec, recording, subChId, nullptr, 0) >= 0; }
  // the super-frames Mp4Processor attempted in the last run; every CRC-good access unit of an accepted one goes to sink, in order
  std::vector<dabstar_superframe> superframes(int recording, int subChId, const Mp4Processor::AuSink & sink = nullptr) const
  {
    const int n = mC.check(dabstar_decoder_superframes(mDec, recording, subChId, nullptr, 0), "dabstar_decoder_superframes");
    std::vector<dabstar_superframe> rec((size_t)n);
    if (n > 0) dabstar_decoder_superframes(mDec, recording, subChId, rec.data(), n);
    if (sink && n > 0)
    {
      std::vector<u8> pay((size_t)dabstar_decoder_superframe_payload(mDec, recording, subChId, nullptr, 0));
      dabstar_decoder_superframe_payload(mDec, recording, subChId, pay.data(), (int64_t)pay.size());
      const size_t sf = pay.size() / (size_t)n;
      for (int i = 0; i < n; i++)
        if (rec[i].ok)
          for (int u = 0; u < rec[i].num_aus; u++)
            if (rec[i].au_state[u] == 1) sink(&pay[(size_t)i * sf + rec[i].au_start[u]], rec[i].au_start[u + 1] - rec[i].au_start[u] - 2, rec[i]);
    }
    return rec;
  }
  // MPEG layer II audio frames of the sub-channel in the next runs, on the device; subChId -1: every sub-channel the recording's
  // own FIG 0/2 lists as MPEG layer II (needs set_auto_config)
  void set_mp2(int recording, int subChId = -1, bool on = true)
  {
    mC.check(dabstar_decoder_set_mp2(mDec, recording, subChId, on ? 1 : 0), "dabstar_decoder_set_mp2");
  }
  bool mp2_decoded(int recording, int subChId) const { return dabstar_decoder_mp2_frames(mDec, recording, subChId, nullptr, 0) >= 0; }
  // the last run's audio-frame slots; every OK frame goes to sink, in order
  std::vector<dabstar_mp2_frame> mp2_frames(int recording, int subChId, const Mp2Processor::FrameSink & sink = nullptr) const
  {
    const int n = mC.check(dabstar_decoder_mp2_frames(mDec, recording, subChId, nullptr, 0), "dabstar_decoder_mp2_frames");
    std::vector<dabstar_mp2_frame> rec((size_t)n);
    if (n > 0) dabstar_decoder_mp2_frames(mDec, recording, subChId, rec.data(), n);
    if (sink && n > 0)
    {
      std::vector<u8> pay((size_t)dabstar_decoder_mp2_payload(mDec, recording, subChId, nullptr, 0));
      dabstar_decoder_mp2_payload(mDec, recording, subChId, pay.data(), (int64_t)pay.size());
      int bitRate = 0;
      for (const auto & s : sub_channels(recording)) if (s.sub_ch_id == subChId) bitRate = s.bit_rate;
      if (bitRate <= 0) throw std::runtime_error("mp2_frames: sub-channel " + std::to_string(subChId) + " is not in the recording's sub-channel list");
      Mp2Processor::deliver(rec, pay.data(), bitRate, sink);
    }
    return rec;
  }
  // packet-mode data groups of (sub-channel, address) in the next runs, on the device; subChId -1: every packet-mode component of
  // the recording's own FIG 0/2 and 0/3 (needs set_auto_config; address ignored)
  void set_packet(int recording, int subChId = -1, int address = 0, bool on = true)
  {
    mC.check(dabstar_decoder_set_packet(mDec, recording, subChId, address, on ? 1 : 0), "dabstar_decoder_set_packet");
  }
  // packet-mode FEC in front of the packet pass: subChId forces it on; -1 every sub-channel the recording's FIG 0/14 flags
  void set_packet_fec(int recording, int subChId = -1, bool on = true)
  {
    mC.check(dabstar_decoder_set_packet_fec(mDec, recording, subChId, on ? 1 : 0), "dabstar_decoder_set_packet_fec");
  }
  bool packet_decoded(int recording, int subChId, int address) const { return dabstar_decoder_data_groups(mDec, recording, subChId, address, nullptr, 0) >= 0; }
  // the last run's data groups of the stream; every group goes to sink, in order
  std::vector<dabstar_data_group> data_groups(int recording, int subChId, int address, const PacketProcessor::GroupSink & sink = nullptr) const
  {
    const int n = mC.check(dabstar_decoder_data_groups(mDec, recording, subChId, address, nullptr, 0), "dabstar_decoder_data_groups");
    std::vector<dabstar_data_group> rec((size_t)n);
    if (n > 0) dabstar_decoder_data_groups(mDec, recording, subChId, address, rec.data(), n);
    if (sink && n > 0)
    {
      std::vector<u8> pay((size_t)dabstar_decoder_data_group_payload(mDec, recording, subChId, address, nullptr, 0));
      dabstar_decoder_data_group_payload(mDec, recording, subChId, address, pay.data(), (int64_t)pay.size());
      PacketProcessor::deliver(rec, pay.data(), sink);
    }
    return rec;
  }
  dabstar_packet_stats packet_stats(int recording, int subChId, int address) const
  {
    dabstar_packet_stats st{};
    mC.check(dabstar_decoder_packet_stats(mDec, recording, subChId, address, &st), "dabstar_decoder_packet_stats");
    return st;
  }
  bool fec_decoded(int recording, int subChId) const { return dabstar_decoder_fec_frames(mDec, recording, subChId, nullptr, 0) >= 0; }
  // the last run's FEC frame records of a sub-channel with packet-mode FEC
  std::vector<dabstar_fec_frame> fec_frames(int recording, int subChId) const
  {
    std::vector<dabstar_fec_frame> v((size_t)mC.check(dabstar_decoder_fec_frames(mDec, recording, subChId, nullptr, 0), "dabstar_decoder_fec_frames"));
    if (!v.empty()) dabstar_decoder_fec_frames(mDec, recording, subChId, v.data(), (int)v.size());
    return v;
  }
  // FIG 0/3 packet-mode components of a self-configured recording after the last run
  std::vector<dabstar_packet_comp> packet_components(int recording) const
  {
    std::vector<dabstar_packet_comp> v((size_t)mC.check(dabstar_decoder_packet_components(mDec, recording, nullptr, 0), "dabstar_decoder_packet_components"));
    if (!v.empty()) dabstar_decoder_packet_components(mDec, recording, v.data(), (int)v.size());
    return v;
  }
  // FIG 0/2 service components of a self-configured recording after the last run
  std::vector<dabstar_service_comp> components(int recording) const
  {
    std::vector<dabstar_service_comp> v((size_t)mC.check(dabstar_decoder_components(mDec, recording, nullptr, 0), "dabstar_decoder_components"));
    if (!v.empty()) dabstar_decoder_components(mDec, recording, v.data(), (int)v.size());
    return v;
  }
  std::vector<u8> eti(int recording) const
  {
    std::vector<u8> v((size_t)std::max<int64_t>(0, dabstar_decoder_eti_size(mDec, recording)));
    if (!v.empty()) dabstar_decoder_eti_copy(mDec, recording, v.data(), (int64_t)v.size());
    return v;
  }
  int n_frames(int recording) const { return dabstar_decoder_n_frames(mDec, recording); }
  // DabProcessor::set_tii_processing / set_tii_threshold / set_tii_collisions / set_tii_sub_id (+ ProcessParams::tiiFramesToCount);
  // needs set_auto_config: the recording's own CIF counter decides which null symbols carry TII
  void set_tii_processing(int recording, bool on, int framesToCount = 5, int thresholdDb = 8, bool collisions = false, int subId = 0)
  {
    mC.check(dabstar_decoder_enable_tii(mDec, recording, on ? 1 : 0, framesToCount, thresholdDb, collisions ? 1 : 0, subId), "dabstar_decoder_enable_tii");
  }
  struct TiiEvent { int frame; std::vector<dabstar_tii_result> transmitterIds; };
  std::vector<TiiEvent> tii_events(int recording) const // what signal_show_tii would have carried, one entry per search
  {
    std::vector<TiiEvent> ev((size_t)std::max(0, dabstar_decoder_tii_events(mDec, recording)));
    for (size_t e = 0; e < ev.size(); e++)
    {
      int32_t frame = 0;
      ev[e].transmitterIds.resize(128);
      const int n = dabstar_decoder_tii_results(mDec, recording, (int)e, ev[e].transmitterIds.data(), 128, &frame);
      ev[e].transmitterIds.resize((size_t)std::max(0, std::min(n, 128)));
      ev[e].frame = frame;
    }
    return ev;
  }
  SLcdData lcd_data(int recording) const // the recording's OfdmDecoder figures at the end of the run
  {
    float q[6];
    mC.check(dabstar_decoder_quality(mDec, recording, q), "dabstar_decoder_quality");
    return SLcdData{ q[0], q[1], q[2], q[3], q[4], q[5] };
  }
  // Capture lcd_data() for every frame of the next runs (frame_lcd_data); off by default.
  void set_frame_quality(bool on) { mC.check(dabstar_decoder_set_frame_quality(mDec, on ? 1 : 0), "dabstar_decoder_set_frame_quality"); }
  // One SLcdData per frame of frame_info(): the figures as they stood after that frame's null symbol (the last run must have
  // captured them). Replaying slot_show_lcd_data from these needs no per-symbol callback.
  std::vector<SLcdData> frame_lcd_data(int recording) const
  {
    std::vector<SLcdData> v((size_t)std::max(0, n_frames(recording)));
    mC.check(dabstar_decoder_frame_quality(mDec, recording, reinterpret_cast<float *>(v.data()), (int)v.size()), "dabstar_decoder_frame_quality");
    return v;
  }
  std::vector<dabstar_frame_info> frame_info(int recording) const
  {
    std::vector<dabstar_frame_info> v((size_t)std::max(0, n_frames(recording)));
    if (!v.empty()) dabstar_decoder_frame_info(mDec, recording, v.data(), (int)v.size());
    return v;
  }
  // Delivers the decoded FIBs (CRC-good only, as FicDecoder does) and MSC logical frames in stream order.
  void deliver(int recording, const FibSink & fibSink, const std::function<void(int subChId, const std::vector<u8> &)> & mscSink,
               const std::vector<dabstar_subch> & sc) const
  {
    const int nf = n_frames(recording);
    std::vector<u8> bits((size_t)nf * 3072), valid((size_t)nf * 4);
    dabstar_decoder_fib_bits(mDec, recording, bits.data(), valid.data());
    if (fibSink)
      for (int f = 0; f < nf; f++)
        for (int fic = 0; fic < 4; fic++)
          if (valid[(size_t)4 * f + fic])
            for (int fib = 0; fib < 3; fib++)
            {
              std::array<u8, 256> one;
              memcpy(one.data(), &bits[(size_t)f * 3072 + fic * 768 + fib * 256], 256);
              fibSink(one, (u16)fic);
            }
    if (mscSink)
      for (const auto & s : sc)
      {
        const int64_t n = dabstar_decoder_msc_size(mDec, recording, s.sub_ch_id);
        std::vector<u8> all((size_t)n);
        dabstar_decoder_msc_copy(mDec, recording, s.sub_ch_id, all.data(), n);
        const size_t fb = (size_t)24 * s.bit_rate;
        for (size_t o = 0; o + fb <= all.size(); o += fb) mscSink(s.sub_ch_id, std::vector<u8>(all.begin() + o, all.begin() + o + fb));
      }
  }
  double last_ms() const { return dabstar_decoder_last_ms(mDec); }
  dabstar_decoder * get() const { return mDec; }

private:
  Context & mC;
  int mN;
  dabstar_decoder * mDec = nullptr;
};
} // namespace dabstar
