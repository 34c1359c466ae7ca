// C++ host-side mirror of the reference's decoder plug-in interface, on top of the C ABI (symgpu.h).
//
// The reference is Rust; its toolchain is not available in this environment (see INTEGRATION.md for
// the Rust adapter a maintainer would add).  This header restates the SAME interface in C++17 with
// the same names, argument meaning and error behaviour, so a C++ host can drop the GPU synthesis
// path in behind a registry exactly as a Rust host would:
//
//   AudioDecoder            symphonia-core/src/codecs/audio.rs:251-298   (reset / codec_params / decode /
//                                                                          finalize / last_decoded)
//   AudioDecoderOptions     symphonia-core/src/codecs/audio.rs:210-227   (gapless = true, verify = false)
//   CodecRegistry, Tier     symphonia-core/src/codecs/registry.rs:176-341, symphonia-core/src/common.rs:54-62
//                           (lookup order preferred -> standard -> fallback)
//   Error                   symphonia-core/src/errors.rs:43-57
//   Packet                  symphonia-core/src/packet.rs:146-170 (PacketRef)
//
// A packet handed to GpuMpaDecoder is what the reference's MpaReader emits: one whole MPEG audio frame, header word
// first (Layers I, II and III; the entropy front-ends of SURVEY.md §8f N1 run on the CPU inside decode(), the
// synthesis on the GPU).  For tests and for hosts with their own bit reader it also accepts the *parsed* Layer III
// frame -- the state the reference has at layer3/mod.rs:421 -- as bytes: symgpu_mp3_gc[2][2] (256 B) followed by
// f32 spectra [2][2][576]; the two cannot be confused, a real frame is at most 2881 bytes.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../symgpu.h"
#include "packetizer.hpp"

namespace symgpu_host {

enum class ErrorKind { None, IoError, DecodeError, SeekError, Unsupported, LimitError, ResetRequired };
struct Error {
    ErrorKind kind = ErrorKind::None;
    const char* message = ""; // static storage, like the reference's &'static str
    explicit operator bool() const { return kind != ErrorKind::None; }
};
template <typename T>
struct Result {
    T value{};
    Error error{};
    bool ok() const { return !error; }
};

inline Error map_status(symgpu_status st) { // INTEGRATION.md §3
    switch (st) {
        case SYMGPU_OK: return {};
        case SYMGPU_ERR_DECODE: return {ErrorKind::DecodeError, symgpu_strerror(st)};
        case SYMGPU_ERR_UNSUPPORTED: return {ErrorKind::Unsupported, symgpu_strerror(st)};
        case SYMGPU_ERR_LIMIT: return {ErrorKind::LimitError, symgpu_strerror(st)};
        case SYMGPU_ERR_RESET: return {ErrorKind::ResetRequired, symgpu_strerror(st)};
        default: return {ErrorKind::IoError, symgpu_strerror(st)};
    }
}

// Codec ids, symphonia-core/src/codecs/audio.rs:404-418, :462.
constexpr uint32_t CODEC_ID_VORBIS = 0x1000, CODEC_ID_MP1 = 0x1004, CODEC_ID_MP2 = 0x1005, CODEC_ID_MP3 = 0x1006, CODEC_ID_AAC = 0x1007;
constexpr uint32_t CODEC_ID_FLAC = 0x2000;

struct AudioCodecParameters {
    uint32_t codec = 0;
    uint32_t sample_rate = 0;
    uint32_t channels = 0;
    std::vector<uint8_t> extra_data;
};
struct AudioDecoderOptions {
    bool gapless = true;
    bool verify = false;
};
struct FinalizeResult {
    bool has_verify = false, verify_ok = false;
};
struct Packet { // PacketRef
    uint32_t track_id = 0;
    uint64_t pts = 0, dur = 0;
    uint32_t trim_start = 0, trim_end = 0;
    const uint8_t* data = nullptr;
    size_t len = 0;
};
// Borrow of the decoder-owned planar buffer, valid until the next call on the decoder (GenericAudioBufferRef over
// AudioBuffer<f32> or AudioBuffer<i32>, symphonia-core/src/audio/buf.rs:68-73).  `format` says which planes are set.
enum class SampleFormat { F32, S32 };
struct AudioBufferRef {
    SampleFormat format = SampleFormat::F32;
    const float* planes[8] = {};        // F32: n_planes of them, in the reference's channel order
    const int32_t* planes_s32[8] = {};  // S32 (FLAC): the same for integer samples
    size_t n_planes = 0;
    size_t frames = 0;
};

class AudioDecoder {
  public:
    virtual ~AudioDecoder() = default;
    virtual void reset() = 0;
    virtual const AudioCodecParameters& codec_params() const = 0;
    virtual Result<AudioBufferRef> decode(const Packet& packet) = 0;
    virtual FinalizeResult finalize() { return {}; }
    virtual AudioBufferRef last_decoded() const = 0;
};

enum class Tier { Preferred, Standard, Fallback };
using AudioDecoderFactory =
    std::function<Result<std::unique_ptr<AudioDecoder>>(const AudioCodecParameters&, const AudioDecoderOptions&)>;

class CodecRegistry {
  public:
    void register_audio_decoder_at_tier(Tier tier, uint32_t codec, AudioDecoderFactory factory) {
        slots_[codec][(int)tier] = std::move(factory);
    }
    // registry.rs:330-341: preferred, then standard, then fallback.
    Result<std::unique_ptr<AudioDecoder>> make_audio_decoder(const AudioCodecParameters& p, const AudioDecoderOptions& o) const {
        auto it = slots_.find(p.codec);
        if (it != slots_.end())
            for (int t = 0; t < 3; ++t)
                if (it->second[t]) return it->second[t](p, o);
        return {nullptr, {ErrorKind::Unsupported, "core (codec): unsupported codec"}};
    }

  private:
    std::map<uint32_t, AudioDecoderFactory[3]> slots_;
};

// A context shared by GPU decoders (one CUDA stream).  Stream-state slots are handed out from a free list under a mutex.
// MPEG Layer III decoders of ANY number of threads may share one context: their decode() goes through the thread-safe
// symgpu_mp3_submit / symgpu_mp3_wait pair, which gathers the packets of all threads into shared launches.  The other decoders
// (Layer I / II, AAC, Vorbis, FLAC) still want one calling thread per context (codecs/audio.rs "Send + Sync": one call at a time).
class GpuContext {
  public:
    static Result<std::shared_ptr<GpuContext>> create(int device, uint32_t max_streams) {
        symgpu_ctx* c = nullptr;
        symgpu_status st = symgpu_ctx_create(device, &c);
        if (st != SYMGPU_OK) return {nullptr, map_status(st)};
        std::shared_ptr<GpuContext> g(new GpuContext(c, max_streams, device));
        st = symgpu_mp3_streams_alloc(c, max_streams);
        if (st == SYMGPU_OK) st = symgpu_aac_streams_alloc(c, max_streams);
        if (st != SYMGPU_OK) return {nullptr, map_status(st)};
        return {g, {}};
    }
    ~GpuContext() { symgpu_ctx_destroy(ctx_); }
    symgpu_ctx* raw() const { return ctx_; }
    int device() const { return device_; }
    int acquire_stream() {
        std::lock_guard<std::mutex> g(m_);
        if (free_.empty()) return -1;
        const int s = free_.back();
        free_.pop_back();
        return s;
    }
    void release_stream(int s) {
        std::lock_guard<std::mutex> g(m_);
        free_.push_back(s);
    }

  private:
    GpuContext(symgpu_ctx* c, uint32_t n, int device) : ctx_(c), device_(device) {
        for (int i = (int)n - 1; i >= 0; --i) free_.push_back(i);
    }
    symgpu_ctx* ctx_;
    int device_;
    std::mutex m_;
    std::vector<int> free_;
};

// MPEG audio decoder (Layers I-III by codec id) whose synthesis stage runs on the GPU (mirrors MpaDecoder,
// symphonia-bundle-mp3/src/decoder.rs:66-197).  See the packet format note at the top of this file.
class GpuMpaDecoder final : public AudioDecoder {
  public:
    static constexpr size_t kPacketBytes = 4 * sizeof(symgpu_mp3_gc) + SYMGPU_MP3_FRAME_FLOATS * sizeof(float);

    static Result<std::unique_ptr<AudioDecoder>> try_new(std::shared_ptr<GpuContext> gpu, const AudioCodecParameters& p,
                                                         const AudioDecoderOptions& o) {
        if (p.codec != CODEC_ID_MP3 && p.codec != CODEC_ID_MP2 && p.codec != CODEC_ID_MP1)
            return {nullptr, {ErrorKind::Unsupported, "mpa: invalid codec type"}};
        const int slot = gpu->acquire_stream();
        if (slot < 0) return {nullptr, {ErrorKind::LimitError, "symgpu: no free stream slot"}};
        symgpu_mp3_fe* fe = nullptr;
        if (p.codec == CODEC_ID_MP3 && symgpu_mp3_fe_create(&fe) != SYMGPU_OK) {
            gpu->release_stream(slot);
            return {nullptr, {ErrorKind::LimitError, "symgpu: out of memory"}};
        }
        return {std::unique_ptr<AudioDecoder>(new GpuMpaDecoder(std::move(gpu), p, o, (uint32_t)slot, fe)), {}};
    }
    ~GpuMpaDecoder() override {
        symgpu_mp3_stream_reset(gpu_->raw(), stream_);
        gpu_->release_stream((int)stream_);
        symgpu_mp3_fe_destroy(fe_);
    }
    void reset() override { // decoder.rs:152-155: the whole decoder state starts over
        symgpu_mp3_stream_reset(gpu_->raw(), stream_);
        symgpu_mp3_fe_reset(fe_);
        have_spec_ = false;
        frames_ = 0;
    }
    const AudioCodecParameters& codec_params() const override { return params_; }
    Result<AudioBufferRef> decode(const Packet& packet) override {
        frames_ = 0; // buf.clear(): on any error the buffer stays empty (codecs/audio.rs:278)
        if (packet.len != kPacketBytes) return decode_frame(packet);
        if (params_.codec != CODEC_ID_MP3) return {{}, {ErrorKind::DecodeError, "mpa: invalid mpeg audio layer"}};
        symgpu_mp3_gc units[4];
        std::memcpy(units, packet.data, sizeof units);
        const float* spectra = reinterpret_cast<const float*>(packet.data + sizeof units);
        const bool mpeg1 = units[0].flags & SYMGPU_MP3_F_MPEG1;
        const bool mono = units[1].flags & SYMGPU_MP3_F_MUTE;
        const bool joint = units[0].flags & (SYMGPU_MP3_F_MID_SIDE | SYMGPU_MP3_F_INTENSITY);
        // stereo.rs:503-505: a parse-level validity check that stays on the host side of the ABI
        for (int gr = 0; gr < (mpeg1 ? 2 : 1) && joint && !mono; ++gr)
            if (units[2 * gr].block_type != units[2 * gr + 1].block_type ||
                ((units[2 * gr].flags ^ units[2 * gr + 1].flags) & SYMGPU_MP3_F_MIXED))
                return {{}, {ErrorKind::DecodeError, "mpa: stereo channel pair block_type mismatch"}};
        symgpu_mp3_run run{};
        run.stream = stream_;
        run.first_frame = 0;
        run.n_frames = 1;
        run.granules_per_frame = mpeg1 ? 2 : 1;
        run.channels = mono ? 1 : 2;
        // thread-safe, batched with the packets other decoders of this context have in flight
        symgpu_ticket ticket;
        symgpu_status st = symgpu_mp3_submit(gpu_->raw(), stream_, units, spectra, run.granules_per_frame, run.channels, &ticket);
        if (st == SYMGPU_OK) st = symgpu_mp3_wait(gpu_->raw(), ticket, pcm_.data());
        if (st != SYMGPU_OK) return {{}, map_status(st)};
        return finish(packet, mpeg1 ? 1152 : 576, mono ? 1 : 2);
    }
    AudioBufferRef last_decoded() const override {
        AudioBufferRef r;
        r.n_planes = planes_;
        r.frames = frames_;
        r.planes[0] = pcm_.data() + first_;
        r.planes[1] = pcm_.data() + 1152 + first_;
        return r;
    }

  private:
    GpuMpaDecoder(std::shared_ptr<GpuContext> gpu, AudioCodecParameters p, AudioDecoderOptions o, uint32_t stream, symgpu_mp3_fe* fe)
        : gpu_(std::move(gpu)), params_(std::move(p)), opts_(o), stream_(stream), fe_(fe), pcm_(SYMGPU_MP3_FRAME_FLOATS, 0.0f),
          planes_(params_.channels ? params_.channels : 2) {}

    // A real frame: entropy front-end on the CPU (MpaDecoder::decode_inner up to the synthesis call), synthesis on the GPU.
    Result<AudioBufferRef> decode_frame(const Packet& packet) {
        symgpu_mp3_frame_info info{};
        symgpu_status st;
        size_t frames;
        if (params_.codec == CODEC_ID_MP3) {
            symgpu_mp3_gc units[4];
            st = symgpu_mp3_fe_decode(fe_, packet.data, packet.len, units, quant_, &info);
            if (st != SYMGPU_OK) return {{}, map_status(st)};
            const bool joint = units[0].flags & (SYMGPU_MP3_F_MID_SIDE | SYMGPU_MP3_F_INTENSITY);
            for (int gr = 0; gr < info.granules && joint && info.channels == 2; ++gr)  // stereo.rs:503-505
                if (units[2 * gr].block_type != units[2 * gr + 1].block_type ||
                    (units[2 * gr].block_type == SYMGPU_MP3_SHORT && ((units[2 * gr].flags ^ units[2 * gr + 1].flags) & SYMGPU_MP3_F_MIXED)))
                    return {{}, {ErrorKind::DecodeError, "mpa: stereo channel pair block_type mismatch"}};
            symgpu_mp3_run run{};
            run.stream = stream_, run.n_frames = 1, run.granules_per_frame = info.granules, run.channels = info.channels;
            symgpu_ticket ticket;
            st = symgpu_mp3_submit_quantized(gpu_->raw(), stream_, units, quant_, run.granules_per_frame, run.channels, &ticket);
            if (st == SYMGPU_OK) st = symgpu_mp3_wait(gpu_->raw(), ticket, pcm_.data());
            frames = info.granules == 2 ? 1152 : 576;
        } else {
            const int layer = params_.codec == CODEC_ID_MP1 ? 1 : 2, n_slots = layer == 1 ? 12 : 36;
            st = symgpu_mpa12_fe_decode(packet.data, packet.len, layer, sub_, &info);
            if (st != SYMGPU_OK) return {{}, map_status(st)};
            // decoder.rs:96-108: the signal specification is fixed by the first frame
            if (!have_spec_) have_spec_ = true, spec_rate_ = info.sample_rate, spec_channels_ = info.channels;
            else if (spec_rate_ != info.sample_rate || spec_channels_ != info.channels)
                return {{}, {ErrorKind::DecodeError, "mpa: invalid audio buffer signal spec for packet"}};
            symgpu_mpa12_run run{};
            run.stream = stream_, run.n_frames = 1, run.channels = info.channels;
            st = symgpu_mpa12_synth_host(gpu_->raw(), sub_, &run, 1, 1, (uint32_t)n_slots, pcm_.data());
            frames = 32 * (size_t)n_slots;
        }
        if (st != SYMGPU_OK) return {{}, map_status(st)};
        return finish(packet, frames, info.channels);
    }
    Result<AudioBufferRef> finish(const Packet& packet, size_t frames, size_t planes) {
        frames_ = frames, planes_ = planes;
        // gapless trimming (decoder.rs:130-132)
        size_t begin = 0, end = frames_;
        if (opts_.gapless) {
            begin = std::min<size_t>(packet.trim_start, frames_);
            end = frames_ - std::min<size_t>(packet.trim_end, frames_ - begin);
        }
        first_ = begin;
        frames_ = end - begin;
        return {last_decoded(), {}};
    }

    std::shared_ptr<GpuContext> gpu_;
    AudioCodecParameters params_;
    AudioDecoderOptions opts_;
    uint32_t stream_;
    symgpu_mp3_fe* fe_;
    std::vector<float> pcm_;
    int16_t quant_[4 * 576];
    float sub_[2 * 32 * 36];
    size_t frames_ = 0, first_ = 0, planes_ = 2;
    bool have_spec_ = false;
    uint32_t spec_rate_ = 0, spec_channels_ = 0;
};

// AAC-LC decoder whose filterbank runs on the GPU (mirrors AacDecoder, symphonia-codec-aac/src/aac/mod.rs:42-304).  A packet is
// one raw_data_block, what the reference's AdtsReader and IsoMp4Reader emit.  Without extra data the stream parameters are the
// codec parameters' (the ADTS case, mod.rs:64-78); with extra data they come from the AudioSpecificConfig, read and judged as the
// reference does (symgpu_aac_fe_create_asc: AAC-LC, no SBR, at most two channels, 1024-sample frames).
class GpuAacDecoder final : public AudioDecoder {
  public:
    static Result<std::unique_ptr<AudioDecoder>> try_new(std::shared_ptr<GpuContext> gpu, const AudioCodecParameters& p,
                                                         const AudioDecoderOptions&) {
        if (p.codec != CODEC_ID_AAC) return {nullptr, {ErrorKind::Unsupported, "aac: invalid codec"}};
        AudioCodecParameters params = p;
        symgpu_aac_fe* fe = nullptr;
        if (!p.extra_data.empty()) {  // AudioSpecificConfig (mod.rs:59-62, :101-108)
            symgpu_aac_asc asc;
            const symgpu_status st = symgpu_aac_fe_create_asc(p.extra_data.data(), p.extra_data.size(), &fe, &asc);
            if (st != SYMGPU_OK) return {nullptr, map_status(st)};
            params.sample_rate = asc.sample_rate, params.channels = asc.channels;
        }
        if (params.sample_rate == 0) return {nullptr, {ErrorKind::Unsupported, "aac: sample rate is required"}};
        if (params.channels == 0) return {nullptr, {ErrorKind::Unsupported, "aac: channels or channel layout is required"}};
        if (params.channels > 2) return {nullptr, {ErrorKind::Unsupported, "aac: aac too complex"}};
        const int slot = gpu->acquire_stream();
        if (slot < 0) {
            symgpu_aac_fe_destroy(fe);
            return {nullptr, {ErrorKind::LimitError, "symgpu: no free stream slot"}};
        }
        if (!fe) {
            const symgpu_status st = symgpu_aac_fe_create(params.sample_rate, params.channels, &fe);
            if (st != SYMGPU_OK) {
                gpu->release_stream(slot);
                return {nullptr, map_status(st)};
            }
        }
        symgpu_aac_stream_reset(gpu->raw(), (uint32_t)slot);
        return {std::unique_ptr<AudioDecoder>(new GpuAacDecoder(std::move(gpu), std::move(params), (uint32_t)slot, fe)), {}};
    }
    ~GpuAacDecoder() override {
        gpu_->release_stream((int)stream_);
        symgpu_aac_fe_destroy(fe_);
    }
    void reset() override {  // mod.rs:259-263: every pair's window history and delay lines
        symgpu_aac_stream_reset(gpu_->raw(), stream_);
        symgpu_aac_fe_reset(fe_);
        frames_ = 0;
    }
    const AudioCodecParameters& codec_params() const override { return params_; }
    Result<AudioBufferRef> decode(const Packet& packet) override {
        frames_ = 0;  // buf.clear() on any error (mod.rs:274-277)
        symgpu_aac_unit units[2];
        uint32_t n_tns = 0;
        symgpu_status st = symgpu_aac_fe_decode(fe_, packet.data, packet.len, 0, units, tns_, &n_tns, coeffs_.data());
        if (st != SYMGPU_OK) return {{}, map_status(st)};
        symgpu_aac_run run{};
        run.stream = stream_, run.first_frame = 0, run.n_frames = 1, run.channels = (uint8_t)params_.channels;
        st = symgpu_aac_synth_host(gpu_->raw(), units, n_tns ? tns_ : nullptr, n_tns, coeffs_.data(), &run, 1, 1, pcm_.data());
        if (st != SYMGPU_OK) return {{}, map_status(st)};
        frames_ = 1024;  // the reference's AAC decoder trims nothing (mod.rs:231-255)
        return {last_decoded(), {}};
    }
    AudioBufferRef last_decoded() const override {
        AudioBufferRef r;
        r.n_planes = params_.channels;
        r.frames = frames_;
        r.planes[0] = pcm_.data();
        r.planes[1] = pcm_.data() + 1024;
        return r;
    }

  private:
    GpuAacDecoder(std::shared_ptr<GpuContext> gpu, AudioCodecParameters p, uint32_t stream, symgpu_aac_fe* fe)
        : gpu_(std::move(gpu)), params_(std::move(p)), stream_(stream), fe_(fe), coeffs_(2048, 0.0f), pcm_(2048, 0.0f) {}
    std::shared_ptr<GpuContext> gpu_;
    AudioCodecParameters params_;
    uint32_t stream_;
    symgpu_aac_fe* fe_;
    symgpu_aac_tns tns_[16];
    std::vector<float> coeffs_, pcm_;
    size_t frames_ = 0;
};

// Vorbis decoder whose floor synthesis, inverse coupling, IMDCT and overlap-add run on the GPU (mirrors VorbisDecoder,
// symphonia-codec-vorbis/src/lib.rs:48-420).  Extra data = the identification packet followed by the setup packet, as the Ogg
// mapping hands them over (mappings/vorbis.rs:196-214).  The library registers Vorbis streams and floor tables per context, all
// at once, so this decoder owns a context of its own on the shared context's device.
class GpuVorbisDecoder final : public AudioDecoder {
  public:
    static Result<std::unique_ptr<AudioDecoder>> try_new(std::shared_ptr<GpuContext> gpu, const AudioCodecParameters& p,
                                                         const AudioDecoderOptions& o) {
        if (p.codec != CODEC_ID_VORBIS) return {nullptr, {ErrorKind::Unsupported, "vorbis: invalid codec type"}};
        if (p.extra_data.size() <= 30) return {nullptr, {ErrorKind::Unsupported, "vorbis: missing extra data"}};
        // a stream the two-plane front-end takes keeps that path; any other (3 to 8 channels, other couplings) opens multichannel
        symgpu_vorbis_fe* fe = nullptr;
        const uint8_t *ident = p.extra_data.data(), *setup = ident + 30;
        symgpu_status st = symgpu_vorbis_fe_create(ident, 30, setup, p.extra_data.size() - 30, &fe);
        const bool mc = st == SYMGPU_ERR_UNSUPPORTED;
        if (mc) st = symgpu_vorbis_fe_create_mc(ident, 30, setup, p.extra_data.size() - 30, &fe);
        if (st != SYMGPU_OK) return {nullptr, map_status(st)};
        symgpu_vorbis_stream stream{};
        symgpu_vorbis_stream_mc stream_mc{};
        std::vector<symgpu_vorbis_floor1> floors(64);
        uint32_t n_floors = 0;
        if (mc) {
            symgpu_vorbis_fe_config_mc(fe, &stream_mc, floors.data(), &n_floors);
            stream = symgpu_vorbis_stream{stream_mc.bs0_exp, stream_mc.bs1_exp, stream_mc.channels, 0};
        } else {
            symgpu_vorbis_fe_config(fe, &stream, floors.data(), &n_floors);
        }
        symgpu_ctx* ctx = nullptr;
        st = symgpu_ctx_create(gpu->device(), &ctx);
        if (st == SYMGPU_OK) st = mc ? symgpu_vorbis_mc_streams_set(ctx, &stream_mc, 1) : symgpu_vorbis_streams_set(ctx, &stream, 1);
        if (st == SYMGPU_OK && n_floors) st = symgpu_vorbis_floors_set(ctx, floors.data(), n_floors);
        if (st != SYMGPU_OK) {
            symgpu_vorbis_fe_destroy(fe);
            if (ctx) symgpu_ctx_destroy(ctx);
            return {nullptr, map_status(st)};
        }
        AudioCodecParameters params = p;
        params.channels = stream.channels;
        return {std::unique_ptr<AudioDecoder>(new GpuVorbisDecoder(ctx, std::move(params), o, fe, stream, mc)), {}};
    }
    ~GpuVorbisDecoder() override {
        symgpu_vorbis_fe_destroy(fe_);
        symgpu_ctx_destroy(ctx_);
    }
    void reset() override {  // lib.rs:336-338 -> dsp.rs:26-32: overlap cleared, no previous block
        if (mc_) symgpu_vorbis_mc_stream_reset(ctx_, 0);
        else symgpu_vorbis_stream_reset(ctx_, 0);
        symgpu_vorbis_fe_reset(fe_);
        have_prev_ = false;
        frames_ = 0;
    }
    const AudioCodecParameters& codec_params() const override { return params_; }
    Result<AudioBufferRef> decode(const Packet& packet) override {
        frames_ = first_ = 0;
        symgpu_vorbis_run run{};
        run.stream = 0, run.first_packet = 0, run.n_packets = 1;
        symgpu_vorbis_unit_mc unit;  // (block flags only, in both paths)
        symgpu_status st;
        if (mc_) {
            const uint32_t C = stream_.channels;
            st = symgpu_vorbis_fe_decode_mc(fe_, packet.data, packet.len, slot_, 0, C, &unit, floor_y_, residue_.data());
            if (st != SYMGPU_OK) return {{}, map_status(st)};
            st = symgpu_vorbis_mc_synth_host(ctx_, &unit, floor_y_, residue_.data(), &run, 1, 1, C, slot_, pcm_.data());
        } else {
            symgpu_vorbis_unit u2;
            st = symgpu_vorbis_fe_decode(fe_, packet.data, packet.len, slot_, 0, &u2, floor_y_, residue_.data());
            if (st != SYMGPU_OK) return {{}, map_status(st)};
            unit.block_flag = u2.block_flag, unit.prev_block_flag = u2.prev_block_flag;
            st = symgpu_vorbis_synth_host(ctx_, &u2, floor_y_, residue_.data(), &run, 1, 1, slot_, pcm_.data());
        }
        if (st != SYMGPU_OK) return {{}, map_status(st)};
        const size_t prev_n = size_t(1) << (unit.prev_block_flag ? stream_.bs1_exp : stream_.bs0_exp);
        const size_t n = size_t(1) << (unit.block_flag ? stream_.bs1_exp : stream_.bs0_exp);
        frames_ = (prev_n + n) / 4;
        if (opts_.gapless) {  // lib.rs:316-326
            if (!have_prev_) {
                frames_ = 0;  // the first packet after a reset is silenced
            } else {
                first_ = std::min<size_t>(packet.trim_start, frames_);
                frames_ -= first_;
                frames_ -= std::min<size_t>(packet.trim_end, frames_);
            }
        }
        have_prev_ = true;
        return {last_decoded(), {}};
    }
    AudioBufferRef last_decoded() const override {
        AudioBufferRef r;
        r.n_planes = params_.channels;
        r.frames = frames_;
        if (!mc_) {
            r.planes[0] = pcm_.data() + first_;
            r.planes[1] = pcm_.data() + slot_ + first_;
            return r;
        }
        for (size_t i = 0; i < params_.channels; ++i) r.planes[map_[i]] = pcm_.data() + i * slot_ + first_;  // lib.rs:307-315
        return r;
    }

  private:
    GpuVorbisDecoder(symgpu_ctx* ctx, AudioCodecParameters p, AudioDecoderOptions o, symgpu_vorbis_fe* fe, symgpu_vorbis_stream stream, bool mc)
        : ctx_(ctx), params_(std::move(p)), opts_(o), fe_(fe), stream_(stream), mc_(mc), slot_((1u << stream.bs1_exp) >> 1),
          residue_(std::max<size_t>(2, stream.channels) * slot_, 0.0f), pcm_(std::max<size_t>(2, stream.channels) * slot_, 0.0f) {
        symgpu_vorbis_channel_map(stream.channels, map_);
    }
    symgpu_ctx* ctx_;
    AudioCodecParameters params_;
    AudioDecoderOptions opts_;
    symgpu_vorbis_fe* fe_;
    symgpu_vorbis_stream stream_;  // (channels and block sizes; `coupled` unused on the multichannel path)
    bool mc_;
    uint32_t slot_;
    uint8_t map_[SYMGPU_VORBIS_MAX_CHANNELS] = {};
    uint16_t floor_y_[SYMGPU_VORBIS_MAX_CHANNELS * 65];
    std::vector<float> residue_, pcm_;
    size_t frames_ = 0, first_ = 0;
    bool have_prev_ = false;
};

// FLAC decoder whose integer restoration (prediction, wasted bits, decorrelation, scaling to 32 bits) runs on the GPU (mirrors
// FlacDecoder, symphonia-bundle-flac/src/decoder.rs:84-313).  A packet is one frame, what the reference's FLAC reader emits; the
// frame header and the sub-frame / Rice reader run on the CPU (symgpu_flac_fe_decode_packets), the restoration as a batch of one
// (symgpu_flac_restore_host).  The result is planar S32, as the reference's AudioBuffer<i32>.  FLAC keeps no state between packets,
// so the decoder takes no stream slot.  finalize() does not check the MD5 of the decoded audio (INTEGRATION.md §4).
class GpuFlacDecoder final : public AudioDecoder {
  public:
    static Result<std::unique_ptr<AudioDecoder>> try_new(std::shared_ptr<GpuContext> gpu, const AudioCodecParameters& p,
                                                         const AudioDecoderOptions&) {
        if (p.codec != CODEC_ID_FLAC) return {nullptr, {ErrorKind::Unsupported, "flac: invalid codec"}};
        if (p.extra_data.empty()) return {nullptr, {ErrorKind::Unsupported, "flac: missing extra data"}};
        symgpu::packet::FlacStreamInfo info{};
        switch (symgpu::packet::flac_read_stream_info(p.extra_data.data(), p.extra_data.size(), info)) {  // StreamInfo::read
            case symgpu::packet::Status::Ok: break;
            case symgpu::packet::Status::EndOfStream: return {nullptr, {ErrorKind::IoError, "flac: stream information block is cut short"}};
            case symgpu::packet::Status::Unsupported: return {nullptr, {ErrorKind::Unsupported, "flac: unsupported stream information"}};
            default: return {nullptr, {ErrorKind::DecodeError, "flac: invalid stream information block"}};
        }
        AudioCodecParameters params = p;
        params.sample_rate = info.sample_rate, params.channels = info.channels;
        return {std::unique_ptr<AudioDecoder>(new GpuFlacDecoder(std::move(gpu), std::move(params), info)), {}};
    }
    void reset() override {}  // no state between packets
    FinalizeResult finalize() override { return {}; }  // no MD5 check: has_verify stays false, also with verify = true
    const AudioCodecParameters& codec_params() const override { return params_; }
    Result<AudioBufferRef> decode(const Packet& packet) override {
        frames_ = 0;  // on any error the buffer is empty
        // decoder.rs:169-171: a block larger than the stream's largest is refused before its sub-frames are read
        size_t at = 0;
        while (at + 2 <= packet.len && !(packet.data[at] == 0xff && (packet.data[at + 1] & 0xfc) == 0xf8)) ++at;
        symgpu::packet::FlacFrameHeader h{};
        if (at + 2 <= packet.len && symgpu::packet::flac_parse_frame_header(packet.data + at, packet.len - at, h) && h.block > info_.block_max)
            return {{}, {ErrorKind::DecodeError, "flac: allocation would overflow buffer"}};
        const symgpu_piece piece{0, (uint32_t)packet.len, 0};
        symgpu_flac_frame_info fi;
        uint32_t frame_of = 0;
        size_t n_good = 0, n_subs = 0, n_samples = 0;
        symgpu_status st = symgpu_flac_fe_decode_packets(packet.data, packet.len, &piece, 1, info_.bits_per_sample, info_.channels, info_.block_max,
                                                         &frame_, &fi, &frame_of, subs_, 8, samples_.data(), samples_.size(), &n_good, &n_subs,
                                                         &n_samples);
        if (st != SYMGPU_OK) return {{}, map_status(st)};
        if (n_good != 1) return {{}, map_status(SYMGPU_ERR_DECODE)};
        st = symgpu_flac_restore_host(gpu_->raw(), &frame_, 1, subs_, (uint32_t)n_subs, samples_.data(), n_samples);
        if (st != SYMGPU_OK) return {{}, map_status(st)};
        frames_ = fi.block_size;
        return {last_decoded(), {}};
    }
    AudioBufferRef last_decoded() const override {
        AudioBufferRef r;
        r.format = SampleFormat::S32;
        r.n_planes = params_.channels;
        r.frames = frames_;
        for (size_t c = 0; c < params_.channels; ++c)  // a frame with fewer channels than the stream leaves the others silent
            r.planes_s32[c] = c < frame_.channels ? samples_.data() + subs_[c].offset : silence_.data();
        return r;
    }

  private:
    GpuFlacDecoder(std::shared_ptr<GpuContext> gpu, AudioCodecParameters p, const symgpu::packet::FlacStreamInfo& info)
        : gpu_(std::move(gpu)), params_(std::move(p)), info_(info), samples_(size_t(info.channels) * info.block_max, 0),
          silence_(info.block_max, 0) {}
    std::shared_ptr<GpuContext> gpu_;
    AudioCodecParameters params_;
    symgpu::packet::FlacStreamInfo info_;
    symgpu_flac_frame frame_{};
    symgpu_flac_subframe subs_[8] = {};
    std::vector<int32_t> samples_, silence_;
    size_t frames_ = 0;
};

// What an application does next to symphonia::default::register_enabled_codecs (symphonia/src/lib.rs:234-255).
inline void register_gpu_decoders(CodecRegistry& registry, std::shared_ptr<GpuContext> gpu) {
    for (uint32_t codec : {CODEC_ID_MP1, CODEC_ID_MP2, CODEC_ID_MP3})
        registry.register_audio_decoder_at_tier(Tier::Preferred, codec, [gpu](const AudioCodecParameters& p, const AudioDecoderOptions& o) {
            return GpuMpaDecoder::try_new(gpu, p, o);
        });
    registry.register_audio_decoder_at_tier(Tier::Preferred, CODEC_ID_AAC, [gpu](const AudioCodecParameters& p, const AudioDecoderOptions& o) {
        return GpuAacDecoder::try_new(gpu, p, o);
    });
    registry.register_audio_decoder_at_tier(Tier::Preferred, CODEC_ID_VORBIS, [gpu](const AudioCodecParameters& p, const AudioDecoderOptions& o) {
        return GpuVorbisDecoder::try_new(gpu, p, o);
    });
    registry.register_audio_decoder_at_tier(Tier::Preferred, CODEC_ID_FLAC, [gpu](const AudioCodecParameters& p, const AudioDecoderOptions& o) {
        return GpuFlacDecoder::try_new(gpu, p, o);
    });
}

} // namespace symgpu_host
