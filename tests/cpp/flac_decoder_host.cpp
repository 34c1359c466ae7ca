// GpuFlacDecoder (include/symgpu/decoder.hpp) driven from C++ the way an application drives the reference's FlacDecoder.
//   flac_decoder_host file IN OUT   GPU tier: a native FLAC file -- FlacIndexer (packetizer.hpp), registry, one decode() per frame --
//                                   interleaved int32 [frames, channels] of every packet, back to back, written to OUT
//   flac_decoder_host errors IN     GPU tier: a wrong codec id and missing extra data -> Unsupported; a block larger than the
//                                   STREAMINFO's largest -> DecodeError with an empty buffer; the decoder still decodes afterwards
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iterator>
#include <vector>

#include "../../include/symgpu/decoder.hpp"
#include "../../include/symgpu/packetizer.hpp"

using namespace symgpu_host;

static int check(bool cond, const char* what) {
    if (!cond) std::fprintf(stderr, "FAILED: %s\n", what);
    return cond ? 0 : 1;
}

static std::vector<uint8_t> read_file(const char* path) {
    std::ifstream f(path, std::ios::binary);
    return std::vector<uint8_t>((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
}

struct Opened {
    std::vector<uint8_t> data;
    std::vector<symgpu::packet::FlacPacket> packets;
    AudioCodecParameters params;
};

// The file, its frames, and the codec parameters a FLAC reader hands to the decoder: the STREAMINFO body as extra data.
static bool open_file(const char* path, Opened& o) {
    o.data = read_file(path);
    symgpu::packet::FlacStreamInfo info{};
    if (symgpu::packet::FlacIndexer::index(o.data.data(), o.data.size(), info, o.packets) != symgpu::packet::Status::Ok) return false;
    o.params.codec = CODEC_ID_FLAC;
    o.params.extra_data.assign(o.data.begin() + 8, o.data.begin() + 8 + 34);  // "fLaC", block header, STREAMINFO (the first block)
    return true;
}

static Packet packet_of(const Opened& o, size_t k) {
    Packet p;
    p.data = o.data.data() + o.packets[k].offset;
    p.len = o.packets[k].size;
    p.pts = o.packets[k].ts;
    p.dur = o.packets[k].dur;
    return p;
}

static int run_file(const char* in, const char* out) {
    Opened o;
    if (!open_file(in, o)) return check(false, "index the file");
    auto gpu = GpuContext::create(0, 4);
    if (!gpu.ok()) return check(false, gpu.error.message);
    CodecRegistry reg;
    register_gpu_decoders(reg, gpu.value);
    auto dec = reg.make_audio_decoder(o.params, {});
    if (!dec.ok()) return check(false, dec.error.message);
    const AudioCodecParameters& cp = dec.value->codec_params();
    std::vector<int32_t> pcm;
    for (size_t k = 0; k < o.packets.size(); ++k) {
        auto r = dec.value->decode(packet_of(o, k));
        if (!r.ok()) {
            std::fprintf(stderr, "packet %zu: %s\n", k, r.error.message);
            return 1;
        }
        const AudioBufferRef& b = r.value;
        if (b.format != SampleFormat::S32 || b.n_planes != cp.channels) return check(false, "planar S32 with the stream's channels");
        for (size_t i = 0; i < b.frames; ++i)
            for (size_t c = 0; c < b.n_planes; ++c) pcm.push_back(b.planes_s32[c][i]);
    }
    AudioDecoderOptions verify;
    verify.verify = true;
    auto dv = reg.make_audio_decoder(o.params, verify);
    if (!dv.ok() || dv.value->finalize().has_verify) return check(false, "finalize() reports no verification");
    std::ofstream f(out, std::ios::binary);
    f.write(reinterpret_cast<const char*>(pcm.data()), std::streamsize(pcm.size() * sizeof(int32_t)));
    std::printf("flac file: %zu packets, %zu samples, %u Hz, %u channels\n", o.packets.size(), pcm.size(), cp.sample_rate, cp.channels);
    return 0;
}

static int run_errors(const char* in) {
    int bad = 0;
    Opened o;
    if (!open_file(in, o)) return check(false, "index the file");
    auto gpu = GpuContext::create(0, 4);
    if (!gpu.ok()) return check(false, gpu.error.message);
    CodecRegistry reg;
    register_gpu_decoders(reg, gpu.value);
    AudioCodecParameters wrong = o.params;
    wrong.codec = CODEC_ID_VORBIS;
    auto w = GpuFlacDecoder::try_new(gpu.value, wrong, {});
    bad += check(w.error.kind == ErrorKind::Unsupported && std::strcmp(w.error.message, "flac: invalid codec") == 0, "wrong codec -> Unsupported");
    AudioCodecParameters bare = o.params;
    bare.extra_data.clear();
    auto m = reg.make_audio_decoder(bare, {});
    bad += check(m.error.kind == ErrorKind::Unsupported && std::strcmp(m.error.message, "flac: missing extra data") == 0,
                 "missing extra data -> Unsupported");
    // STREAMINFO that promises blocks of at most 16 samples: every frame of the file is larger
    AudioCodecParameters small = o.params;
    small.extra_data[0] = 0, small.extra_data[1] = 16, small.extra_data[2] = 0, small.extra_data[3] = 16;
    auto s = reg.make_audio_decoder(small, {});
    if (!s.ok()) return check(false, s.error.message);
    auto r = s.value->decode(packet_of(o, 0));
    bad += check(r.error.kind == ErrorKind::DecodeError && std::strcmp(r.error.message, "flac: allocation would overflow buffer") == 0,
                 "oversized block -> DecodeError");
    bad += check(r.value.frames == 0 && s.value->last_decoded().frames == 0, "the buffer is empty after an error");
    auto d = reg.make_audio_decoder(o.params, {});
    if (!d.ok()) return check(false, d.error.message);
    auto r2 = d.value->decode(packet_of(o, 0));
    bad += check(r2.ok() && r2.value.frames == o.packets[0].dur, "a decoder of the same context decodes afterwards");
    if (!bad) std::printf("flac errors: ok\n");
    return bad;
}

int main(int argc, char** argv) {
    if (argc == 4 && std::strcmp(argv[1], "file") == 0) return run_file(argv[2], argv[3]);
    if (argc == 3 && std::strcmp(argv[1], "errors") == 0) return run_errors(argv[2]);
    std::fprintf(stderr, "usage: flac_decoder_host file IN OUT | errors IN\n");
    return 2;
}
