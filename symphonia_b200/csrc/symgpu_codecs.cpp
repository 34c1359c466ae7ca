// AAC-LC and Vorbis entry points of the C ABI (include/symgpu.h).  Like the MP3 ones they only
// stage buffers, cut runs into per-CTA chunks and launch CUDA kernels: there is no CPU path.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <vector>

#include "ctx.h"
#include "flac_kernel.h"

using namespace symgpu;
using namespace symgpu_detail;

namespace {

// Key of a chunk list: which codec built it, from which runs, with which parameters.
std::vector<unsigned char> chunk_key_of(uint32_t tag, uint32_t a, uint32_t b, const void* runs, size_t run_bytes) {
    std::vector<unsigned char> k(12 + run_bytes);
    std::memcpy(k.data(), &tag, 4);
    std::memcpy(k.data() + 4, &a, 4);
    std::memcpy(k.data() + 8, &b, 4);
    if (run_bytes) std::memcpy(k.data() + 12, runs, run_bytes);
    return k;
}

symgpu_status upload_chunks(symgpu_ctx* ctx, const std::vector<CodecChunk>& chunks) {
    // Chunk lists are small; rewriting them needs the previous launch to have consumed the old list.
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    if (chunks.size() > ctx->chunks_cap) {
        if (ctx->d_chunks) cudaFree(ctx->d_chunks);
        if (ctx->h_chunks) cudaFreeHost(ctx->h_chunks);
        ctx->d_chunks = nullptr;
        ctx->h_chunks = nullptr;
        ctx->chunks_cap = 0;
        const size_t cap = chunks.size() * 2 + 64;
        CU(ctx, cudaMalloc(&ctx->d_chunks, cap * sizeof(CodecChunk)));
        CU(ctx, cudaMallocHost(&ctx->h_chunks, cap * sizeof(CodecChunk)));
        ctx->chunks_cap = cap;
    }
    std::memcpy(ctx->h_chunks, chunks.data(), chunks.size() * sizeof(CodecChunk));
    CU(ctx, cudaMemcpyAsync(ctx->d_chunks, ctx->h_chunks, chunks.size() * sizeof(CodecChunk), cudaMemcpyHostToDevice, ctx->stream));
    return SYMGPU_OK;
}

// Splits [0, n) into ceil(n / per) near-equal pieces.
template <typename F>
void split_even(uint32_t n, uint32_t per, F&& f) {
    const uint32_t pieces = (n + per - 1) / per;
    uint32_t lo = 0;
    for (uint32_t k = 0; k < pieces; ++k) {
        const uint32_t hi = (uint32_t)(((uint64_t)n * (k + 1)) / pieces);
        f(lo, hi, k == 0, k + 1 == pieces);
        lo = hi;
    }
}

symgpu_status ensure_codec_tables(symgpu_ctx* ctx) {
    if (ctx->d_codec_tab) return SYMGPU_OK;
    const CodecTables& t = codec_tables_host();
    CU(ctx, cudaMalloc(&ctx->d_codec_tab, sizeof t));
    CU(ctx, cudaMemcpy(ctx->d_codec_tab, &t, sizeof t, cudaMemcpyHostToDevice));
    return SYMGPU_OK;
}

} // namespace

extern "C" {

// ---- AAC ---------------------------------------------------------------------------------------

symgpu_status symgpu_aac_streams_alloc(symgpu_ctx* ctx, uint32_t n_streams) {
    if (!ctx || n_streams == 0) return SYMGPU_ERR_ARG;
    DeviceGuard guard(ctx->device);
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    symgpu_status s = ensure_codec_tables(ctx);
    if (s != SYMGPU_OK) return s;
    if (ctx->d_aac_states) cudaFree(ctx->d_aac_states);
    if (ctx->d_aac_gen) cudaFree(ctx->d_aac_gen);
    ctx->d_aac_states = nullptr;
    ctx->d_aac_gen = nullptr;
    ctx->n_aac_streams = 0;
    const size_t bytes = (size_t)n_streams * 2 * 2 * 1024 * sizeof(float);
    CU(ctx, cudaMalloc(&ctx->d_aac_states, bytes));
    CU(ctx, cudaMemset(ctx->d_aac_states, 0, bytes));
    CU(ctx, cudaMalloc(&ctx->d_aac_gen, ((size_t)n_streams + 1) * sizeof(uint32_t)));
    CU(ctx, cudaMemset(ctx->d_aac_gen, 0, ((size_t)n_streams + 1) * sizeof(uint32_t)));
    ctx->n_aac_streams = n_streams;
    ctx->chunk_key.clear();
    return SYMGPU_OK;
}

symgpu_status symgpu_aac_stream_reset(symgpu_ctx* ctx, uint32_t stream) {
    if (!ctx) return SYMGPU_ERR_ARG;
    if (stream >= ctx->n_aac_streams) return SYMGPU_ERR_LIMIT;
    DeviceGuard guard(ctx->device);
    CU(ctx, cudaMemsetAsync(ctx->d_aac_states + (size_t)stream * 4096, 0, 4096 * sizeof(float), ctx->stream));
    return SYMGPU_OK;
}

symgpu_status symgpu_aac_synth_dev(symgpu_ctx* ctx, const symgpu_aac_unit* units, const symgpu_aac_tns* tns,
                                   uint32_t n_tns, const float* coeffs, const symgpu_aac_run* runs, uint32_t n_runs,
                                   uint32_t n_frames, float* pcm) {
    if (!ctx || !units || !coeffs || !runs || !pcm || (n_tns && !tns)) return SYMGPU_ERR_ARG;
    if (n_frames == 0) return SYMGPU_OK;
    if (!ctx->d_aac_states) return SYMGPU_ERR_LIMIT;
    DeviceGuard guard(ctx->device);
    std::vector<CodecChunk> chunks;
    uint64_t covered = 0;
    const std::vector<unsigned char> key = chunk_key_of(0x41414300u, n_frames, ctx->n_aac_streams, runs, (size_t)n_runs * sizeof *runs);
    const bool reuse = key == ctx->chunk_key;
    // frames per chunk: a function of the runs alone (so a cached plan stays valid), shorter chunks for short runs
    uint64_t run_frames = 0, run_count = 0;
    for (uint32_t r = 0; r < n_runs; ++r)
        if (runs[r].n_frames) run_frames += runs[r].n_frames, ++run_count;
    const int chunk_frames = aac_chunk_frames_for(run_count ? (uint32_t)(run_frames / run_count) : 1u);
    for (uint32_t r = 0; r < n_runs && !reuse; ++r) {
        const symgpu_aac_run& run = runs[r];
        const int n_ch = run.channels ? run.channels : 2;
        if (n_ch < 1 || n_ch > 2) return SYMGPU_ERR_ARG;
        if (run.n_frames == 0) continue;
        if ((uint64_t)run.first_frame + run.n_frames > n_frames) return SYMGPU_ERR_ARG;
        if (run.stream >= ctx->n_aac_streams) return SYMGPU_ERR_LIMIT;
        covered += run.n_frames;
        for (int ch = 0; ch < n_ch; ++ch)
            split_even(run.n_frames, (uint32_t)chunk_frames, [&](uint32_t lo, uint32_t hi, bool first, bool last) {
                CodecChunk c{};
                c.first = run.first_frame + lo;
                c.stream = run.stream;
                c.count = (uint16_t)(hi - lo);
                c.channel = (uint8_t)ch;
                c.flags = (uint8_t)((first ? kChunkLoadState : 0) | (last ? kChunkStoreState : 0));
                chunks.push_back(c);
            });
    }
    symgpu_status s = SYMGPU_OK;
    if (!reuse) {
        if (covered > n_frames) return SYMGPU_ERR_ARG; // runs may leave frames out (a stream that lost packets), never overlap
        ctx->chunk_key.clear();
        // A CTA pass takes a GROUP of consecutive chunks whose frame slots (count + 1 each: the state or the frame before the
        // chunk rides along) fit its warps, so short runs (a stream that submits a few frames per call) still fill the CTA.
        // group_first[g] .. group_first[g + 1] are the chunks of group g; the array travels behind the chunk list.
        const size_t n_chunks = chunks.size();
        std::vector<uint32_t> group_first;
        const uint32_t cap_slots = (uint32_t)chunk_frames + 1;
        uint32_t used = cap_slots + 1; // forces the first chunk to open a group
        for (size_t i = 0; i < n_chunks; ++i) {
            const uint32_t need = (uint32_t)chunks[i].count + 1;
            if (used + need > cap_slots) {
                group_first.push_back((uint32_t)i);
                used = 0;
            }
            used += need;
        }
        const size_t n_groups = group_first.size();
        group_first.push_back((uint32_t)n_chunks);
        chunks.resize(n_chunks + (group_first.size() * sizeof(uint32_t) + sizeof(CodecChunk) - 1) / sizeof(CodecChunk));
        std::memcpy(static_cast<void*>(chunks.data() + n_chunks), group_first.data(), group_first.size() * sizeof(uint32_t));
        s = upload_chunks(ctx, chunks);
        if (s != SYMGPU_OK) return s;
        ctx->chunk_key = key;
        ctx->cached_chunks = (int)n_chunks;
        ctx->cached_groups = (int)n_groups;
    }
    const size_t spec_bytes = (size_t)n_frames * 2 * 1024 * sizeof(float);
    if (n_tns && spec_bytes > ctx->aac_scratch_cap) {
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        if (ctx->d_aac_scratch) cudaFree(ctx->d_aac_scratch);
        ctx->d_aac_scratch = nullptr;
        ctx->aac_scratch_cap = 0;
        CU(ctx, cudaMalloc(&ctx->d_aac_scratch, spec_bytes));
        ctx->aac_scratch_cap = spec_bytes;
    }
    if (n_tns > ctx->aac_tns_idx_cap) {
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        if (ctx->d_aac_tns_idx) cudaFree(ctx->d_aac_tns_idx);
        ctx->d_aac_tns_idx = nullptr;
        ctx->aac_tns_idx_cap = 0;
        const size_t cap = (size_t)n_tns + n_tns / 2 + 256;
        CU(ctx, cudaMalloc(&ctx->d_aac_tns_idx, 2 * cap * sizeof(uint32_t)));
        ctx->aac_tns_idx_cap = cap;
    }
    AacArgs a{units, tns, coeffs, ctx->d_aac_scratch, ctx->d_aac_scratch,
              ctx->d_aac_tns_idx, ctx->d_aac_tns_idx ? ctx->d_aac_tns_idx + ctx->aac_tns_idx_cap : nullptr, n_tns, 0, chunk_frames, 0, 0,
              pcm, ctx->d_chunks, ctx->d_aac_states, ctx->d_aac_gen, ctx->d_aac_gen + ctx->n_aac_streams, ctx->d_codec_tab};
    CU(ctx, aac_launch(a, n_frames * 2, n_tns != 0, ctx->cached_chunks, ctx->cached_groups, ctx->stream));
    ctx->launches += aac_launch_count(n_tns != 0);
    return SYMGPU_OK;
}

symgpu_status symgpu_aac_units_check(const symgpu_aac_unit* units, const symgpu_aac_tns* tns, uint32_t n_tns, uint32_t n_frames) {
    if (!units || (n_tns && !tns)) return SYMGPU_ERR_ARG;
    for (size_t k = 0; k < (size_t)n_frames * 2; ++k) {
        const symgpu_aac_unit& u = units[k];
        if (u.window_sequence > SYMGPU_AAC_LONG_STOP || u.window_shape > 1 || u.prev_window_shape > 1) return SYMGPU_ERR_DECODE;
        if (u.n_tns && ((uint64_t)u.tns_first + u.n_tns > n_tns)) return SYMGPU_ERR_DECODE;
    }
    for (uint32_t f = 0; f < n_tns; ++f)
        if (tns[f].order > 20 || tns[f].start > tns[f].end || tns[f].end > 1024) return SYMGPU_ERR_DECODE;
    return SYMGPU_OK;
}

symgpu_status symgpu_aac_synth_host(symgpu_ctx* ctx, const symgpu_aac_unit* units, const symgpu_aac_tns* tns,
                                    uint32_t n_tns, const float* coeffs, const symgpu_aac_run* runs, uint32_t n_runs,
                                    uint32_t n_frames, float* pcm) {
    if (!ctx || !units || !coeffs || !runs || !pcm || (n_tns && !tns)) return SYMGPU_ERR_ARG;
    if (n_frames == 0) return SYMGPU_OK;
    {
        const symgpu_status chk = symgpu_aac_units_check(units, tns, n_tns, n_frames);
        if (chk != SYMGPU_OK) return chk;
    }
    DeviceGuard guard(ctx->device);
    const size_t unit_bytes = (size_t)n_frames * 2 * sizeof(symgpu_aac_unit);
    const size_t spec_bytes = (size_t)n_frames * 2 * 1024 * sizeof(float);
    const size_t tns_bytes = ((size_t)n_tns * sizeof(symgpu_aac_tns) + 15) & ~(size_t)15;
    symgpu_status s = ensure_stage(ctx, 2 * spec_bytes + unit_bytes + tns_bytes);
    if (s != SYMGPU_OK) return s;
    char* base = static_cast<char*>(ctx->d_stage);
    float* d_spec = reinterpret_cast<float*>(base);
    float* d_pcm = reinterpret_cast<float*>(base + spec_bytes);
    symgpu_aac_unit* d_units = reinterpret_cast<symgpu_aac_unit*>(base + 2 * spec_bytes);
    symgpu_aac_tns* d_tns = reinterpret_cast<symgpu_aac_tns*>(base + 2 * spec_bytes + unit_bytes);
    CU(ctx, cudaMemcpyAsync(d_units, units, unit_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (n_tns) CU(ctx, cudaMemcpyAsync(d_tns, tns, (size_t)n_tns * sizeof(symgpu_aac_tns), cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemcpyAsync(d_spec, coeffs, spec_bytes, cudaMemcpyHostToDevice, ctx->stream));
    // planes no run writes (channel 1 of a mono stream, frames no run names) are defined as zero
    bool mono = false;
    uint64_t covered = 0;
    for (uint32_t r = 0; r < n_runs; ++r) {
        mono |= runs[r].channels == 1;
        covered += runs[r].n_frames;
    }
    if (mono || covered != n_frames) CU(ctx, cudaMemsetAsync(d_pcm, 0, spec_bytes, ctx->stream));
    // A pinned (device-mapped) output buffer is written by the kernel itself: its PCM stores cross PCIe while it is still
    // computing, and the D2H copy disappears (every plane is written when no stream is mono and the runs cover the batch).
    float* d_out = d_pcm;
    if (ctx->zero_copy && !mono && covered == n_frames) {
        cudaPointerAttributes at{};
        if (cudaPointerGetAttributes(&at, pcm) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer)
            d_out = static_cast<float*>(at.devicePointer);
        else
            cudaGetLastError();
    }
    s = symgpu_aac_synth_dev(ctx, d_units, d_tns, n_tns, d_spec, runs, n_runs, n_frames, d_out);
    if (s != SYMGPU_OK) return s;
    if (d_out == d_pcm) CU(ctx, cudaMemcpyAsync(pcm, d_pcm, spec_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return SYMGPU_OK;
}

// ---- table broadcast over a caller-supplied NCCL communicator (SURVEY 8b / 8e: the one collective of this path) -----------
// libnccl is not a link-time dependency: it is looked up in the process on first use (the host application, which made
// the communicator, has it loaded already).
symgpu_status symgpu_tables_broadcast(symgpu_ctx* ctx, void* nccl_comm, int root) {
    if (!ctx) return SYMGPU_ERR_ARG;
    if (!nccl_comm) return SYMGPU_OK; // single GPU: the locally built tables stand
    using BroadcastFn = int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t);
    static BroadcastFn bcast = nullptr;
    if (!bcast) {
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (h) bcast = reinterpret_cast<BroadcastFn>(dlsym(h, "ncclBroadcast"));
        if (!bcast) {
            std::snprintf(ctx->cuda_err, sizeof ctx->cuda_err, "symgpu_tables_broadcast: libnccl.so.2 / ncclBroadcast not found");
            return SYMGPU_ERR_UNSUPPORTED;
        }
    }
    DeviceGuard guard(ctx->device);
    symgpu_status s = ensure_codec_tables(ctx);
    if (s != SYMGPU_OK) return s;
    constexpr int kNcclUint8 = 1; // ncclDataType_t: ncclUint8
    int rc = bcast(ctx->d_mp3_tab, ctx->d_mp3_tab, sizeof(Mp3Tables), kNcclUint8, root, nccl_comm, ctx->stream);
    if (rc == 0) rc = bcast(ctx->d_codec_tab, ctx->d_codec_tab, sizeof(CodecTables), kNcclUint8, root, nccl_comm, ctx->stream);
    if (rc != 0) {
        std::snprintf(ctx->cuda_err, sizeof ctx->cuda_err, "ncclBroadcast failed with ncclResult_t %d", rc);
        return SYMGPU_ERR_CUDA;
    }
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    // the uniformly indexed tables also live in constant memory: refresh them from what arrived
    std::vector<unsigned char> blob(sizeof(Mp3Tables));
    CU(ctx, cudaMemcpy(blob.data(), ctx->d_mp3_tab, blob.size(), cudaMemcpyDeviceToHost));
    alignas(16) static thread_local Mp3Tables host_copy;
    std::memcpy(&host_copy, blob.data(), sizeof host_copy);
    CU(ctx, mp3_upload_const(host_copy, ctx->stream));
    CU(ctx, mp3v2_upload_const(host_copy, ctx->stream));
    return SYMGPU_OK;
}

// ---- Vorbis ------------------------------------------------------------------------------------

symgpu_status symgpu_vorbis_streams_set(symgpu_ctx* ctx, const symgpu_vorbis_stream* streams, uint32_t n_streams) {
    if (!ctx || !streams || n_streams == 0) return SYMGPU_ERR_ARG;
    for (uint32_t i = 0; i < n_streams; ++i) {
        const symgpu_vorbis_stream& s = streams[i];
        if (s.bs0_exp < 6 || s.bs1_exp > 13 || s.bs0_exp > s.bs1_exp) return SYMGPU_ERR_ARG; // lib.rs:404-417
        if (s.channels < 1 || s.channels > 2) return SYMGPU_ERR_UNSUPPORTED;
        if (s.coupled && s.channels != 2) return SYMGPU_ERR_ARG;
    }
    DeviceGuard guard(ctx->device);
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    symgpu_status st = ensure_codec_tables(ctx);
    if (st != SYMGPU_OK) return st;
    if (ctx->d_vorbis_streams) cudaFree(ctx->d_vorbis_streams);
    if (ctx->d_vorbis_states) cudaFree(ctx->d_vorbis_states);
    if (ctx->d_vorbis_gen) cudaFree(ctx->d_vorbis_gen);
    ctx->d_vorbis_streams = nullptr;
    ctx->d_vorbis_states = nullptr;
    ctx->d_vorbis_gen = nullptr;
    ctx->n_vorbis_streams = 0;
    CU(ctx, cudaMalloc(&ctx->d_vorbis_streams, (size_t)n_streams * sizeof *streams));
    CU(ctx, cudaMemcpy(ctx->d_vorbis_streams, streams, (size_t)n_streams * sizeof *streams, cudaMemcpyHostToDevice));
    const size_t bytes = (size_t)n_streams * 2 * kVorbisStateFloats * sizeof(float);
    CU(ctx, cudaMalloc(&ctx->d_vorbis_states, bytes));
    CU(ctx, cudaMemset(ctx->d_vorbis_states, 0, bytes));
    CU(ctx, cudaMalloc(&ctx->d_vorbis_gen, ((size_t)n_streams + 1) * sizeof(uint32_t)));
    CU(ctx, cudaMemset(ctx->d_vorbis_gen, 0, ((size_t)n_streams + 1) * sizeof(uint32_t)));
    ctx->h_vorbis_streams.assign(streams, streams + n_streams);
    ctx->n_vorbis_mc_streams = 0; // (symgpu_vorbis_mc_streams_set sets it again after this call)
    ctx->vorbis_cfg_epoch = (ctx->vorbis_cfg_epoch + 1) & 0xffu;
    ctx->chunk_key.clear();
    ctx->n_vorbis_streams = n_streams;
    return SYMGPU_OK;
}

symgpu_status symgpu_vorbis_floors_set(symgpu_ctx* ctx, const symgpu_vorbis_floor1* floors, uint32_t n_floors) {
    if (!ctx || !floors || n_floors == 0) return SYMGPU_ERR_ARG;
    std::vector<FloorAux> aux(n_floors);
    {
        static_assert(sizeof(FloorAux) == 72, "symgpu_vorbis_floors_levels writes 65 levels + the maximum + 6 pad bytes per setup");
        const symgpu_status chk = symgpu_vorbis_floors_levels(floors, n_floors, reinterpret_cast<uint8_t*>(aux.data()));
        if (chk != SYMGPU_OK) return chk;
    }
    DeviceGuard guard(ctx->device);
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->d_vorbis_floors) cudaFree(ctx->d_vorbis_floors);
    if (ctx->d_vorbis_floor_aux) cudaFree(ctx->d_vorbis_floor_aux);
    ctx->d_vorbis_floors = nullptr;
    ctx->d_vorbis_floor_aux = nullptr;
    ctx->n_vorbis_floors = 0;
    CU(ctx, cudaMalloc(&ctx->d_vorbis_floors, (size_t)n_floors * sizeof *floors));
    CU(ctx, cudaMemcpy(ctx->d_vorbis_floors, floors, (size_t)n_floors * sizeof *floors, cudaMemcpyHostToDevice));
    CU(ctx, cudaMalloc(&ctx->d_vorbis_floor_aux, (size_t)n_floors * sizeof(FloorAux)));
    CU(ctx, cudaMemcpy(ctx->d_vorbis_floor_aux, aux.data(), (size_t)n_floors * sizeof(FloorAux), cudaMemcpyHostToDevice));
    ctx->n_vorbis_floors = n_floors;
    return SYMGPU_OK;
}

symgpu_status symgpu_vorbis_stream_reset(symgpu_ctx* ctx, uint32_t stream) {
    if (!ctx) return SYMGPU_ERR_ARG;
    if (stream >= ctx->n_vorbis_streams) return SYMGPU_ERR_LIMIT;
    DeviceGuard guard(ctx->device);
    CU(ctx, cudaMemsetAsync(ctx->d_vorbis_states + (size_t)stream * 2 * kVorbisStateFloats, 0,
                            2 * kVorbisStateFloats * sizeof(float), ctx->stream));
    return SYMGPU_OK;
}

// The Vorbis launch behind the classic and the multichannel entry points: planes [p][pkt_ch][...] of which this launch works on
// ch_base, ch_base + 1; run.stream s stands for registered stream s * stream_mul + stream_add.
static symgpu_status vorbis_synth_dev_impl(symgpu_ctx* ctx, const symgpu_vorbis_unit* units, const uint16_t* floor_y, const float* residue,
                                           const symgpu_vorbis_run* runs, uint32_t n_runs, uint32_t n_packets, uint32_t slot, float* pcm,
                                           uint32_t pkt_ch, uint32_t ch_base, uint32_t stream_mul, uint32_t stream_add) {
    if (!ctx || !units || !floor_y || !residue || !runs || !pcm) return SYMGPU_ERR_ARG;
    if (n_packets == 0) return SYMGPU_OK;
    if (!ctx->d_vorbis_states || !ctx->d_vorbis_floors) return SYMGPU_ERR_LIMIT;
    DeviceGuard guard(ctx->device);
    std::vector<CodecChunk> chunks;
    uint64_t covered = 0;
    int max_bs1 = 6;
    auto reg = [&](uint32_t s) { return (uint64_t)s * stream_mul + stream_add; };
    for (uint32_t r = 0; r < n_runs; ++r)
        if (runs[r].n_packets && reg(runs[r].stream) < ctx->n_vorbis_streams)
            max_bs1 = std::max(max_bs1, (int)ctx->h_vorbis_streams[reg(runs[r].stream)].bs1_exp);
    uint32_t per_chunk = (uint32_t)vorbis_slots_for(max_bs1) - 1; // one slot is the packet before the chunk
    {
        // Short runs (a stream that submits a few packets per call): cut every run into equal chunks and size the CTA for them --
        // a run of 8 packets is two chunks of 4 in CTAs of 5 slots, not two chunks of 4 in CTAs of 8.  A function of the runs
        // alone, so a cached plan stays valid.
        uint64_t run_packets = 0, run_count = 0;
        for (uint32_t r = 0; r < n_runs; ++r)
            if (runs[r].n_packets) run_packets += runs[r].n_packets, ++run_count;
        const uint32_t mean = run_count ? (uint32_t)(run_packets / run_count) : 0;
        if (mean && mean <= 4 * per_chunk) {
            const uint32_t pieces = (mean + per_chunk - 1) / per_chunk;
            const uint32_t fit = (mean + pieces - 1) / pieces;
            if (fit >= 1 && fit < per_chunk) per_chunk = fit;
        }
    }
    const std::vector<unsigned char> key = chunk_key_of(0x564f5200u + ctx->vorbis_cfg_epoch + (stream_add << 8) + (stream_mul << 12), n_packets, slot, runs,
                                                        (size_t)n_runs * sizeof *runs);
    const bool reuse = key == ctx->chunk_key;
    for (uint32_t r = 0; r < n_runs && !reuse; ++r) {
        const symgpu_vorbis_run& run = runs[r];
        if (run.n_packets == 0) continue;
        if ((uint64_t)run.first_packet + run.n_packets > n_packets || run.reserved) return SYMGPU_ERR_ARG;
        if (reg(run.stream) >= ctx->n_vorbis_streams) return SYMGPU_ERR_LIMIT;
        const symgpu_vorbis_stream& cfg = ctx->h_vorbis_streams[reg(run.stream)];
        if ((1u << (cfg.bs1_exp - 1)) > slot) return SYMGPU_ERR_ARG; // slot too small for this stream
        covered += run.n_packets;
        split_even(run.n_packets, per_chunk, [&](uint32_t lo, uint32_t hi, bool first, bool last) {
            CodecChunk c{};
            c.first = run.first_packet + lo;
            c.stream = (uint32_t)reg(run.stream);
            c.count = (uint16_t)(hi - lo);
            c.flags = (uint8_t)((first ? kChunkLoadState : 0) | (last ? kChunkStoreState : 0));
            chunks.push_back(c);
        });
    }
    if (!reuse) {
        if (covered > n_packets) return SYMGPU_ERR_ARG; // runs may leave packets out, never overlap
        ctx->chunk_key.clear();
        symgpu_status s = upload_chunks(ctx, chunks);
        if (s != SYMGPU_OK) return s;
        ctx->chunk_key = key;
        ctx->cached_chunks = (int)chunks.size();
    }
    if (ctx->cached_chunks == 0) return SYMGPU_OK;
    VorbisArgs a{units, floor_y, residue, pcm, ctx->d_chunks, ctx->d_vorbis_streams, ctx->d_vorbis_floors,
                 ctx->d_vorbis_floor_aux, ctx->n_vorbis_floors, slot, pkt_ch, ch_base, ctx->d_vorbis_states, ctx->d_vorbis_gen,
                 ctx->d_vorbis_gen + ctx->n_vorbis_streams, ctx->d_codec_tab};
    CU(ctx, vorbis_launch(a, ctx->cached_chunks, max_bs1, (int)per_chunk + 1, ctx->stream));
    ctx->launches += 1;
    return SYMGPU_OK;
}

symgpu_status symgpu_vorbis_synth_dev(symgpu_ctx* ctx, const symgpu_vorbis_unit* units, const uint16_t* floor_y,
                                      const float* residue, const symgpu_vorbis_run* runs, uint32_t n_runs,
                                      uint32_t n_packets, uint32_t slot, float* pcm) {
    if (ctx && ctx->n_vorbis_mc_streams) return SYMGPU_ERR_ARG; // the context holds multichannel streams
    return vorbis_synth_dev_impl(ctx, units, floor_y, residue, runs, n_runs, n_packets, slot, pcm, 2, 0, 1, 0);
}

// ---- multichannel (symgpu_vorbis_mc_*) ---------------------------------------------------------------------------------
static constexpr uint32_t kMcPairs = SYMGPU_VORBIS_MAX_CHANNELS / 2; // registered pseudo-streams per multichannel stream

symgpu_status symgpu_vorbis_mc_streams_set(symgpu_ctx* ctx, const symgpu_vorbis_stream_mc* streams, uint32_t n_streams) {
    if (!ctx || !streams || n_streams == 0) return SYMGPU_ERR_ARG;
    std::vector<symgpu_vorbis_stream> pseudo((size_t)n_streams * kMcPairs);
    for (uint32_t i = 0; i < n_streams; ++i) {
        const symgpu_vorbis_stream_mc& m = streams[i];
        if (m.channels < 1 || m.channels > SYMGPU_VORBIS_MAX_CHANNELS) return SYMGPU_ERR_UNSUPPORTED;
        if (m.n_couplings > SYMGPU_VORBIS_MAX_COUPLINGS) return SYMGPU_ERR_UNSUPPORTED;
        for (int c = 0; c < m.n_couplings; ++c) // lib.rs:741-752: distinct channels inside the stream
            if (m.magnitude_ch[c] == m.angle_ch[c] || m.magnitude_ch[c] >= m.channels || m.angle_ch[c] >= m.channels) return SYMGPU_ERR_ARG;
        for (uint32_t k = 0; k < kMcPairs; ++k) {
            const int left = (int)m.channels - 2 * (int)k;
            // pairs beyond the stream's channels are placeholders no run ever names
            pseudo[(size_t)i * kMcPairs + k] = symgpu_vorbis_stream{m.bs0_exp, m.bs1_exp, (uint8_t)(left >= 2 ? 2 : 1), 0};
        }
    }
    symgpu_status s = symgpu_vorbis_streams_set(ctx, pseudo.data(), (uint32_t)pseudo.size());
    if (s != SYMGPU_OK) return s;
    DeviceGuard guard(ctx->device);
    if (ctx->d_vorbis_mc_streams) cudaFree(ctx->d_vorbis_mc_streams);
    ctx->d_vorbis_mc_streams = nullptr;
    CU(ctx, cudaMalloc(&ctx->d_vorbis_mc_streams, (size_t)n_streams * sizeof *streams));
    CU(ctx, cudaMemcpy(ctx->d_vorbis_mc_streams, streams, (size_t)n_streams * sizeof *streams, cudaMemcpyHostToDevice));
    ctx->h_vorbis_mc_streams.assign(streams, streams + n_streams);
    ctx->n_vorbis_mc_streams = n_streams;
    return SYMGPU_OK;
}

symgpu_status symgpu_vorbis_mc_stream_reset(symgpu_ctx* ctx, uint32_t stream) {
    if (!ctx) return SYMGPU_ERR_ARG;
    if (stream >= ctx->n_vorbis_mc_streams) return SYMGPU_ERR_LIMIT;
    for (uint32_t k = 0; k < kMcPairs; ++k) {
        const symgpu_status s = symgpu_vorbis_stream_reset(ctx, stream * kMcPairs + k);
        if (s != SYMGPU_OK) return s;
    }
    return SYMGPU_OK;
}

symgpu_status symgpu_vorbis_mc_synth_dev(symgpu_ctx* ctx, const symgpu_vorbis_unit_mc* units, const uint16_t* floor_y, float* residue,
                                         const symgpu_vorbis_run* runs, uint32_t n_runs, uint32_t n_packets, uint32_t channels, uint32_t slot,
                                         float* pcm) {
    if (!ctx || !units || !floor_y || !residue || !runs || !pcm) return SYMGPU_ERR_ARG;
    if (channels < 1 || channels > SYMGPU_VORBIS_MAX_CHANNELS) return SYMGPU_ERR_ARG;
    if (n_packets == 0) return SYMGPU_OK;
    if (!ctx->n_vorbis_mc_streams) return SYMGPU_ERR_LIMIT;
    DeviceGuard guard(ctx->device);
    // which stream a packet belongs to (0xffffffff: no run names it), and the channel pairs in use
    std::vector<uint32_t> stream_of((size_t)n_packets, 0xffffffffu);
    uint32_t max_ch = 0;
    for (uint32_t r = 0; r < n_runs; ++r) {
        const symgpu_vorbis_run& run = runs[r];
        if (run.n_packets == 0) continue;
        if ((uint64_t)run.first_packet + run.n_packets > n_packets || run.reserved) return SYMGPU_ERR_ARG;
        if (run.stream >= ctx->n_vorbis_mc_streams) return SYMGPU_ERR_LIMIT;
        if (ctx->h_vorbis_mc_streams[run.stream].channels > channels) return SYMGPU_ERR_ARG;
        max_ch = std::max<uint32_t>(max_ch, ctx->h_vorbis_mc_streams[run.stream].channels);
        for (uint32_t p = run.first_packet; p < run.first_packet + run.n_packets; ++p) stream_of[p] = run.stream;
    }
    const size_t need = (size_t)n_packets * (sizeof(uint32_t) + sizeof(symgpu_vorbis_unit));
    if (need > ctx->vorbis_mc_scratch_cap) {
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        if (ctx->d_vorbis_mc_scratch) cudaFree(ctx->d_vorbis_mc_scratch);
        ctx->d_vorbis_mc_scratch = nullptr;
        ctx->vorbis_mc_scratch_cap = 0;
        CU(ctx, cudaMalloc(&ctx->d_vorbis_mc_scratch, need + need / 2));
        ctx->vorbis_mc_scratch_cap = need + need / 2;
    }
    symgpu_vorbis_unit* d_pair_units = static_cast<symgpu_vorbis_unit*>(ctx->d_vorbis_mc_scratch);
    uint32_t* d_stream_of = reinterpret_cast<uint32_t*>(d_pair_units + n_packets);
    CU(ctx, cudaMemcpyAsync(d_stream_of, stream_of.data(), (size_t)n_packets * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream)); // stream_of is a local vector
    CU(ctx, vorbis_mc_decouple_launch(units, d_stream_of, ctx->d_vorbis_mc_streams, residue, n_packets, channels, slot, ctx->stream));
    ctx->launches += 1;
    for (uint32_t k = 0; 2 * k < max_ch; ++k) {
        // the runs of this pair: streams that have the pair's first channel
        std::vector<symgpu_vorbis_run> pr;
        for (uint32_t r = 0; r < n_runs; ++r)
            if (runs[r].n_packets && ctx->h_vorbis_mc_streams[runs[r].stream].channels > 2 * k) pr.push_back(runs[r]);
        if (pr.empty()) continue;
        CU(ctx, vorbis_mc_split_units_launch(units, n_packets, k, d_pair_units, ctx->stream));
        ctx->launches += 1;
        const symgpu_status s = vorbis_synth_dev_impl(ctx, d_pair_units, floor_y, residue, pr.data(), (uint32_t)pr.size(), n_packets, slot, pcm, channels,
                                                      2 * k, kMcPairs, k);
        if (s != SYMGPU_OK) return s;
    }
    return SYMGPU_OK;
}

symgpu_status symgpu_vorbis_mc_synth_host(symgpu_ctx* ctx, const symgpu_vorbis_unit_mc* units, const uint16_t* floor_y, const float* residue,
                                          const symgpu_vorbis_run* runs, uint32_t n_runs, uint32_t n_packets, uint32_t channels, uint32_t slot,
                                          float* pcm) {
    if (!ctx || !units || !floor_y || !residue || !runs || !pcm) return SYMGPU_ERR_ARG;
    if (channels < 1 || channels > SYMGPU_VORBIS_MAX_CHANNELS) return SYMGPU_ERR_ARG;
    if (n_packets == 0) return SYMGPU_OK;
    DeviceGuard guard(ctx->device);
    const size_t unit_bytes = (size_t)n_packets * sizeof(symgpu_vorbis_unit_mc);
    const size_t fy_bytes = ((size_t)n_packets * channels * 65 * sizeof(uint16_t) + 15) & ~(size_t)15;
    const size_t spec_bytes = (size_t)n_packets * channels * slot * sizeof(float);
    symgpu_status s = ensure_stage(ctx, 2 * spec_bytes + unit_bytes + fy_bytes);
    if (s != SYMGPU_OK) return s;
    char* base = static_cast<char*>(ctx->d_stage);
    float* d_res = reinterpret_cast<float*>(base);
    float* d_pcm = reinterpret_cast<float*>(base + spec_bytes);
    symgpu_vorbis_unit_mc* d_units = reinterpret_cast<symgpu_vorbis_unit_mc*>(base + 2 * spec_bytes);
    uint16_t* d_fy = reinterpret_cast<uint16_t*>(base + 2 * spec_bytes + unit_bytes);
    CU(ctx, cudaMemcpyAsync(d_units, units, unit_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemcpyAsync(d_fy, floor_y, (size_t)n_packets * channels * 65 * sizeof(uint16_t), cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemcpyAsync(d_res, residue, spec_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemsetAsync(d_pcm, 0, spec_bytes, ctx->stream)); // packets fill only (prev_n + n) / 4 of their slot
    s = symgpu_vorbis_mc_synth_dev(ctx, d_units, d_fy, d_res, runs, n_runs, n_packets, channels, slot, d_pcm);
    if (s != SYMGPU_OK) return s;
    CU(ctx, cudaMemcpyAsync(pcm, d_pcm, spec_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return SYMGPU_OK;
}

symgpu_status symgpu_vorbis_synth_host(symgpu_ctx* ctx, const symgpu_vorbis_unit* units, const uint16_t* floor_y,
                                       const float* residue, const symgpu_vorbis_run* runs, uint32_t n_runs,
                                       uint32_t n_packets, uint32_t slot, float* pcm) {
    if (!ctx || !units || !floor_y || !residue || !runs || !pcm) return SYMGPU_ERR_ARG;
    if (n_packets == 0) return SYMGPU_OK;
    DeviceGuard guard(ctx->device);
    const size_t unit_bytes = (size_t)n_packets * sizeof(symgpu_vorbis_unit);
    const size_t fy_bytes = ((size_t)n_packets * 2 * 65 * sizeof(uint16_t) + 15) & ~(size_t)15;
    const size_t spec_bytes = (size_t)n_packets * 2 * slot * sizeof(float);
    symgpu_status s = ensure_stage(ctx, 2 * spec_bytes + unit_bytes + fy_bytes);
    if (s != SYMGPU_OK) return s;
    char* base = static_cast<char*>(ctx->d_stage);
    float* d_res = reinterpret_cast<float*>(base);
    float* d_pcm = reinterpret_cast<float*>(base + spec_bytes);
    symgpu_vorbis_unit* d_units = reinterpret_cast<symgpu_vorbis_unit*>(base + 2 * spec_bytes);
    uint16_t* d_fy = reinterpret_cast<uint16_t*>(base + 2 * spec_bytes + unit_bytes);
    CU(ctx, cudaMemcpyAsync(d_units, units, unit_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemcpyAsync(d_fy, floor_y, (size_t)n_packets * 2 * 65 * sizeof(uint16_t), cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemcpyAsync(d_res, residue, spec_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemsetAsync(d_pcm, 0, spec_bytes, ctx->stream)); // packets fill only (prev_n + n) / 4 of their slot
    s = symgpu_vorbis_synth_dev(ctx, d_units, d_fy, d_res, runs, n_runs, n_packets, slot, d_pcm);
    if (s != SYMGPU_OK) return s;
    CU(ctx, cudaMemcpyAsync(pcm, d_pcm, spec_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return SYMGPU_OK;
}

// ---- FLAC integer restoration (SURVEY 8f N4) --------------------------------------------------------------
symgpu_status symgpu_flac_restore_dev(symgpu_ctx* ctx, const symgpu_flac_frame* frames, uint32_t n_frames,
                                      const symgpu_flac_subframe* subframes, uint32_t n_subframes, int32_t* samples,
                                      size_t n_samples) {
    if (!ctx || !frames || !subframes || !samples) return SYMGPU_ERR_ARG;
    if (n_frames == 0 && n_subframes == 0) return SYMGPU_OK;
    DeviceGuard guard(ctx->device);
    CU(ctx, flac_launch(frames, n_frames, subframes, n_subframes, samples, n_samples, ctx->stream));
    ctx->launches += (n_subframes ? 1 : 0) + (n_frames ? 1 : 0);
    return SYMGPU_OK;
}

} // extern "C"

// What read_subframe / decode_linear / decode_fixed_linear refuse (decoder.rs:335-347, :429-431, :456-474,
// :503-505) is refused here; the kernels additionally never leave the buffer.
static symgpu_status flac_descriptors_check(const symgpu_flac_frame* frames, uint32_t n_frames, const symgpu_flac_subframe* subframes,
                                            uint32_t n_subframes, size_t n_samples) {
    for (uint32_t k = 0; k < n_subframes; ++k) {
        const symgpu_flac_subframe& sf = subframes[k];
        if (sf.n == 0 || sf.offset > n_samples || sf.n > n_samples - sf.offset) return SYMGPU_ERR_ARG;
        if (sf.type > SYMGPU_FLAC_LPC || sf.wasted > 32) return SYMGPU_ERR_DECODE;
        if (sf.type == SYMGPU_FLAC_FIXED && (sf.order > 4 || sf.order > sf.n)) return SYMGPU_ERR_DECODE;
        if (sf.type == SYMGPU_FLAC_LPC && (sf.order < 1 || sf.order > 32 || sf.order > sf.n)) return SYMGPU_ERR_DECODE;
        if (sf.type == SYMGPU_FLAC_LPC && sf.shift > 15) return SYMGPU_ERR_UNSUPPORTED;
    }
    for (uint32_t f = 0; f < n_frames; ++f) {
        const symgpu_flac_frame& fr = frames[f];
        if (fr.channels < 1 || fr.channels > 8 || (uint64_t)fr.first_subframe + fr.channels > n_subframes) return SYMGPU_ERR_ARG;
        if (fr.bits_per_sample < 1 || fr.bits_per_sample > 32) return SYMGPU_ERR_DECODE;
        if (fr.assignment > SYMGPU_FLAC_RIGHT_SIDE) return SYMGPU_ERR_DECODE;
        if (fr.assignment != SYMGPU_FLAC_INDEPENDENT &&
            (fr.channels != 2 || subframes[fr.first_subframe].n != subframes[fr.first_subframe + 1].n))
            return SYMGPU_ERR_DECODE;
    }
    return SYMGPU_OK;
}

extern "C" {

symgpu_status symgpu_flac_restore_host(symgpu_ctx* ctx, const symgpu_flac_frame* frames, uint32_t n_frames,
                                       const symgpu_flac_subframe* subframes, uint32_t n_subframes, int32_t* samples,
                                       size_t n_samples) {
    if (!ctx || !frames || !subframes || !samples) return SYMGPU_ERR_ARG;
    symgpu_status s = flac_descriptors_check(frames, n_frames, subframes, n_subframes, n_samples);
    if (s != SYMGPU_OK) return s;
    if (n_frames == 0 && n_subframes == 0) return SYMGPU_OK;
    DeviceGuard guard(ctx->device);
    const size_t sample_bytes = (n_samples * sizeof(int32_t) + 255) & ~(size_t)255;
    const size_t sub_bytes = ((size_t)n_subframes * sizeof(symgpu_flac_subframe) + 255) & ~(size_t)255;
    const size_t frame_bytes = (size_t)n_frames * sizeof(symgpu_flac_frame);
    s = ensure_stage(ctx, sample_bytes + sub_bytes + frame_bytes);
    if (s != SYMGPU_OK) return s;
    char* base = static_cast<char*>(ctx->d_stage);
    int32_t* d_samples = reinterpret_cast<int32_t*>(base);
    symgpu_flac_subframe* d_subs = reinterpret_cast<symgpu_flac_subframe*>(base + sample_bytes);
    symgpu_flac_frame* d_frames = reinterpret_cast<symgpu_flac_frame*>(base + sample_bytes + sub_bytes);
    CU(ctx, cudaMemcpyAsync(d_samples, samples, n_samples * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemcpyAsync(d_subs, subframes, (size_t)n_subframes * sizeof(symgpu_flac_subframe), cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemcpyAsync(d_frames, frames, frame_bytes, cudaMemcpyHostToDevice, ctx->stream));
    s = symgpu_flac_restore_dev(ctx, d_frames, n_frames, d_subs, n_subframes, d_samples, n_samples);
    if (s != SYMGPU_OK) return s;
    CU(ctx, cudaMemcpyAsync(samples, d_samples, n_samples * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return SYMGPU_OK;
}

// ---- FLAC restoration + output stage (FromSample<i32>, conv.rs:514-532) -------------------------------------------------------
symgpu_status symgpu_flac_decode_dev(symgpu_ctx* ctx, const symgpu_flac_frame* frames, uint32_t n_frames,
                                     const symgpu_flac_subframe* subframes, uint32_t n_subframes, int32_t* samples,
                                     size_t n_samples, const uint64_t* dst, int format, void* out, size_t out_samples) {
    if (!ctx || !frames || !subframes || !samples || !dst || !out) return SYMGPU_ERR_ARG;
    if (symgpu_sample_bytes(format) == 0) return SYMGPU_ERR_ARG;
    if (n_frames == 0 && n_subframes == 0) return SYMGPU_OK;
    DeviceGuard guard(ctx->device);
    CU(ctx, flac_decode_launch(frames, n_frames, subframes, n_subframes, samples, n_samples, dst, format, out, out_samples, ctx->stream));
    ctx->launches += (n_subframes ? 1 : 0) + (n_frames ? 1 : 0);
    return SYMGPU_OK;
}

symgpu_status symgpu_flac_decode_host(symgpu_ctx* ctx, const symgpu_flac_frame* frames, uint32_t n_frames,
                                      const symgpu_flac_subframe* subframes, uint32_t n_subframes, const int32_t* samples,
                                      size_t n_samples, const uint64_t* dst, int format, void* out, size_t out_bytes) {
    if (!ctx || !frames || !subframes || !samples || !dst || !out) return SYMGPU_ERR_ARG;
    const size_t sb = symgpu_sample_bytes(format);
    if (sb == 0) return SYMGPU_ERR_ARG;
    symgpu_status s = flac_descriptors_check(frames, n_frames, subframes, n_subframes, n_samples);
    if (s != SYMGPU_OK) return s;
    // Interleaving needs one block size per frame, and every frame's samples inside `out`.
    const uint64_t out_samples = out_bytes / sb;
    for (uint32_t f = 0; f < n_frames; ++f) {
        const symgpu_flac_frame& fr = frames[f];
        const uint32_t n = subframes[fr.first_subframe].n;
        for (uint32_t c = 1; c < fr.channels; ++c)
            if (subframes[fr.first_subframe + c].n != n) return SYMGPU_ERR_DECODE;
        if (dst[f] > out_samples || (uint64_t)n * fr.channels > out_samples - dst[f]) return SYMGPU_ERR_LIMIT;
    }
    if (n_frames == 0 && n_subframes == 0) return SYMGPU_OK;
    DeviceGuard guard(ctx->device);
    const size_t sample_bytes = (n_samples * sizeof(int32_t) + 255) & ~(size_t)255;
    const size_t sub_bytes = ((size_t)n_subframes * sizeof(symgpu_flac_subframe) + 255) & ~(size_t)255;
    const size_t frame_bytes = ((size_t)n_frames * sizeof(symgpu_flac_frame) + 255) & ~(size_t)255;
    const size_t dst_bytes = ((size_t)n_frames * sizeof(uint64_t) + 255) & ~(size_t)255;
    const size_t packed = out_samples * sb;
    s = ensure_stage(ctx, sample_bytes + sub_bytes + frame_bytes + dst_bytes + packed);
    if (s != SYMGPU_OK) return s;
    char* base = static_cast<char*>(ctx->d_stage);
    int32_t* d_samples = reinterpret_cast<int32_t*>(base);
    symgpu_flac_subframe* d_subs = reinterpret_cast<symgpu_flac_subframe*>(base + sample_bytes);
    symgpu_flac_frame* d_frames = reinterpret_cast<symgpu_flac_frame*>(base + sample_bytes + sub_bytes);
    uint64_t* d_dst = reinterpret_cast<uint64_t*>(base + sample_bytes + sub_bytes + frame_bytes);
    void* d_out = base + sample_bytes + sub_bytes + frame_bytes + dst_bytes;
    CU(ctx, cudaMemcpyAsync(d_samples, samples, n_samples * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemcpyAsync(d_subs, subframes, (size_t)n_subframes * sizeof(symgpu_flac_subframe), cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemcpyAsync(d_frames, frames, (size_t)n_frames * sizeof(symgpu_flac_frame), cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemcpyAsync(d_dst, dst, (size_t)n_frames * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemsetAsync(d_out, 0, packed, ctx->stream)); // samples no frame writes are zero
    s = symgpu_flac_decode_dev(ctx, d_frames, n_frames, d_subs, n_subframes, d_samples, n_samples, d_dst, format, d_out, out_samples);
    if (s != SYMGPU_OK) return s;
    CU(ctx, cudaMemcpyAsync(out, d_out, packed, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return SYMGPU_OK;
}

} // extern "C"
