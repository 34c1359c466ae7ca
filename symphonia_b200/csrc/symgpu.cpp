// libsymgpu.so -- implementation of the C ABI in include/symgpu.h.
//
// There is deliberately no CPU implementation of the synthesis path in this library: every entry
// point that produces PCM launches the CUDA kernels, and context creation fails loudly when no
// CUDA device is usable.
#include <cuda_runtime.h>
#include <sched.h>

#include <algorithm>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "ctx.h"
#include "pack_kernel.h"


using namespace symgpu;
using namespace symgpu_detail;

namespace {

// The work plan of one launch, as the kernel reads it: a header of n_ctas + 1 tile indices followed by
// the tiles (mp3_kernel.h).  The header is padded to whole 16-byte entries so that the tiles stay aligned.
struct Mp3Plan {
    std::vector<Mp3Tile> buf; // [header entries][tiles]
    int hdr = 0;              // header size in Mp3Tile entries
    int n_tiles = 0;
    int n_ctas = 0;
    bool multi = false;       // some group holds more than one tile
    bool v2 = false;          // laid out for the second-generation kernel: n_ctas counts SHARES (one per warp)
};

// Cuts the caller's runs into CHAINS of tiles, one chain per CTA of the persistent grid: the batch's
// granules (in run order) are split into n_ctas contiguous shares; inside a share every run segment is
// cut into equal tiles that hand their state on through shared memory.  Only a segment that starts
// inside a run recomputes the 2-granule halo.  Returns SYMGPU_OK or an argument / limit error.
// T: units (granules; whole frames for Layer I / II) per tile; T_halo: limit for a tile that recomputes its halo;
// group: mark groups of tiles for the Layer III kernel.
symgpu_status build_plan_for(int grid, uint32_t T, uint32_t T_halo, bool group, uint32_t n_streams, const symgpu_mp3_run* runs,
                             uint32_t n_runs, uint32_t n_frames, Mp3Plan& plan, bool whole_batch) {
    uint64_t covered = 0, total_gran = 0, plain_tiles = 0;
    for (uint32_t r = 0; r < n_runs; ++r) {
        const symgpu_mp3_run& run = runs[r];
        const int gpf = run.granules_per_frame ? run.granules_per_frame : 2;
        const int n_ch = run.channels ? run.channels : 2;
        if (gpf < 1 || gpf > 2 || n_ch < 1 || n_ch > 2 || run.reserved != 0) return SYMGPU_ERR_ARG;
        if (run.n_frames == 0) continue;
        if ((uint64_t)run.first_frame + run.n_frames > n_frames) return SYMGPU_ERR_ARG;
        if (run.stream >= n_streams) return SYMGPU_ERR_LIMIT;
        covered += run.n_frames;
        const uint64_t n_gran = (uint64_t)run.n_frames * (uint32_t)gpf;
        total_gran += n_gran;
        plain_tiles += (n_gran + T - 1) / T;
    }
    if (whole_batch && covered != n_frames) return SYMGPU_ERR_ARG; // runs must tile the batch exactly
    plan.multi = false;
    plan.n_ctas = (int)std::min<uint64_t>((uint64_t)grid, std::max<uint64_t>(plain_tiles, 1));
    plan.hdr = (plan.n_ctas + 1 + 3) / 4;
    plan.buf.assign((size_t)plan.hdr, Mp3Tile{});
    std::vector<uint32_t> first((size_t)plan.n_ctas + 1, 0);

    uint64_t pos = 0;  // granules of earlier runs
    int cta = 0;       // share being filled
    uint32_t n_tiles = 0;
    // End of share `c` in batch granules; a cut that would leave fewer than 2 granules of a run before
    // it moves to the run's start (a halo needs two earlier granules of the same run in the batch).
    auto share_end = [&](int c) { return total_gran * (uint64_t)(c + 1) / (uint64_t)plan.n_ctas; };
    for (uint32_t r = 0; r < n_runs; ++r) {
        const symgpu_mp3_run& run = runs[r];
        if (run.n_frames == 0) continue;
        const uint32_t gpf = run.granules_per_frame ? run.granules_per_frame : 2;
        const uint32_t n_ch = run.channels ? run.channels : 2;
        const uint32_t n_gran = run.n_frames * gpf;
        uint32_t q0 = 0;
        while (q0 < n_gran) {
            // this segment ends at the share boundary or at the end of the run
            while (cta + 1 < plan.n_ctas && share_end(cta) <= pos + q0) first[(size_t)++cta] = n_tiles;
            uint32_t q1 = n_gran;
            if (cta + 1 < plan.n_ctas) {
                const uint64_t cut = share_end(cta);
                if (cut < pos + n_gran) {
                    q1 = (uint32_t)(cut - pos);
                    if (q1 < q0 + 1) q1 = q0 + 1;
                    if (q1 < 2) q1 = n_gran < 2 ? n_gran : 2; // keep two granules before any mid-run cut
                    if (n_gran - q1 < 1) q1 = n_gran;
                }
            }
            const bool halo = q0 != 0;
            const uint32_t len = q1 - q0;
            // equal tiles; the first tile of a halo segment is capped at T_halo granules
            uint32_t n_t = (len + T - 1) / T;
            if (halo) n_t = len <= T_halo ? 1 : 1 + (len - T_halo + T - 1) / T;
            const uint32_t head = halo ? std::min(T_halo, (len + n_t - 1) / n_t) : 0; // size of the halo tile
            uint32_t a0 = q0;
            for (uint32_t k = 0; k < n_t; ++k) {
                uint32_t a1;
                if (!halo) a1 = q0 + (uint32_t)(((uint64_t)len * (k + 1)) / n_t);
                else if (n_t == 1) a1 = q1;
                else a1 = q0 + head + (uint32_t)(((uint64_t)(len - head) * k) / (n_t - 1));
                Mp3Tile t{};
                t.first_frame = run.first_frame + a0 / gpf;
                t.first_gr = (uint16_t)(a0 % gpf);
                t.stream = run.stream;
                t.n_granules = (uint16_t)(a1 - a0);
                t.gpf = (uint8_t)gpf;
                t.n_ch = (uint8_t)n_ch;
                uint8_t fl = 0;
                if (k == 0) fl |= halo ? 0 : kTileLoadState;
                else fl |= kTileCarryIn;
                if (k + 1 < n_t) fl |= kTileCarryOut;
                else if (a1 == n_gran) fl |= kTileStoreState;
                t.flags = fl;
                plan.buf.push_back(t);
                ++n_tiles;
                a0 = a1;
            }
            q0 = q1;
            if (q0 < n_gran) first[(size_t)++cta] = n_tiles; // the rest of the run belongs to the next share
        }
        pos += n_gran;
    }
    while (cta < plan.n_ctas) first[(size_t)++cta] = n_tiles;
    plan.n_tiles = (int)n_tiles;
    // Groups: consecutive tiles of a chain that the CTA processes together (mp3_kernel.h).  Greedy: a tile
    // joins the open group unless the group would exceed its job / region / tile budget, the tile takes its
    // state from the previous group (kTileCarryIn starts a group) or the previous tile hands its state on
    // (kTileCarryOut ends one).
    if (group) {
        const int n_warps = mp3_cta_warps(); // granule jobs per group
        Mp3Tile* tiles = plan.buf.data() + plan.hdr;
        for (int c = 0; c < plan.n_ctas; ++c) {
            int jobs = 0, regions = 0, count = 0;
            for (uint32_t i = first[(size_t)c]; i < first[(size_t)c + 1]; ++i) {
                Mp3Tile& t = tiles[i];
                const int tj = t.n_granules + ((t.flags & (kTileLoadState | kTileCarryIn)) ? 0 : 2);
                const int tr = t.n_granules + 1;
                const bool fits = count > 0 && count < kMp3GroupTiles && jobs + tj <= n_warps && regions + tr <= kMp3GroupRegions &&
                                  !(t.flags & kTileCarryIn) && !(tiles[i - 1].flags & kTileCarryOut);
                if (!fits && count > 0) {
                    tiles[i - 1].flags |= kTileGroupEnd;
                    jobs = regions = count = 0;
                }
                if (fits) plan.multi = true;
                jobs += tj;
                regions += tr;
                ++count;
            }
            if (count > 0) tiles[first[(size_t)c + 1] - 1].flags |= kTileGroupEnd;
        }
    }
    std::memcpy(plan.buf.data(), first.data(), first.size() * sizeof(uint32_t));
    return SYMGPU_OK;
}


// ---- launch plan of the second-generation kernel (mp3_kernel_v2.cu) ------------------------------------
// The batch's granules, in run order, are cut into at most `max_shares` SHARES, one per warp of the launch.
// A cut prefers a run boundary (no halo) when one is within a quarter of a share of the ideal position, and
// never leaves fewer than two granules of the run before it (a halo recomputes two earlier granules, which
// must be in the batch).  Same container as the first-generation plan: a header of n_shares + 1 tile
// offsets (padded to 16-byte entries) followed by the tiles; a tile is one run segment of one share.
symgpu_status build_plan_v2_for(int max_shares, uint32_t n_streams, const symgpu_mp3_run* runs, uint32_t n_runs,
                                uint32_t n_frames, Mp3Plan& plan, bool whole_batch) {
    constexpr uint64_t kMinShare = 4;     // granules: below this a share is not worth its halo
    constexpr uint32_t kMaxTile = 32768;  // Mp3Tile::n_granules is 16 bits
    uint64_t covered = 0, total_gran = 0;
    for (uint32_t r = 0; r < n_runs; ++r) {
        const symgpu_mp3_run& run = runs[r];
        const int gpf = run.granules_per_frame ? run.granules_per_frame : 2;
        const int n_ch = run.channels ? run.channels : 2;
        if (gpf < 1 || gpf > 2 || n_ch < 1 || n_ch > 2 || run.reserved != 0) return SYMGPU_ERR_ARG;
        if (run.n_frames == 0) continue;
        if ((uint64_t)run.first_frame + run.n_frames > n_frames) return SYMGPU_ERR_ARG;
        if (run.stream >= n_streams) return SYMGPU_ERR_LIMIT;
        covered += run.n_frames;
        total_gran += (uint64_t)run.n_frames * (uint32_t)gpf;
    }
    if (whole_batch && covered != n_frames) return SYMGPU_ERR_ARG; // runs must tile the batch exactly
    if (max_shares < 1) return SYMGPU_ERR_ARG;
    const uint64_t n_shares = std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)max_shares, total_gran / kMinShare));
    plan.multi = false;
    plan.n_ctas = (int)n_shares; // shares, for this plan
    plan.hdr = (int)((n_shares + 1 + 3) / 4);
    plan.buf.assign((size_t)plan.hdr, Mp3Tile{});
    std::vector<uint32_t> first((size_t)n_shares + 1, 0);
    const uint64_t tol = total_gran / n_shares / 4; // snap distance

    uint64_t pos = 0;    // granules of earlier runs
    uint64_t share = 0;  // share being filled
    uint32_t n_tiles = 0;
    auto ideal_end = [&](uint64_t c) { return total_gran * (c + 1) / n_shares; };
    for (uint32_t r = 0; r < n_runs; ++r) {
        const symgpu_mp3_run& run = runs[r];
        if (run.n_frames == 0) continue;
        const uint32_t gpf = run.granules_per_frame ? run.granules_per_frame : 2;
        const uint32_t n_ch = run.channels ? run.channels : 2;
        const uint64_t n_gran = (uint64_t)run.n_frames * gpf;
        uint64_t q0 = 0;
        while (q0 < n_gran) {
            // shares whose ideal end lies at or before this position are closed (possibly empty)
            while (share + 1 < n_shares) {
                const uint64_t cut = ideal_end(share);
                bool close = cut <= pos + q0;
                // a cut just behind this run's start snaps back to the start
                if (!close && q0 == 0 && cut < pos + n_gran && (cut - pos <= tol || cut - pos < 2)) close = true;
                if (!close) break;
                first[(size_t)++share] = n_tiles;
            }
            uint64_t q1 = n_gran;
            if (share + 1 < n_shares) {
                const uint64_t cut = ideal_end(share);
                if (cut < pos + n_gran) {
                    q1 = cut - pos;            // > q0, and >= 2 or it would have snapped to the run start above
                    if (q1 <= q0) q1 = q0 + 1;
                    if (q1 < 2) q1 = 2;
                    if (n_gran - q1 <= tol || q1 >= n_gran) q1 = n_gran; // a cut just before the run's end snaps to the end
                }
            }
            bool first_piece = true;
            for (uint64_t a0 = q0; a0 < q1;) { // pieces of at most kMaxTile granules, the state stays in the warp between them
                const uint64_t a1 = std::min<uint64_t>(q1, a0 + kMaxTile);
                Mp3Tile t{};
                t.first_frame = run.first_frame + (uint32_t)(a0 / gpf);
                t.first_gr = (uint16_t)(a0 % gpf);
                t.stream = run.stream;
                t.n_granules = (uint16_t)(a1 - a0);
                t.gpf = (uint8_t)gpf;
                t.n_ch = (uint8_t)n_ch;
                uint8_t fl = 0;
                if (!first_piece) fl |= kTileCarryIn;
                else if (a0 == 0) fl |= kTileLoadState;
                if (a1 < q1) fl |= kTileCarryOut;
                else if (a1 == n_gran) fl |= kTileStoreState;
                t.flags = fl;
                plan.buf.push_back(t);
                ++n_tiles;
                first_piece = false;
                a0 = a1;
            }
            q0 = q1;
            if (q0 < n_gran && share + 1 < n_shares) first[(size_t)++share] = n_tiles; // the rest of the run goes to the next share
        }
        pos += n_gran;
    }
    while (share < n_shares) first[(size_t)++share] = n_tiles;
    plan.n_tiles = (int)n_tiles;
    std::memcpy(plan.buf.data(), first.data(), first.size() * sizeof(uint32_t));
    return SYMGPU_OK;
}

symgpu_status build_plan(symgpu_ctx* ctx, const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames, Mp3Plan& plan,
                         bool whole_batch = true) {
    cudaError_t ce = cudaSuccess;
    // Which kernel: the second generation (one warp per share, state in registers) wins where runs are short -- the serving
    // shape, a frame or two per stream: 143 us against 219 us for 8192 one-frame streams -- the first generation (CTA-wide
    // tiles of 16 consecutive granules, one halo per CTA chain) with the packed window phase where runs are long: 128 us
    // against 135 us for 64 streams x 128 frames (profiles/r02_mp3_variants_log.txt).
    bool v2 = ctx->mp3_kernel_mode == 2;
    if (ctx->mp3_kernel_mode == 0) {
        uint64_t gran = 0, n = 0;
        for (uint32_t r = 0; r < n_runs; ++r)
            if (runs[r].n_frames) {
                gran += (uint64_t)runs[r].n_frames * (runs[r].granules_per_frame == 1 ? 1u : 2u);
                ++n;
            }
        v2 = n > 0 && gran < 16 * n; // fewer than 16 granules per run on average
    }
    plan.v2 = v2;
    if (v2) {
        const int n_sm = mp3v2_sm_count(&ce);
        if (ce != cudaSuccess || n_sm <= 0) return cuda_fail(ctx, ce, "mp3v2_sm_count");
        return build_plan_v2_for(n_sm * mp3v2_ctas_per_sm() * mp3v2_cta_warps(), ctx->n_mp3_streams, runs, n_runs, n_frames, plan, whole_batch);
    }
    const int grid = mp3_grid_size(&ce);
    if (ce != cudaSuccess || grid <= 0) return cuda_fail(ctx, ce, "mp3_grid_size");
    return build_plan_for(grid, (uint32_t)mp3_tile_granules(), (uint32_t)mp3_halo_tile_granules(), true, ctx->n_mp3_streams, runs,
                          n_runs, n_frames, plan, whole_batch);
}

// Launches the Layer III kernel the context is configured for over a plan whose entries sit at `d_plan`.
cudaError_t launch_plan(symgpu_ctx* ctx, const Mp3Tile* d_plan, int hdr, int n_tiles, int n_ctas, bool multi, bool v2,
                        const symgpu_mp3_gc* units, const float* spectra, float* pcm, cudaStream_t stream) {
    if (v2) {
        cudaError_t ce = cudaSuccess;
        const int n_sm = mp3v2_sm_count(&ce);
        if (ce != cudaSuccess) return ce;
        const int n_shares = n_ctas; // the v2 plan counts shares
        const Mp3V2Args a{units, spectra, pcm, reinterpret_cast<const uint32_t*>(d_plan), d_plan + hdr, n_tiles, n_shares,
                          ctx->d_mp3_states, ctx->d_mp3_gen, ctx->d_mp3_gen + ctx->n_mp3_streams, ctx->d_mp3_tab, 1.0f, -1.0f};
        // many short run segments per share = the serving shape (a frame or two per stream)
        const bool short_runs = n_tiles >= 2 * n_shares;
        return mp3v2_launch(a, std::min(n_sm * mp3v2_ctas_per_sm(), n_shares), stream, short_runs);
    }
    const Mp3Args a{units, spectra, pcm, reinterpret_cast<const uint32_t*>(d_plan), d_plan + hdr, n_tiles, n_ctas, multi ? 1 : 0,
                    ctx->d_mp3_states, ctx->d_mp3_gen, ctx->d_mp3_gen + ctx->n_mp3_streams, ctx->d_mp3_tab, 1.0f};
    return mp3_launch(a, stream);
}

// Makes room for `entries` plan entries in the device / pinned host buffers.
symgpu_status reserve_plan(symgpu_ctx* ctx, size_t entries) {
    ctx->slice_plans_valid = false; // whoever asks for room is about to rewrite d_tiles
    CU(ctx, cudaStreamSynchronize(ctx->stream)); // the previous launch may still read d_tiles; h_tiles is rewritten
    if (entries <= ctx->tiles_cap) return SYMGPU_OK;
    if (ctx->d_tiles) cudaFree(ctx->d_tiles);
    if (ctx->h_tiles) cudaFreeHost(ctx->h_tiles);
    ctx->d_tiles = nullptr;
    ctx->h_tiles = nullptr;
    ctx->tiles_cap = 0;
    const size_t cap = entries + entries / 2 + 64;
    CU(ctx, cudaMalloc(&ctx->d_tiles, cap * sizeof(Mp3Tile)));
    CU(ctx, cudaMallocHost(&ctx->h_tiles, cap * sizeof(Mp3Tile)));
    ctx->tiles_cap = cap;
    return SYMGPU_OK;
}

symgpu_status ensure_plan(symgpu_ctx* ctx, const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames) {
    if (ctx->cached_frames == n_frames && ctx->cached_runs.size() == n_runs &&
        (n_runs == 0 || std::memcmp(ctx->cached_runs.data(), runs, n_runs * sizeof *runs) == 0))
        return SYMGPU_OK;
    Mp3Plan plan;
    symgpu_status s = build_plan(ctx, runs, n_runs, n_frames, plan);
    if (s != SYMGPU_OK) return s;
    s = reserve_plan(ctx, plan.buf.size());
    if (s != SYMGPU_OK) return s;
    std::memcpy(ctx->h_tiles, plan.buf.data(), plan.buf.size() * sizeof(Mp3Tile));
    CU(ctx, cudaMemcpyAsync(ctx->d_tiles, ctx->h_tiles, plan.buf.size() * sizeof(Mp3Tile), cudaMemcpyHostToDevice, ctx->stream));
    ctx->cached_runs.assign(runs, runs + n_runs);
    ctx->cached_frames = n_frames;
    ctx->cached_tiles = plan.n_tiles;
    ctx->cached_hdr = plan.hdr;
    ctx->cached_ctas = plan.n_ctas;
    ctx->cached_multi = plan.multi;
    ctx->cached_v2 = plan.v2;
    return SYMGPU_OK;
}

} // namespace


// ---- NUMA placement ------------------------------------------------------------------------------------------------
// A B200 node has its GPUs behind two sockets; a rank whose thread (and therefore its first-touched pinned buffers)
// sits on the far socket pays for every H2D / D2H byte twice on the inter-socket link, and eight ranks doing so at once
// is what bent round 1's end-to-end scaling (0.62 at 8 GPUs).  Parses "0-3,8,10-11" style lists.
static bool parse_cpulist(const char* text, cpu_set_t* set) {
    CPU_ZERO(set);
    int n = 0;
    const char* p = text;
    while (*p) {
        char* end = nullptr;
        const long a = std::strtol(p, &end, 10);
        if (end == p) break;
        long b = a;
        p = end;
        if (*p == '-') {
            b = std::strtol(p + 1, &end, 10);
            if (end == p + 1) return false;
            p = end;
        }
        for (long c = a; c <= b && c < CPU_SETSIZE; ++c) {
            CPU_SET((int)c, set);
            ++n;
        }
        while (*p == ',' || *p == '\n' || *p == ' ') ++p;
    }
    return n > 0;
}

static bool read_small_file(const char* path, char* buf, size_t cap) {
    std::FILE* f = std::fopen(path, "r");
    if (!f) return false;
    const size_t n = std::fread(buf, 1, cap - 1, f);
    std::fclose(f);
    buf[n] = 0;
    return n > 0;
}

extern "C" int symgpu_numa_node_of_device(int device) {
    char bdf[32] = {0};
    if (cudaDeviceGetPCIBusId(bdf, sizeof bdf, device) != cudaSuccess) return -1;
    for (char* c = bdf; *c; ++c) *c = (char)std::tolower((unsigned char)*c);
    char path[128], buf[64];
    std::snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bdf);
    if (!read_small_file(path, buf, sizeof buf)) return -1;
    return std::atoi(buf); // -1 when the platform does not say
}

extern "C" int symgpu_bind_thread_to_device_numa(int device) {
    const int node = symgpu_numa_node_of_device(device);
    if (node < 0) return -1;
    char path[128], buf[4096];
    std::snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    if (!read_small_file(path, buf, sizeof buf)) return -1;
    cpu_set_t want, have, both;
    if (!parse_cpulist(buf, &want)) return -1;
    // stay inside the CPUs this process is allowed to use (containers, taskset)
    if (sched_getaffinity(0, sizeof have, &have) != 0) return -1;
    CPU_AND(&both, &want, &have);
    if (CPU_COUNT(&both) == 0) return -1;
    if (sched_setaffinity(0, sizeof both, &both) != 0) return -1;
    return node;
}

extern "C" {

int symgpu_abi_version(void) { return SYMGPU_ABI_VERSION; }

// Test hook (not part of include/symgpu.h): the launch plan the host would build for a persistent grid of
// `grid` CTAs, as n_ctas + 1 chain offsets followed by the tiles (16 bytes each, mp3_kernel.h).  Needs no
// device.  Returns the number of 16-byte entries, writes at most `cap` of them, *n_ctas / *n_tiles / *hdr
// describe the layout; 0 on an argument error.
size_t symgpu_debug_mp3_plan(int grid, uint32_t n_streams, const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames,
                             void* out, size_t cap, int* n_ctas, int* n_tiles, int* hdr) {
    Mp3Plan plan;
    if (build_plan_for(grid, (uint32_t)mp3_tile_granules(), (uint32_t)mp3_halo_tile_granules(), true, n_streams, runs, n_runs,
                       n_frames, plan, true) != SYMGPU_OK)
        return 0;
    if (out) std::memcpy(out, plan.buf.data(), std::min(cap, plan.buf.size()) * sizeof(Mp3Tile));
    if (n_ctas) *n_ctas = plan.n_ctas;
    if (n_tiles) *n_tiles = plan.n_tiles;
    if (hdr) *hdr = plan.hdr;
    return plan.buf.size();
}

// Same for the second-generation kernel: the plan for a launch of at most `max_shares` warps (n_sm * warps per CTA
// on a device).  *n_shares / *n_tiles / *hdr describe the layout; 0 on an argument error.
size_t symgpu_debug_mp3_plan_v2(int max_shares, uint32_t n_streams, const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames,
                                void* out, size_t cap, int* n_shares, int* n_tiles, int* hdr) {
    Mp3Plan plan;
    if (build_plan_v2_for(max_shares, n_streams, runs, n_runs, n_frames, plan, true) != SYMGPU_OK) return 0;
    if (out) std::memcpy(out, plan.buf.data(), std::min(cap, plan.buf.size()) * sizeof(Mp3Tile));
    if (n_shares) *n_shares = plan.n_ctas;
    if (n_tiles) *n_tiles = plan.n_tiles;
    if (hdr) *hdr = plan.hdr;
    return plan.buf.size();
}

// Experiments: selects the instantiation of the second-generation kernel (warps per CTA, variant bits) for contexts
// created afterwards; 1 if that variant is built.
int symgpu_debug_mp3_v2_variant(int nw, int mode) { return mp3v2_set_variant(nw, mode) ? 1 : 0; }

const char* symgpu_strerror(symgpu_status status) {
    switch (status) {
        case SYMGPU_OK: return "ok";
        case SYMGPU_ERR_DECODE: return "symgpu: malformed synthesis unit";
        case SYMGPU_ERR_UNSUPPORTED: return "symgpu: unsupported stream configuration";
        case SYMGPU_ERR_LIMIT: return "symgpu: batch or stream limit exceeded";
        case SYMGPU_ERR_RESET: return "symgpu: decoder reset required";
        case SYMGPU_ERR_CUDA: return "symgpu: CUDA failure (see symgpu_last_cuda_error)";
        case SYMGPU_ERR_ARG: return "symgpu: invalid argument";
    }
    return "symgpu: unknown status";
}

const char* symgpu_last_cuda_error(const symgpu_ctx* ctx) { return ctx ? ctx->cuda_err : ""; }

size_t symgpu_tables_host_blob(void* out, size_t cap) {
    const Mp3Tables& t = mp3_tables_host();
    if (out && cap >= sizeof t) std::memcpy(out, &t, sizeof t);
    return sizeof t;
}

size_t symgpu_codec_tables_host_blob(void* out, size_t cap) {
    const CodecTables& t = codec_tables_host();
    if (out && cap >= sizeof t) std::memcpy(out, &t, sizeof t);
    return sizeof t;
}

size_t symgpu_mp3_pow43(float* out, size_t cap) {
    const Mp3Tables& t = mp3_tables_host();
    if (out) std::memcpy(out, t.pow43, sizeof(float) * (cap < 8207 ? cap : 8207));
    return 8207;
}

symgpu_status symgpu_tables_upload(symgpu_ctx* ctx, const void* blob, size_t bytes) {
    if (!ctx || !blob || bytes != sizeof(Mp3Tables)) return SYMGPU_ERR_ARG;
    DeviceGuard guard(ctx->device);
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    CU(ctx, cudaMemcpy(ctx->d_mp3_tab, blob, bytes, cudaMemcpyHostToDevice));
    CU(ctx, mp3_upload_const(*static_cast<const Mp3Tables*>(blob), ctx->stream));
    CU(ctx, mp3v2_upload_const(*static_cast<const Mp3Tables*>(blob), ctx->stream));
    return SYMGPU_OK;
}

symgpu_status symgpu_ctx_create(int device, symgpu_ctx** out) {
    if (!out) return SYMGPU_ERR_ARG;
    *out = nullptr;
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || device < 0 || device >= n_dev) {
        std::fprintf(stderr, "symgpu: no usable CUDA device %d (%s); this library has no CPU path\n", device,
                     e != cudaSuccess ? cudaGetErrorString(e) : "ordinal out of range");
        return SYMGPU_ERR_CUDA;
    }
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major < 10) {
        std::fprintf(stderr, "symgpu: device %d is not sm_100-class; kernels are built for sm_100a only\n", device);
        return SYMGPU_ERR_UNSUPPORTED;
    }
    symgpu_ctx* ctx = new (std::nothrow) symgpu_ctx();
    if (!ctx) return SYMGPU_ERR_LIMIT;
    ctx->device = device;
    // SYMGPU_ZERO_COPY = 0 never (default) | 1 output only | 2 input and output
    if (const char* env = std::getenv("SYMGPU_COPY_STREAMS")) ctx->copy_streams = std::atoi(env) >= 2 ? 2 : 1;
    if (const char* env = std::getenv("SYMGPU_ZERO_COPY")) {
        ctx->zero_copy = env[0] == '0' ? 0 : env[0] == '2' ? 2 : 1;
        ctx->zero_copy_small = env[0] != '0' && env[0] != 's'; // "0": never; "s": staged copies for small batches too
        if (env[0] == 's') ctx->zero_copy = 0;
    }
    if (const char* env = std::getenv("SYMGPU_H2D_AHEAD")) { // H2D copies queued before the host's check / planning (tuning)
        const int v = std::atoi(env);
        if (v >= 1 && v <= symgpu_ctx::kMaxSlices) ctx->h2d_ahead = v;
    }
    if (const char* env = std::getenv("SYMGPU_SLICES")) {
        const int v = std::atoi(env);
        if (v >= 1 && v <= symgpu_ctx::kMaxSlices) ctx->n_slices = v;
    }
    // SYMGPU_MP3_KERNEL=v1 selects the first-generation Layer III kernel (mp3_kernel.cu), kept for comparison
    // SYMGPU_MP3_KERNEL = auto (default) | v1 (first generation, scalar window) | v1p (first generation, packed window) | v2
    mp3_v1_set_packed_window(true);
    if (const char* env = std::getenv("SYMGPU_MP3_KERNEL")) {
        ctx->mp3_kernel_mode = std::strncmp(env, "v1", 2) == 0 ? 1 : std::strcmp(env, "v2") == 0 ? 2 : 0;
        mp3_v1_set_packed_window(std::strcmp(env, "v1") != 0);
    }
    if (const char* env = std::getenv("SYMGPU_MP3_V2_VARIANT")) { // "<warps>:<mode>", experiments
        int nw = 0, mode = 0;
        if (std::sscanf(env, "%d:%d", &nw, &mode) != 2 || !mp3v2_set_variant(nw, mode)) {
            std::fprintf(stderr, "symgpu: SYMGPU_MP3_V2_VARIANT=%s is not a built variant\n", env);
            delete ctx;
            return SYMGPU_ERR_ARG;
        }
    }
    // The calling thread moves to the CPUs of the GPU's NUMA node (pinned buffers it allocates from now on are local by
    // first touch); SYMGPU_NUMA_BIND=0 leaves the affinity alone.
    {
        const char* env = std::getenv("SYMGPU_NUMA_BIND");
        ctx->numa_node = (env && env[0] == '0') ? -2 : symgpu_bind_thread_to_device_numa(device);
    }
    DeviceGuard guard(device);
    auto fail = [&](cudaError_t err, const char* where) {
        std::fprintf(stderr, "symgpu: %s failed: %s\n", where, cudaGetErrorString(err));
        symgpu_ctx_destroy(ctx);
        return SYMGPU_ERR_CUDA;
    };
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return fail(e, "cudaStreamCreate");
    if ((e = cudaMalloc(&ctx->d_mp3_tab, sizeof(Mp3Tables))) != cudaSuccess) return fail(e, "cudaMalloc(tables)");
    const Mp3Tables& t = mp3_tables_host();
    if ((e = cudaMemcpy(ctx->d_mp3_tab, &t, sizeof t, cudaMemcpyHostToDevice)) != cudaSuccess) return fail(e, "cudaMemcpy(tables)");
    if ((e = mp3_upload_const(t, ctx->stream)) != cudaSuccess) return fail(e, "cudaMemcpyToSymbol(tables)");
    if ((e = mp3v2_upload_const(t, ctx->stream)) != cudaSuccess) return fail(e, "cudaMemcpyToSymbol(tables v2)");
    *out = ctx;
    return SYMGPU_OK;
}

void symgpu_ctx_destroy(symgpu_ctx* ctx) {
    if (!ctx) return;
    DeviceGuard guard(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    symgpu_async_mp3_destroy(ctx->async_mp3);
    if (ctx->d_mp3_tab) cudaFree(ctx->d_mp3_tab);
    if (ctx->d_mp3_states) cudaFree(ctx->d_mp3_states);
    if (ctx->d_mp3_gen) cudaFree(ctx->d_mp3_gen);
    if (ctx->d_tiles) cudaFree(ctx->d_tiles);
    if (ctx->h_tiles) cudaFreeHost(ctx->h_tiles);
    if (ctx->d_stage) cudaFree(ctx->d_stage);
    if (ctx->d_codec_tab) cudaFree(ctx->d_codec_tab);
    if (ctx->d_chunks) cudaFree(ctx->d_chunks);
    if (ctx->h_chunks) cudaFreeHost(ctx->h_chunks);
    if (ctx->d_aac_states) cudaFree(ctx->d_aac_states);
    if (ctx->d_aac_gen) cudaFree(ctx->d_aac_gen);
    if (ctx->d_aac_scratch) cudaFree(ctx->d_aac_scratch);
    if (ctx->d_aac_tns_idx) cudaFree(ctx->d_aac_tns_idx);
    if (ctx->d_vorbis_streams) cudaFree(ctx->d_vorbis_streams);
    if (ctx->d_vorbis_floors) cudaFree(ctx->d_vorbis_floors);
    if (ctx->d_vorbis_floor_aux) cudaFree(ctx->d_vorbis_floor_aux);
    if (ctx->d_vorbis_states) cudaFree(ctx->d_vorbis_states);
    if (ctx->d_vorbis_gen) cudaFree(ctx->d_vorbis_gen);
    if (ctx->d_vorbis_mc_streams) cudaFree(ctx->d_vorbis_mc_streams);
    if (ctx->d_vorbis_mc_scratch) cudaFree(ctx->d_vorbis_mc_scratch);
    if (ctx->copy_in) cudaStreamDestroy(ctx->copy_in);
    if (ctx->copy_out) cudaStreamDestroy(ctx->copy_out);
    if (ctx->copy_in2) cudaStreamDestroy(ctx->copy_in2);
    if (ctx->ev_units) cudaEventDestroy(ctx->ev_units);
    if (ctx->copy_out2) cudaStreamDestroy(ctx->copy_out2);
    for (int i = 0; i < symgpu_ctx::kMaxSlices; ++i) {
        if (ctx->ev_in[i]) cudaEventDestroy(ctx->ev_in[i]);
        if (ctx->ev_k[i]) cudaEventDestroy(ctx->ev_k[i]);
    }
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

symgpu_status symgpu_sync(symgpu_ctx* ctx) {
    if (!ctx) return SYMGPU_ERR_ARG;
    DeviceGuard guard(ctx->device);
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return SYMGPU_OK;
}

void* symgpu_cuda_stream(symgpu_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
int symgpu_ctx_numa_node(const symgpu_ctx* ctx) { return ctx ? ctx->numa_node : -1; }
uint64_t symgpu_launch_count(const symgpu_ctx* ctx) { return ctx ? ctx->launches : 0; }

symgpu_status symgpu_mp3_streams_alloc(symgpu_ctx* ctx, uint32_t n_streams) {
    if (!ctx || n_streams == 0) return SYMGPU_ERR_ARG;
    DeviceGuard guard(ctx->device);
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->d_mp3_states) cudaFree(ctx->d_mp3_states);
    if (ctx->d_mp3_gen) cudaFree(ctx->d_mp3_gen);
    ctx->d_mp3_states = nullptr;
    ctx->d_mp3_gen = nullptr;
    ctx->n_mp3_streams = 0;
    ctx->cached_runs.clear();
    ctx->cached_frames = 0;
    ctx->slice_plans_valid = false;
    CU(ctx, cudaMalloc(&ctx->d_mp3_states, (size_t)n_streams * 2 * sizeof(Mp3StreamState)));
    CU(ctx, cudaMemset(ctx->d_mp3_states, 0, (size_t)n_streams * 2 * sizeof(Mp3StreamState)));
    CU(ctx, cudaMalloc(&ctx->d_mp3_gen, ((size_t)n_streams + 1) * sizeof(uint32_t)));
    CU(ctx, cudaMemset(ctx->d_mp3_gen, 0, ((size_t)n_streams + 1) * sizeof(uint32_t)));
    ctx->n_mp3_streams = n_streams;
    return SYMGPU_OK;
}

symgpu_status symgpu_mp3_stream_reset(symgpu_ctx* ctx, uint32_t stream) {
    if (!ctx) return SYMGPU_ERR_ARG;
    if (stream >= ctx->n_mp3_streams) return SYMGPU_ERR_LIMIT;
    DeviceGuard guard(ctx->device);
    CU(ctx, cudaMemsetAsync(ctx->d_mp3_states + (size_t)stream * 2, 0, 2 * sizeof(Mp3StreamState), ctx->stream));
    return SYMGPU_OK;
}

symgpu_status symgpu_mp3_synth_dev(symgpu_ctx* ctx, const symgpu_mp3_gc* units, const float* spectra,
                                   const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames, float* pcm) {
    if (!ctx || !units || !spectra || !runs || !pcm) return SYMGPU_ERR_ARG;
    if (n_frames == 0) return SYMGPU_OK;
    DeviceGuard guard(ctx->device);
    symgpu_status s = ensure_plan(ctx, runs, n_runs, n_frames);
    if (s != SYMGPU_OK) return s;
    if (ctx->cached_tiles == 0) return SYMGPU_OK;
    CU(ctx, launch_plan(ctx, ctx->d_tiles, ctx->cached_hdr, ctx->cached_tiles, ctx->cached_ctas, ctx->cached_multi, ctx->cached_v2, units, spectra, pcm,
                        ctx->stream));
    ctx->launches += 1;
    return SYMGPU_OK;
}

} // extern "C"

constexpr uint32_t kPipelineMinFrames = 512; // smaller host batches: no slice pipeline (and zero-copy when the buffers are mapped)
static inline float* d_spec_base(char* stage_base) { return reinterpret_cast<float*>(stage_base); }


// symgpu_mp3_units_check over the runs in four parts on as many threads (the 64-byte descriptors of 8192 frames take ~190 us on
// one thread, which is 9 % of an end-to-end step).
static symgpu_status units_check_mt(const symgpu_mp3_gc* units, const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames) {
    if (n_frames < 1024 || n_runs < 4) return symgpu_mp3_units_check(units, runs, n_runs, n_frames);
    symgpu_status chk[4] = {SYMGPU_OK, SYMGPU_OK, SYMGPU_OK, SYMGPU_OK};
    std::thread workers[3];
    const uint32_t per = (n_runs + 3) / 4;
    auto part = [&](int k) {
        const uint32_t r0 = std::min<uint32_t>(n_runs, per * (uint32_t)k), r1 = std::min<uint32_t>(n_runs, r0 + per);
        if (r1 > r0) chk[k] = symgpu_mp3_units_check(units, runs + r0, r1 - r0, n_frames);
    };
    for (int k = 1; k < 4; ++k) workers[k - 1] = std::thread(part, k);
    part(0);
    for (auto& w : workers) w.join();
    for (symgpu_status c : chk)
        if (c != SYMGPU_OK) return c;
    return SYMGPU_OK;
}

// Host-buffer MP3 synthesis.  format < 0: planar f32 into `out` (the AudioBuffer layout); otherwise the
// output stage runs on the device after each slice's kernel and `out` receives interleaved samples.
static symgpu_status mp3_synth_host_impl(symgpu_ctx* ctx, const symgpu_mp3_gc* units, const float* spectra, const int16_t* quant,
                                         const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames, int format,
                                         void* out) {
    // exactly one of `spectra` (f32) and `quant` (i16, expanded on the device) describes the input
    if (!ctx || !units || (!spectra == !quant) || !runs || !out) return SYMGPU_ERR_ARG;
    const size_t sample_bytes = format < 0 ? sizeof(float) : symgpu_sample_bytes(format);
    if (sample_bytes == 0) return SYMGPU_ERR_ARG;
    if (n_frames == 0) return SYMGPU_OK;
    // The runs' geometry is checked now (cheap); the 64-byte descriptors of every granule-channel (~200 us of host time
    // for 8192 frames) are checked while the first H2D copies are already on their way.
    for (uint32_t r = 0; r < n_runs; ++r) {
        const int gpf = runs[r].granules_per_frame ? runs[r].granules_per_frame : 2;
        const int n_ch = runs[r].channels ? runs[r].channels : 2;
        if (gpf < 1 || gpf > 2 || n_ch < 1 || n_ch > 2) return SYMGPU_ERR_ARG;
        if ((uint64_t)runs[r].first_frame + runs[r].n_frames > n_frames) return SYMGPU_ERR_ARG;
    }
    DeviceGuard guard(ctx->device);
    const size_t unit_bytes = (size_t)n_frames * 4 * sizeof(symgpu_mp3_gc);
    const size_t spec_bytes = (size_t)n_frames * SYMGPU_MP3_FRAME_FLOATS * sizeof(float);
    // ---- zero-copy: pinned, device-mapped host buffers are read and written by the kernel itself --------------------------------
    // When `units`, `spectra` and `out` are pinned host memory (cudaHostAlloc / cudaHostRegister: device-accessible under unified
    // addressing), the synthesis kernel takes them as they are: its TMA bulk copies pull the next granule's spectra across PCIe
    // one granule (or tile) ahead of the arithmetic and its coalesced 128-byte PCM stores go straight to host memory.  H2D
    // traffic, arithmetic and D2H traffic overlap inside ONE launch -- no staging copy, no slice pipeline, no copy-engine
    // scheduling between them.  Opt-in (SYMGPU_ZERO_COPY=2): measured 2.36 ms per 8192-frame step against 2.20 ms for the
    // staged pipeline below (profiles/r02l_*), bit-identical output (tests/test_mp3_parity_gpu.py).
    // Small batches (a single packet is the extreme: config 1) take this path by default when the buffers allow it: one launch and
    // one synchronisation instead of two or three copy set-ups around them (SYMGPU_ZERO_COPY=0 switches it off).
    const bool small_auto = ctx->zero_copy_small && n_frames < kPipelineMinFrames;
    if ((ctx->zero_copy == 2 || small_auto) && !quant && format < 0) {
        bool whole = true;
        for (uint32_t r = 0; r < n_runs; ++r) whole &= runs[r].granules_per_frame != 1 && runs[r].channels != 1;
        auto mapped = [](const void* p) -> void* {
            cudaPointerAttributes at{};
            if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
                cudaGetLastError(); // pageable memory on older drivers: clear the error
                return nullptr;
            }
            return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
        };
        void* d_u = whole ? mapped(units) : nullptr;
        void* d_s = d_u ? mapped(spectra) : nullptr;
        void* d_o = d_s ? mapped(out) : nullptr;
        if (d_o) {
            // descriptors are checked before anything runs on them (four host threads: ~50 us for 8192 frames)
            {
                const symgpu_status c = units_check_mt(units, runs, n_runs, n_frames);
                if (c != SYMGPU_OK) return c;
            }
            symgpu_status zs = symgpu_mp3_synth_dev(ctx, static_cast<const symgpu_mp3_gc*>(d_u), static_cast<const float*>(d_s), runs, n_runs,
                                                    n_frames, static_cast<float*>(d_o));
            if (zs != SYMGPU_OK) return zs;
            CU(ctx, cudaStreamSynchronize(ctx->stream));
            return SYMGPU_OK;
        }
    }
    const size_t packed_bytes = format < 0 ? 0 : (size_t)n_frames * SYMGPU_MP3_FRAME_FLOATS * sample_bytes;
    const size_t quant_bytes = quant ? spec_bytes / 2 : 0;
    symgpu_status s = ensure_stage(ctx, unit_bytes + 2 * spec_bytes + packed_bytes + quant_bytes);
    if (s != SYMGPU_OK) return s;
    char* base = static_cast<char*>(ctx->d_stage);
    int16_t* d_quant = reinterpret_cast<int16_t*>(base + 2 * spec_bytes + unit_bytes + packed_bytes);
    // H2D copy of frames [f0, f0 + nf): the f32 spectra, or the quantised values followed by their expansion
    auto copy_in = [&](uint32_t f0, size_t nf, cudaStream_t cs) -> cudaError_t {
        const size_t off = (size_t)f0 * SYMGPU_MP3_FRAME_FLOATS, cnt = nf * SYMGPU_MP3_FRAME_FLOATS;
        if (!quant) return cudaMemcpyAsync(d_spec_base(base) + off, spectra + off, cnt * sizeof(float), cudaMemcpyHostToDevice, cs);
        cudaError_t e = cudaMemcpyAsync(d_quant + off, quant + off, cnt * sizeof(int16_t), cudaMemcpyHostToDevice, cs);
        if (e != cudaSuccess) return e;
        ctx->launches += 1;
        return symgpu::dequant_launch(d_quant + off, d_spec_base(base) + off, cnt, ctx->d_mp3_tab->pow43, cs);
    };
    float* d_spec = reinterpret_cast<float*>(base);
    float* d_pcm = reinterpret_cast<float*>(base + spec_bytes);
    symgpu_mp3_gc* d_units = reinterpret_cast<symgpu_mp3_gc*>(base + 2 * spec_bytes);
    char* d_packed = base + 2 * spec_bytes + unit_bytes; // unit_bytes is a multiple of 256
    char* out_bytes = static_cast<char*>(out);
    // Device source and per-frame size of what travels back to the host.
    const char* d_result = format < 0 ? reinterpret_cast<const char*>(d_pcm) : d_packed;
    const size_t frame_out_bytes = (size_t)SYMGPU_MP3_FRAME_FLOATS * sample_bytes;
    auto pack = [&](uint32_t f0, uint32_t nf) -> cudaError_t {
        if (format < 0) return cudaSuccess;
        symgpu::PackArgs pa{d_pcm + (size_t)f0 * SYMGPU_MP3_FRAME_FLOATS, nullptr, nf, 2, 1152, 1152,
                            d_packed + (size_t)f0 * frame_out_bytes};
        ctx->launches += 1;
        return symgpu::pack_launch(pa, format, ctx->stream);
    };
    // Mono / MPEG-2 frames leave part of each PCM slot untouched: define it as zero.
    bool partial = false, sorted = true;
    uint64_t next = 0;
    for (uint32_t r = 0; r < n_runs; ++r) {
        partial |= runs[r].granules_per_frame == 1 || runs[r].channels == 1;
        sorted &= runs[r].first_frame == next;
        next += runs[r].n_frames;
    }
    sorted &= next == n_frames;
    if (partial && format >= 0) return SYMGPU_ERR_UNSUPPORTED;
    if (partial) CU(ctx, cudaMemsetAsync(d_pcm, 0, spec_bytes, ctx->stream));
    // Output zero-copy: a pinned (device-mapped) f32 output buffer is written by the kernels themselves -- coalesced 128-byte
    // PCM stores that cross PCIe while the next slice is still coming in -- so the D2H copies and their scheduling disappear.
    bool out_mapped = false;
    if (ctx->zero_copy && format < 0 && !partial) {
        cudaPointerAttributes at{};
        if (cudaPointerGetAttributes(&at, out) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) {
            d_pcm = static_cast<float*>(at.devicePointer);
            out_mapped = true;
        } else {
            cudaGetLastError();
        }
    }

    if (!sorted || n_frames < kPipelineMinFrames || n_runs < 2) {
        // small or unsorted batch: one copy in, one launch, one copy out
        CU(ctx, cudaMemcpyAsync(d_units, units, unit_bytes, cudaMemcpyHostToDevice, ctx->stream));
        CU(ctx, copy_in(0, n_frames, ctx->stream));
        s = units_check_mt(units, runs, n_runs, n_frames); // overlaps the copies; nothing has been launched yet
        if (s == SYMGPU_OK) s = symgpu_mp3_synth_dev(ctx, d_units, d_spec, runs, n_runs, n_frames, d_pcm);
        if (s != SYMGPU_OK) {
            cudaStreamSynchronize(ctx->stream); // the copies read the caller's buffers
            return s;
        }
        CU(ctx, pack(0, n_frames));
        if (!out_mapped) CU(ctx, cudaMemcpyAsync(out_bytes, d_result, (size_t)n_frames * frame_out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        return SYMGPU_OK;
    }

    // Copy pipeline: the batch is cut into slices of whole runs; the H2D copy of slice i+1 (copy_in),
    // the kernel of slice i (ctx->stream) and the D2H copy of slice i-1 (copy_out) overlap, so both
    // PCIe directions stay busy.
    if (!ctx->copy_in) {
        CU(ctx, cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking));
        CU(ctx, cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking));
        CU(ctx, cudaStreamCreateWithFlags(&ctx->copy_in2, cudaStreamNonBlocking));
        CU(ctx, cudaStreamCreateWithFlags(&ctx->copy_out2, cudaStreamNonBlocking));
        CU(ctx, cudaEventCreateWithFlags(&ctx->ev_units, cudaEventDisableTiming));
        for (int i = 0; i < symgpu_ctx::kMaxSlices; ++i) {
            CU(ctx, cudaEventCreateWithFlags(&ctx->ev_in[i], cudaEventDisableTiming));
            CU(ctx, cudaEventCreateWithFlags(&ctx->ev_k[i], cudaEventDisableTiming));
        }
    }
    const int n_slices = (int)std::min<uint32_t>((uint32_t)ctx->n_slices, n_runs);
    struct Slice { uint32_t r0, r1, f0, f1; int t0, hdr, n_tiles, n_ctas; bool multi, v2; };
    std::vector<Slice> slices;
    uint32_t r = 0;
    // Both PCIe directions carry about the same bytes, so the run is as long as the D2H chain, which cannot start
    // before the first slice is in and cannot end before the last slice is out: the slices taper at both ends
    // (weights 0.25, 0.5, 1, ..., 1, 0.5, 0.25); every extra slice costs two copy set-ups (~20 us each).
    double w_total = 0.0, w_acc = 0.0;
    auto weight = [&](int i) {
        const int edge = std::min(i, n_slices - 1 - i);
        return n_slices < 4 ? 1.0 : edge == 0 ? 0.25 : edge == 1 ? 0.5 : 1.0;
    };
    for (int i = 0; i < n_slices; ++i) w_total += weight(i);
    for (int i = 0; i < n_slices; ++i) {
        w_acc += weight(i);
        const uint32_t target = (uint32_t)((double)n_frames * (w_acc / w_total));
        Slice sl{r, r, runs[r].first_frame, 0, 0, 0, 0, 0, false, false};
        while (r < n_runs && (runs[r].first_frame + runs[r].n_frames <= target || sl.r1 == sl.r0)) {
            ++r;
            sl.r1 = r;
        }
        if (i + 1 == n_slices) { r = n_runs; sl.r1 = n_runs; }
        sl.f1 = sl.r1 < n_runs ? runs[sl.r1].first_frame : n_frames;
        if (sl.r1 > sl.r0 && sl.f1 > sl.f0) slices.push_back(sl);
        if (r >= n_runs) break;
    }
    // 1. the H2D copies of the first `ahead` slices are queued at once, so that the copy engine has work while the host checks
    //    the descriptors and plans the launches.  The rest is queued slice by slice BEHIND the D2H copy of an earlier slice:
    //    queueing every H2D copy up front was measured to serialise the two directions (2.9 ms instead of 2.2 ms per step).
    // (with the output written by the kernels there are no D2H copies to interleave with: everything is queued at once)
    const size_t ahead = out_mapped ? slices.size() : std::min<size_t>(slices.size(), (size_t)std::max(1, ctx->h2d_ahead));
    // SYMGPU_E2E_TRACE=1: timing events around every copy and launch of the pipeline, printed after the call (diagnostics only)
    static const bool trace = [] { const char* e = std::getenv("SYMGPU_E2E_TRACE"); return e && e[0] == '1'; }();
    std::vector<cudaEvent_t> tev;
    auto mark = [&](cudaStream_t st) {
        if (!trace) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, st);
        tev.push_back(e);
    };
    const bool two = ctx->copy_streams >= 2;
    auto cin = [&](size_t i) { return (two && (i & 1)) ? ctx->copy_in2 : ctx->copy_in; };
    auto cout_ = [&](size_t i) { return (two && (i & 1)) ? ctx->copy_out2 : ctx->copy_out; };
    mark(ctx->copy_in); // t0
    CU(ctx, cudaMemcpyAsync(d_units, units, unit_bytes, cudaMemcpyHostToDevice, ctx->copy_in)); // 256 B per frame: one copy
    // the descriptors travel on the first copy stream; the second one must not overtake them
    if (two) {
        CU(ctx, cudaEventRecord(ctx->ev_units, ctx->copy_in));
        CU(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_units, 0));
    }
    for (size_t i = 0; i < ahead; ++i) {
        mark(cin(i));
        CU(ctx, copy_in(slices[i].f0, slices[i].f1 - slices[i].f0, cin(i)));
        mark(cin(i));
        CU(ctx, cudaEventRecord(ctx->ev_in[i], cin(i)));
    }
    // 2. host work under those copies: descriptor check (helper threads) and the launch plans of the slices -- which are kept
    //    (and stay on the device) while the caller repeats the same runs
    symgpu_status chk = SYMGPU_OK;
    std::thread checker([&] { chk = units_check_mt(units, runs, n_runs, n_frames); });
    const bool plans_cached = ctx->slice_plans_valid && ctx->slice_frames == n_frames && ctx->slice_key_slices == n_slices &&
                              ctx->slice_key_mode == ctx->mp3_kernel_mode && ctx->slice_runs.size() == n_runs &&
                              std::memcmp(ctx->slice_runs.data(), runs, n_runs * sizeof *runs) == 0 && ctx->slice_plans.size() == slices.size();
    s = SYMGPU_OK;
    if (plans_cached) {
        for (size_t i = 0; i < slices.size(); ++i) {
            const symgpu_ctx::SlicePlan& c = ctx->slice_plans[i];
            slices[i].t0 = c.t0, slices[i].hdr = c.hdr, slices[i].n_tiles = c.n_tiles, slices[i].n_ctas = c.n_ctas;
            slices[i].multi = c.multi, slices[i].v2 = c.v2;
        }
        checker.join();
        s = chk;
    } else {
        std::vector<Mp3Tile> all_tiles;
        Mp3Plan plan;
        for (size_t i = 0; i < slices.size() && s == SYMGPU_OK; ++i) {
            Slice& sl = slices[i];
            s = build_plan(ctx, runs + sl.r0, sl.r1 - sl.r0, n_frames, plan, false);
            sl.t0 = (int)all_tiles.size();
            all_tiles.insert(all_tiles.end(), plan.buf.begin(), plan.buf.end());
            sl.hdr = plan.hdr;
            sl.n_tiles = plan.n_tiles;
            sl.n_ctas = plan.n_ctas;
            sl.multi = plan.multi;
            sl.v2 = plan.v2;
        }
        if (s == SYMGPU_OK) s = reserve_plan(ctx, all_tiles.size());
        checker.join();
        if (s == SYMGPU_OK) s = chk;
        if (s == SYMGPU_OK) {
            ctx->cached_runs.clear(); // the cached plan of the device entry point is replaced
            ctx->cached_frames = 0;
            std::memcpy(ctx->h_tiles, all_tiles.data(), all_tiles.size() * sizeof(Mp3Tile));
            cudaError_t ce = cudaMemcpyAsync(ctx->d_tiles, ctx->h_tiles, all_tiles.size() * sizeof(Mp3Tile), cudaMemcpyHostToDevice, ctx->stream);
            if (ce != cudaSuccess) s = cuda_fail(ctx, ce, "cudaMemcpyAsync(slice plans)");
        }
        if (s == SYMGPU_OK) {
            ctx->slice_plans.clear();
            for (const Slice& sl : slices) ctx->slice_plans.push_back({sl.r0, sl.r1, sl.f0, sl.f1, sl.t0, sl.hdr, sl.n_tiles, sl.n_ctas, sl.multi, sl.v2});
            ctx->slice_runs.assign(runs, runs + n_runs);
            ctx->slice_frames = n_frames;
            ctx->slice_key_slices = n_slices;
            ctx->slice_key_mode = ctx->mp3_kernel_mode;
            ctx->slice_plans_valid = true;
        }
    }
    if (s != SYMGPU_OK) {
        cudaStreamSynchronize(ctx->copy_in); // the copies read the caller's buffers; nothing has been launched
        if (two) cudaStreamSynchronize(ctx->copy_in2);
        return s;
    }
    // 3. kernels as the slices land, D2H copies as the kernels finish, the next H2D copy behind each D2H copy
    for (size_t i = 0; i < slices.size(); ++i) {
        const Slice& sl = slices[i];
        const size_t nf = sl.f1 - sl.f0;
        CU(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_in[i], 0));
        mark(ctx->stream);
        if (sl.n_tiles > 0) {
            CU(ctx, launch_plan(ctx, ctx->d_tiles + sl.t0, sl.hdr, sl.n_tiles, sl.n_ctas, sl.multi, sl.v2, d_units, d_spec, d_pcm, ctx->stream));
            ctx->launches += 1;
        }
        CU(ctx, pack(sl.f0, (uint32_t)nf));
        mark(ctx->stream);
        if (!out_mapped) {
            CU(ctx, cudaEventRecord(ctx->ev_k[i], ctx->stream));
            CU(ctx, cudaStreamWaitEvent(cout_(i), ctx->ev_k[i], 0));
            mark(cout_(i));
            CU(ctx, cudaMemcpyAsync(out_bytes + (size_t)sl.f0 * frame_out_bytes, d_result + (size_t)sl.f0 * frame_out_bytes,
                                    nf * frame_out_bytes, cudaMemcpyDeviceToHost, cout_(i)));
            mark(cout_(i));
        }
        if (i + ahead < slices.size()) {
            const Slice& nx = slices[i + ahead];
            mark(cin(i + ahead));
            CU(ctx, copy_in(nx.f0, nx.f1 - nx.f0, cin(i + ahead)));
            mark(cin(i + ahead));
            CU(ctx, cudaEventRecord(ctx->ev_in[i + ahead], cin(i + ahead)));
        }
    }
    CU(ctx, cudaStreamSynchronize(ctx->copy_out));
    if (two) CU(ctx, cudaStreamSynchronize(ctx->copy_out2));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    if (trace && !tev.empty()) {
        // marks in issue order: t0 | (h2d start, end) x ahead | per slice: k start, k end, [d2h start, end], [h2d start, end]
        std::fprintf(stderr, "symgpu e2e trace (ms from the first copy; %zu slices, %zu H2D ahead):", slices.size(), ahead);
        for (size_t i = 1; i < tev.size(); ++i) {
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, tev[0], tev[i]);
            std::fprintf(stderr, "%s%.3f", (i % 2) ? "  " : "-", ms);
        }
        std::fprintf(stderr, "\n");
        for (cudaEvent_t e : tev) cudaEventDestroy(e);
    }
    return SYMGPU_OK;
}

extern "C" {

symgpu_status symgpu_mp3_units_check(const symgpu_mp3_gc* units, const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames) {
    if (!units || !runs) return SYMGPU_ERR_ARG;
    for (uint32_t r = 0; r < n_runs; ++r) {
        const symgpu_mp3_run& run = runs[r];
        const int gpf = run.granules_per_frame ? run.granules_per_frame : 2;
        const int n_ch = run.channels ? run.channels : 2;
        if (gpf < 1 || gpf > 2 || n_ch < 1 || n_ch > 2) return SYMGPU_ERR_ARG;
        if ((uint64_t)run.first_frame + run.n_frames > n_frames) return SYMGPU_ERR_ARG;
        for (uint32_t f = run.first_frame; f < run.first_frame + run.n_frames; ++f)
            for (int gr = 0; gr < gpf; ++gr) {
                const symgpu_mp3_gc* u = units + ((size_t)f * 2 + gr) * 2;
                for (int ch = 0; ch < n_ch; ++ch) {
                    const symgpu_mp3_gc& g = u[ch];
                    if (g.block_type > SYMGPU_MP3_END || g.sample_rate_idx > 8 || g.rzero > 576) return SYMGPU_ERR_DECODE;
                    if (g.subblock_gain[0] > 7 || g.subblock_gain[1] > 7 || g.subblock_gain[2] > 7) return SYMGPU_ERR_DECODE;
                }
                // stereo.rs:503-505: joint stereo needs the same block type (and mixed flag) on both channels
                if (n_ch == 2 && (u[0].flags & (SYMGPU_MP3_F_MID_SIDE | SYMGPU_MP3_F_INTENSITY)) &&
                    (u[0].block_type != u[1].block_type ||
                     ((u[0].flags ^ u[1].flags) & SYMGPU_MP3_F_MIXED && u[0].block_type == SYMGPU_MP3_SHORT)))
                    return SYMGPU_ERR_DECODE;
                if (n_ch == 2 && u[0].sample_rate_idx != u[1].sample_rate_idx) return SYMGPU_ERR_DECODE;
            }
    }
    return SYMGPU_OK;
}

symgpu_status symgpu_mp3_synth_host(symgpu_ctx* ctx, const symgpu_mp3_gc* units, const float* spectra,
                                    const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames, float* pcm) {
    return mp3_synth_host_impl(ctx, units, spectra, nullptr, runs, n_runs, n_frames, -1, pcm);
}

symgpu_status symgpu_mp3_synth_host_packed(symgpu_ctx* ctx, const symgpu_mp3_gc* units, const float* spectra,
                                           const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames,
                                           int format, void* out) {
    if (format < 0) return SYMGPU_ERR_ARG;
    return mp3_synth_host_impl(ctx, units, spectra, nullptr, runs, n_runs, n_frames, format, out);
}

symgpu_status symgpu_mp3_synth_host_quantized(symgpu_ctx* ctx, const symgpu_mp3_gc* units, const int16_t* quant,
                                              const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames,
                                              int format, void* out) {
    return mp3_synth_host_impl(ctx, units, nullptr, quant, runs, n_runs, n_frames, format, out);
}

uint32_t symgpu_pcm_span_kept(const symgpu_pcm_span* s) {
    if (!s) return 0;
    const uint32_t n = s->frames > s->trim_end ? s->frames - s->trim_end : 0;
    return s->trim_start >= n ? 0 : n - s->trim_start;
}

size_t symgpu_sample_bytes(int format) {
    switch (format) {
    case SYMGPU_FMT_F32: case SYMGPU_FMT_S24: case SYMGPU_FMT_S32: return 4;
    case SYMGPU_FMT_S16: return 2;
    case SYMGPU_FMT_U8: return 1;
    default: return 0;
    }
}

// map: nullptr, or the plane of every output channel (checked: < channels), packed into PackArgs::plane_map
static symgpu_status pcm_pack_dev_impl(symgpu_ctx* ctx, const float* pcm, const symgpu_pcm_span* spans, uint32_t n_spans, uint32_t channels,
                                       uint32_t plane_stride, uint32_t frames, const uint8_t* map, int format, void* out) {
    if (!ctx || !pcm || !out || channels == 0 || channels > 8) return SYMGPU_ERR_ARG;
    if (symgpu_sample_bytes(format) == 0) return SYMGPU_ERR_ARG;
    uint32_t plane_map = 0;
    if (map)
        for (uint32_t c = 0; c < channels; ++c) {
            if (map[c] >= channels) return SYMGPU_ERR_ARG;
            plane_map |= (uint32_t)map[c] << (4 * c);
        }
    if (n_spans == 0) return SYMGPU_OK;
    DeviceGuard guard(ctx->device);
    symgpu::PackArgs pa{pcm, spans, n_spans, channels, plane_stride, frames, out, plane_map};
    CU(ctx, symgpu::pack_launch(pa, format, ctx->stream, map != nullptr));
    ctx->launches += 1;
    return SYMGPU_OK;
}

static symgpu_status pcm_pack_host_impl(symgpu_ctx* ctx, const float* pcm, size_t pcm_floats, const symgpu_pcm_span* spans, uint32_t n_spans,
                                        uint32_t channels, uint32_t plane_stride, uint32_t frames, const uint8_t* map, int format, void* out,
                                        size_t out_bytes) {
    if (!ctx || !pcm || !out || channels == 0 || channels > 8) return SYMGPU_ERR_ARG;
    const size_t sb = symgpu_sample_bytes(format);
    if (sb == 0) return SYMGPU_ERR_ARG;
    if (map)
        for (uint32_t c = 0; c < channels; ++c)
            if (map[c] >= channels) return SYMGPU_ERR_ARG;
    if (n_spans == 0) return SYMGPU_OK;
    // Every span must stay inside the buffers the caller described.
    for (uint32_t p = 0; p < n_spans; ++p) {
        symgpu_pcm_span sp;
        if (spans) sp = spans[p];
        else sp = symgpu_pcm_span{(uint64_t)p * channels * plane_stride, plane_stride, frames, 0, 0, (uint64_t)p * frames};
        const uint32_t kept = symgpu_pcm_span_kept(&sp);
        if (kept == 0) continue;
        if (sp.src + (uint64_t)(channels - 1) * sp.plane_stride + sp.trim_start + kept > pcm_floats) return SYMGPU_ERR_LIMIT;
        if ((sp.dst_frame + kept) * channels * sb > out_bytes) return SYMGPU_ERR_LIMIT;
    }
    DeviceGuard guard(ctx->device);
    const size_t in_bytes = (pcm_floats * sizeof(float) + 255) & ~(size_t)255;
    const size_t span_bytes = spans ? ((size_t)n_spans * sizeof(symgpu_pcm_span) + 255) & ~(size_t)255 : 0;
    symgpu_status s = ensure_stage(ctx, in_bytes + span_bytes + out_bytes);
    if (s != SYMGPU_OK) return s;
    char* base = static_cast<char*>(ctx->d_stage);
    CU(ctx, cudaMemcpyAsync(base, pcm, pcm_floats * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    if (spans) CU(ctx, cudaMemcpyAsync(base + in_bytes, spans, (size_t)n_spans * sizeof(symgpu_pcm_span), cudaMemcpyHostToDevice, ctx->stream));
    // Samples no span writes keep the caller's bytes.
    CU(ctx, cudaMemcpyAsync(base + in_bytes + span_bytes, out, out_bytes, cudaMemcpyHostToDevice, ctx->stream));
    s = pcm_pack_dev_impl(ctx, reinterpret_cast<const float*>(base), spans ? reinterpret_cast<const symgpu_pcm_span*>(base + in_bytes) : nullptr,
                          n_spans, channels, plane_stride, frames, map, format, base + in_bytes + span_bytes);
    if (s != SYMGPU_OK) return s;
    CU(ctx, cudaMemcpyAsync(out, base + in_bytes + span_bytes, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return SYMGPU_OK;
}

symgpu_status symgpu_pcm_pack_dev(symgpu_ctx* ctx, const float* pcm, const symgpu_pcm_span* spans, uint32_t n_spans,
                                  uint32_t channels, uint32_t plane_stride, uint32_t frames, int format, void* out) {
    return pcm_pack_dev_impl(ctx, pcm, spans, n_spans, channels, plane_stride, frames, nullptr, format, out);
}

symgpu_status symgpu_pcm_pack_host(symgpu_ctx* ctx, const float* pcm, size_t pcm_floats, const symgpu_pcm_span* spans,
                                   uint32_t n_spans, uint32_t channels, uint32_t plane_stride, uint32_t frames,
                                   int format, void* out, size_t out_bytes) {
    return pcm_pack_host_impl(ctx, pcm, pcm_floats, spans, n_spans, channels, plane_stride, frames, nullptr, format, out, out_bytes);
}

symgpu_status symgpu_pcm_pack_mapped_dev(symgpu_ctx* ctx, const float* pcm, const symgpu_pcm_span* spans, uint32_t n_spans,
                                         uint32_t channels, uint32_t plane_stride, uint32_t frames, const uint8_t* plane_of_channel,
                                         int format, void* out) {
    if (!plane_of_channel) return SYMGPU_ERR_ARG;
    return pcm_pack_dev_impl(ctx, pcm, spans, n_spans, channels, plane_stride, frames, plane_of_channel, format, out);
}

symgpu_status symgpu_pcm_pack_mapped_host(symgpu_ctx* ctx, const float* pcm, size_t pcm_floats, const symgpu_pcm_span* spans,
                                          uint32_t n_spans, uint32_t channels, uint32_t plane_stride, uint32_t frames,
                                          const uint8_t* plane_of_channel, int format, void* out, size_t out_bytes) {
    if (!plane_of_channel) return SYMGPU_ERR_ARG;
    return pcm_pack_host_impl(ctx, pcm, pcm_floats, spans, n_spans, channels, plane_stride, frames, plane_of_channel, format, out, out_bytes);
}

// ---- MPEG Layer I / II ---------------------------------------------------------------------------------
static symgpu_status mpa12_plan(symgpu_ctx* ctx, const symgpu_mpa12_run* runs, uint32_t n_runs, uint32_t n_frames, uint32_t n_slots,
                                Mp3Plan& plan) {
    if (n_slots != 12 && n_slots != 36) return SYMGPU_ERR_ARG;
    cudaError_t ce = cudaSuccess;
    const int grid = mp3_grid_size(&ce);
    if (ce != cudaSuccess || grid <= 0) return cuda_fail(ctx, ce, "mp3_grid_size");
    std::vector<symgpu_mp3_run> as_frames(n_runs); // units of the planner = frames
    for (uint32_t r = 0; r < n_runs; ++r) {
        if (runs[r].reserved[0] || runs[r].reserved[1] || runs[r].reserved[2]) return SYMGPU_ERR_ARG;
        as_frames[r] = symgpu_mp3_run{runs[r].stream, runs[r].first_frame, runs[r].n_frames, 1, runs[r].channels, 0};
    }
    const uint32_t T = (uint32_t)mpa12_tile_frames((int)n_slots);
    return build_plan_for(grid, T, T, false, ctx->n_mp3_streams, as_frames.data(), n_runs, n_frames, plan, true);
}

symgpu_status symgpu_mpa12_synth_dev(symgpu_ctx* ctx, const float* subbands, const symgpu_mpa12_run* runs, uint32_t n_runs,
                                     uint32_t n_frames, uint32_t n_slots, float* pcm) {
    if (!ctx || !subbands || !runs || !pcm) return SYMGPU_ERR_ARG;
    if (n_frames == 0) return SYMGPU_OK;
    DeviceGuard guard(ctx->device);
    Mp3Plan plan;
    symgpu_status s = mpa12_plan(ctx, runs, n_runs, n_frames, n_slots, plan);
    if (s != SYMGPU_OK) return s;
    s = reserve_plan(ctx, plan.buf.size());
    if (s != SYMGPU_OK) return s;
    ctx->cached_runs.clear(); // the Layer III plan on the device is being replaced
    ctx->cached_frames = 0;
    std::memcpy(ctx->h_tiles, plan.buf.data(), plan.buf.size() * sizeof(Mp3Tile));
    CU(ctx, cudaMemcpyAsync(ctx->d_tiles, ctx->h_tiles, plan.buf.size() * sizeof(Mp3Tile), cudaMemcpyHostToDevice, ctx->stream));
    if (plan.n_tiles == 0) return SYMGPU_OK;
    Mpa12Args a{subbands, pcm, reinterpret_cast<const uint32_t*>(ctx->d_tiles), ctx->d_tiles + plan.hdr, plan.n_tiles, plan.n_ctas,
                (int)n_slots, ctx->d_mp3_states, ctx->d_mp3_gen, ctx->d_mp3_gen + ctx->n_mp3_streams, ctx->d_mp3_tab};
    CU(ctx, mpa12_launch(a, ctx->stream));
    ctx->launches += 1;
    return SYMGPU_OK;
}

symgpu_status symgpu_mpa12_synth_host(symgpu_ctx* ctx, const float* subbands, const symgpu_mpa12_run* runs, uint32_t n_runs,
                                      uint32_t n_frames, uint32_t n_slots, float* pcm) {
    if (!ctx || !subbands || !runs || !pcm) return SYMGPU_ERR_ARG;
    if (n_slots != 12 && n_slots != 36) return SYMGPU_ERR_ARG;
    if (n_frames == 0) return SYMGPU_OK;
    DeviceGuard guard(ctx->device);
    const size_t in_bytes = (size_t)n_frames * 64 * n_slots * sizeof(float);
    const size_t out_bytes = (size_t)n_frames * SYMGPU_MP3_FRAME_FLOATS * sizeof(float);
    symgpu_status s = ensure_stage(ctx, in_bytes + out_bytes);
    if (s != SYMGPU_OK) return s;
    float* d_in = static_cast<float*>(ctx->d_stage);
    float* d_out = reinterpret_cast<float*>(static_cast<char*>(ctx->d_stage) + in_bytes);
    CU(ctx, cudaMemcpyAsync(d_in, subbands, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemsetAsync(d_out, 0, out_bytes, ctx->stream)); // the part of a plane a layer does not fill is defined as zero
    s = symgpu_mpa12_synth_dev(ctx, d_in, runs, n_runs, n_frames, n_slots, d_out);
    if (s != SYMGPU_OK) return s;
    CU(ctx, cudaMemcpyAsync(pcm, d_out, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return SYMGPU_OK;
}

} // extern "C"
