// FLAC integer restoration for sm_100a (SURVEY §8f N4): what FlacDecoder::decode_inner does after the Rice stage.
//   fixed_predict / lpc_predict   symphonia-bundle-flac/src/decoder.rs:663-752
//   samples_shl                   decoder.rs:387-394
//   decorrelate_*                 decoder.rs:32-82
//   sample << (32 - bps)          decoder.rs:237-240
// Integer arithmetic throughout, so the result is bit-exact by construction (wrapping i32 add / sub / shl, i64
// accumulation of the prediction, arithmetic right shift).
//
// The predictor is a recurrence over the samples of a sub-frame (serial), independent between sub-frames:
// flac_predict_kernel packs one sub-frame per lane, 8 per warp (a scheduler needs several such warps to stay busy),
// and moves the samples between global and shared memory with the whole warp, 32 samples of every sub-frame per
// round (one coalesced request per sub-frame), the fetch of round r+1 in flight during the recurrences of round r.
// Like the reference (decoder.rs:483-501) the predictor is instantiated for a few maximum orders with the
// coefficients zero-padded -- exact in integer arithmetic.  flac_finish_kernel then applies the channel
// decorrelation and the output scaling, element-wise and coalesced.  flac_finish_pack_kernel does the same and goes on
// to FromSample<i32> (symphonia-core/src/audio/conv.rs:514-532) and an interleaved store of the caller's format, so
// that only the packed samples leave the device (symgpu_flac_decode_*).
#include <cuda_runtime.h>

#include <cstdint>

#include "../../include/symgpu.h"
#include "flac_kernel.h"

namespace symgpu {
namespace {

constexpr int kFlacWarps = 4;
constexpr int kFlacPerWarp = 8;
constexpr int kStride = kFlacPerWarp + 1; // tile row stride in words: lanes of a row and rows of a column hit distinct banks

__device__ __forceinline__ int32_t wadd(int32_t a, int32_t b) { return (int32_t)((uint32_t)a + (uint32_t)b); }
__device__ __forceinline__ int32_t wsub(int32_t a, int32_t b) { return (int32_t)((uint32_t)a - (uint32_t)b); }
__device__ __forceinline__ int32_t wshl(int32_t a, unsigned s) { return (int32_t)((uint32_t)a << (s & 31u)); }

// One sample with the N-term predictor: h[j] = the restored sample j + 1 positions back.
template <int N>
__device__ __forceinline__ int32_t flac_step(int32_t residual, int32_t (&h)[32], const int32_t (&c)[32], unsigned shift) {
    long long acc = 0;
#pragma unroll
    for (int j = 0; j < N; ++j) acc += (long long)c[j] * (long long)h[j];
    const int32_t v = wadd(residual, (int32_t)(acc >> shift));
#pragma unroll
    for (int j = N - 1; j > 0; --j) h[j] = h[j - 1];
    h[0] = v;
    return v;
}

// `cnt` consecutive samples of one sub-frame, held in a column of the warp's tile (row stride kStride words).
// Samples before `order` are warm-up samples: they only enter the history.
template <int N>
__device__ __forceinline__ void flac_samples(int32_t* col, int cnt, int m0, int order, int32_t (&h)[32], const int32_t (&c)[32],
                                             unsigned shift, unsigned wasted) {
    int k = 0;
    for (; k < cnt && m0 + k < order; ++k) {
        const int32_t v = col[kStride * k];
#pragma unroll
        for (int j = N - 1; j > 0; --j) h[j] = h[j - 1];
        h[0] = v;
        col[kStride * k] = wshl(v, wasted);
    }
    for (; k + 4 <= cnt; k += 4) {
        int32_t x[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) x[u] = col[kStride * (k + u)];
#pragma unroll
        for (int u = 0; u < 4; ++u) x[u] = flac_step<N>(x[u], h, c, shift);
#pragma unroll
        for (int u = 0; u < 4; ++u) col[kStride * (k + u)] = wshl(x[u], wasted);
    }
    for (; k < cnt; ++k) col[kStride * k] = wshl(flac_step<N>(col[kStride * k], h, c, shift), wasted);
}

__global__ void __launch_bounds__(kFlacWarps * 32) flac_predict_kernel(const symgpu_flac_subframe* __restrict__ subs, uint32_t n_subs,
                                                                       int32_t* __restrict__ samples, unsigned long long n_samples) {
    __shared__ int32_t tile_s[kFlacWarps][32 * kStride];
    __shared__ int32_t* base_s[kFlacWarps][kFlacPerWarp];
    __shared__ int len_s[kFlacWarps][kFlacPerWarp];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int32_t* tile = tile_s[warp];
    const uint32_t i = (blockIdx.x * kFlacWarps + warp) * kFlacPerWarp + lane;
    int n = 0, type = SYMGPU_FLAC_VERBATIM, order = 0, bucket = 0;
    unsigned shift = 0, wasted = 0;
    int32_t* base = samples;
    int32_t c[32], h[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) c[j] = h[j] = 0;
    if (lane < kFlacPerWarp && i < n_subs) {
        const symgpu_flac_subframe* sf = subs + i;
        const unsigned long long off = sf->offset;
        const uint32_t len = sf->n;
        if (len > 0 && off + len <= n_samples) { // a sub-frame that leaves the buffer is not touched
            n = (int)len;
            base = samples + off;
            type = sf->type;
            wasted = sf->wasted;
            if (type == SYMGPU_FLAC_FIXED) {
                // s(i) = 1 s(i-1) | 2 s(i-1) - s(i-2) | 3 s(i-1) - 3 s(i-2) + s(i-3) | 4 s(i-1) - 6 s(i-2) + 4 s(i-3) - s(i-4)
                // (decoder.rs:672-705).  Written as a switch over literal coefficients: the first version derived
                // them from min(order, 4) with chained selects, which ptxas 12.9 compiled to a packed 16-bit min
                // whose predicate was wrong for order 1 (c[1] became -6) -- found by the GPU parity run.
                order = sf->order;
                switch (order) {
                    case 1: c[0] = 1; break;
                    case 2: c[0] = 2; c[1] = -1; break;
                    case 3: c[0] = 3; c[1] = -3; c[2] = 1; break;
                    case 4: c[0] = 4; c[1] = -6; c[2] = 4; c[3] = -1; break;
                    default: // order 0 predicts nothing; orders above 4 are refused by the host entry point
                        order = 0;
                        type = SYMGPU_FLAC_VERBATIM;
                        break;
                }
                bucket = 4;
            } else if (type == SYMGPU_FLAC_LPC) {
                order = min(max((int)sf->order, 1), 32);
                shift = sf->shift & 63u;
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (j < order) c[j] = sf->coeffs[j];
                bucket = order <= 4 ? 4 : order <= 6 ? 6 : order <= 8 ? 8 : order <= 10 ? 10 : order <= 12 ? 12 : 32;
            }
            order = min(order, n);
        }
    }
    if (lane < kFlacPerWarp) {
        base_s[warp][lane] = base;
        len_s[warp][lane] = n;
    }
    int max_len = n;
#pragma unroll
    for (int d = 16; d; d >>= 1) max_len = max(max_len, __shfl_xor_sync(0xffffffffu, max_len, d));
    __syncwarp();

    int32_t r[kFlacPerWarp]; // samples in flight: r[j] = sample (round * 32 + lane) of sub-frame j
    auto fetch = [&](int round) {
        const int m = round * 32 + lane;
#pragma unroll
        for (int j = 0; j < kFlacPerWarp; ++j) {
            r[j] = 0;
            if (m < len_s[warp][j]) r[j] = base_s[warp][j][m];
        }
    };
    fetch(0);
    int32_t constant = 0;
    for (int round = 0; round * 32 < max_len; ++round) {
#pragma unroll
        for (int j = 0; j < kFlacPerWarp; ++j) tile[kStride * lane + j] = r[j]; // row = sample in the round, column = sub-frame
        __syncwarp();
        if ((round + 1) * 32 < max_len) fetch(round + 1);
        const int m0 = round * 32;
        const int cnt = min(32, n - m0);
        if (cnt > 0) { // lanes >= kFlacPerWarp have n = 0
            int32_t* col = tile + lane;
            if (type == SYMGPU_FLAC_CONSTANT) { // decode_constant, decoder.rs:396-404
                if (round == 0) constant = col[0];
                for (int k = 0; k < cnt; ++k) col[kStride * k] = wshl(constant, wasted);
            } else if (type == SYMGPU_FLAC_VERBATIM) {
                if (wasted)
                    for (int k = 0; k < cnt; ++k) col[kStride * k] = wshl(col[kStride * k], wasted);
            } else {
                switch (bucket) {
                    case 4: flac_samples<4>(col, cnt, m0, order, h, c, shift, wasted); break;
                    case 6: flac_samples<6>(col, cnt, m0, order, h, c, shift, wasted); break;
                    case 8: flac_samples<8>(col, cnt, m0, order, h, c, shift, wasted); break;
                    case 10: flac_samples<10>(col, cnt, m0, order, h, c, shift, wasted); break;
                    case 12: flac_samples<12>(col, cnt, m0, order, h, c, shift, wasted); break;
                    default: flac_samples<32>(col, cnt, m0, order, h, c, shift, wasted); break;
                }
            }
        }
        __syncwarp();
        const int m = m0 + lane;
#pragma unroll
        for (int j = 0; j < kFlacPerWarp; ++j)
            if (m < len_s[warp][j]) base_s[warp][j][m] = tile[kStride * lane + j];
        __syncwarp();
    }
}

// One CTA per frame: channel decorrelation, then the scaling to 32 bits.
__global__ void __launch_bounds__(256) flac_finish_kernel(const symgpu_flac_frame* __restrict__ frames, const symgpu_flac_subframe* __restrict__ subs,
                                                          uint32_t n_subs, int32_t* __restrict__ samples, unsigned long long n_samples) {
    const symgpu_flac_frame fr = frames[blockIdx.x];
    const int channels = fr.channels;
    if (channels < 1 || channels > 8 || (unsigned long long)fr.first_subframe + channels > n_subs) return;
    const unsigned sh = fr.bits_per_sample < 32 ? 32u - fr.bits_per_sample : 0u;
    const symgpu_flac_subframe* s0 = subs + fr.first_subframe;
    if (fr.assignment != SYMGPU_FLAC_INDEPENDENT && channels == 2) {
        const uint32_t n = s0[0].n;
        if (s0[1].n != n || s0[0].offset + n > n_samples || s0[1].offset + n > n_samples) return;
        int32_t* a = samples + s0[0].offset;
        int32_t* b = samples + s0[1].offset;
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
            int32_t x = a[i], y = b[i];
            if (fr.assignment == SYMGPU_FLAC_LEFT_SIDE) { // right = left - side
                y = wsub(x, y);
            } else if (fr.assignment == SYMGPU_FLAC_MID_SIDE) {
                const int32_t mid = wshl(x, 1) | (y & 1);
                x = wadd(mid, y) >> 1;
                y = wsub(mid, y) >> 1;
            } else { // RIGHT_SIDE: plane 0 = side, plane 1 = right; left = side + right
                x = wadd(x, y);
            }
            a[i] = wshl(x, sh);
            b[i] = wshl(y, sh);
        }
    } else if (sh) {
        for (int ch = 0; ch < channels; ++ch) {
            const uint32_t n = s0[ch].n;
            if (s0[ch].offset + n > n_samples) continue;
            int32_t* a = samples + s0[ch].offset;
            for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) a[i] = wshl(a[i], sh);
        }
    }
}

// FromSample<i32> of conv.rs:514-532 for the output formats; every rule is exact.
template <int FMT>
struct FromS32;
template <>
struct FromS32<SYMGPU_FMT_F32> { // (s as f64 / 2^31) as f32: a power-of-two scale commutes with the rounding
    using T = float;
    static __device__ __forceinline__ T of(int32_t s) { return __int2float_rn(s) * 0x1p-31f; }
};
template <>
struct FromS32<SYMGPU_FMT_S16> {
    using T = int16_t;
    static __device__ __forceinline__ T of(int32_t s) { return (int16_t)(s >> 16); }
};
template <>
struct FromS32<SYMGPU_FMT_S24> { // i24::from(s >> 8), in the 4-byte container of the f32 output stage
    using T = int32_t;
    static __device__ __forceinline__ T of(int32_t s) { return s >> 8; }
};
template <>
struct FromS32<SYMGPU_FMT_S32> {
    using T = int32_t;
    static __device__ __forceinline__ T of(int32_t s) { return s; }
};
template <>
struct FromS32<SYMGPU_FMT_U8> {
    using T = uint8_t;
    static __device__ __forceinline__ T of(int32_t s) { return (uint8_t)(((uint32_t)s + 0x80000000u) >> 24); }
};

// flac_finish_kernel followed by the output stage: one CTA per frame decorrelates, scales to 32 bits, converts to FMT and
// stores frame f interleaved at out[dst[f] ..], n * channels samples.  The restored planes are only read.  A frame whose
// descriptors leave `samples` or `out`, or whose sub-frames disagree on the block size, is not written.
template <int FMT>
__global__ void __launch_bounds__(256) flac_finish_pack_kernel(const symgpu_flac_frame* __restrict__ frames, const symgpu_flac_subframe* __restrict__ subs,
                                                               uint32_t n_subs, const int32_t* __restrict__ samples, unsigned long long n_samples,
                                                               const unsigned long long* __restrict__ dst, void* __restrict__ out_v,
                                                               unsigned long long out_samples) {
    using C = FromS32<FMT>;
    using T = typename C::T;
    const symgpu_flac_frame fr = frames[blockIdx.x];
    const int channels = fr.channels;
    if (channels < 1 || channels > 8 || (unsigned long long)fr.first_subframe + channels > n_subs) return;
    const symgpu_flac_subframe* s0 = subs + fr.first_subframe;
    const uint32_t n = s0[0].n;
    const unsigned long long d = dst[blockIdx.x];
    if (d > out_samples || (unsigned long long)n * channels > out_samples - d) return;
    for (int ch = 0; ch < channels; ++ch)
        if (s0[ch].n != n || s0[ch].offset + n > n_samples) return;
    const unsigned sh = fr.bits_per_sample < 32 ? 32u - fr.bits_per_sample : 0u;
    T* __restrict__ out = static_cast<T*>(out_v) + d;
    if (fr.assignment != SYMGPU_FLAC_INDEPENDENT && channels == 2) {
        const int32_t* a = samples + s0[0].offset;
        const int32_t* b = samples + s0[1].offset;
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
            int32_t x = __ldg(a + i), y = __ldg(b + i);
            if (fr.assignment == SYMGPU_FLAC_LEFT_SIDE) { // as flac_finish_kernel
                y = wsub(x, y);
            } else if (fr.assignment == SYMGPU_FLAC_MID_SIDE) {
                const int32_t mid = wshl(x, 1) | (y & 1);
                x = wadd(mid, y) >> 1;
                y = wsub(mid, y) >> 1;
            } else {
                x = wadd(x, y);
            }
            out[2 * i] = C::of(wshl(x, sh));
            out[2 * i + 1] = C::of(wshl(y, sh));
        }
    } else {
        // one output sample per step: the stores of a warp are consecutive
        const uint32_t total = n * (uint32_t)channels;
        for (uint32_t j = threadIdx.x; j < total; j += blockDim.x) {
            const uint32_t i = j / channels, c = j - i * channels;
            out[j] = C::of(wshl(__ldg(samples + s0[c].offset + i), sh));
        }
    }
}

template <int FMT>
void finish_pack_as(const symgpu_flac_frame* frames, uint32_t n_frames, const symgpu_flac_subframe* subs, uint32_t n_subs, const int32_t* samples,
                    size_t n_samples, const uint64_t* dst, void* out, size_t out_samples, cudaStream_t stream) {
    flac_finish_pack_kernel<FMT><<<n_frames, 256, 0, stream>>>(frames, subs, n_subs, samples, n_samples,
                                                               reinterpret_cast<const unsigned long long*>(dst), out, out_samples);
}

} // namespace

cudaError_t flac_decode_launch(const symgpu_flac_frame* frames, uint32_t n_frames, const symgpu_flac_subframe* subs, uint32_t n_subs,
                               int32_t* samples, size_t n_samples, const uint64_t* dst, int format, void* out, size_t out_samples,
                               cudaStream_t stream) {
    if (format < SYMGPU_FMT_F32 || format > SYMGPU_FMT_U8) return cudaErrorInvalidValue;
    if (n_subs) {
        const unsigned per_block = kFlacWarps * kFlacPerWarp;
        flac_predict_kernel<<<(n_subs + per_block - 1) / per_block, kFlacWarps * 32, 0, stream>>>(subs, n_subs, samples, n_samples);
    }
    if (n_frames) {
        switch (format) {
        case SYMGPU_FMT_F32: finish_pack_as<SYMGPU_FMT_F32>(frames, n_frames, subs, n_subs, samples, n_samples, dst, out, out_samples, stream); break;
        case SYMGPU_FMT_S16: finish_pack_as<SYMGPU_FMT_S16>(frames, n_frames, subs, n_subs, samples, n_samples, dst, out, out_samples, stream); break;
        case SYMGPU_FMT_S24: finish_pack_as<SYMGPU_FMT_S24>(frames, n_frames, subs, n_subs, samples, n_samples, dst, out, out_samples, stream); break;
        case SYMGPU_FMT_S32: finish_pack_as<SYMGPU_FMT_S32>(frames, n_frames, subs, n_subs, samples, n_samples, dst, out, out_samples, stream); break;
        default: finish_pack_as<SYMGPU_FMT_U8>(frames, n_frames, subs, n_subs, samples, n_samples, dst, out, out_samples, stream); break;
        }
    }
    return cudaGetLastError();
}

cudaError_t flac_launch(const symgpu_flac_frame* frames, uint32_t n_frames, const symgpu_flac_subframe* subs, uint32_t n_subs,
                        int32_t* samples, size_t n_samples, cudaStream_t stream) {
    if (n_subs) {
        const unsigned per_block = kFlacWarps * kFlacPerWarp;
        flac_predict_kernel<<<(n_subs + per_block - 1) / per_block, kFlacWarps * 32, 0, stream>>>(subs, n_subs, samples, n_samples);
    }
    if (n_frames) flac_finish_kernel<<<n_frames, 256, 0, stream>>>(frames, subs, n_subs, samples, n_samples);
    return cudaGetLastError();
}

} // namespace symgpu
