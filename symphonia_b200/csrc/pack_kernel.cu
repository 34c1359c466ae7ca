// Output stage: planar f32 PCM -> trimmed, interleaved samples of the caller's format (SURVEY §8f N3).
//
// Replaces AudioBuffer::trim (symphonia-core/src/audio/buf.rs:404-433), copy_to_slice_interleaved
// (buf.rs:469-476) and FromSample<f32> (audio/conv.rs:592-607) for a whole batch.  Pure streaming:
// 4 bytes read per sample, 1-4 written; bound by HBM.  One CTA walks spans grid-stride; for stereo
// spans whose source and destination are 16-byte aligned each thread converts four frames from two
// float4 loads and writes them with one or two 16-byte stores, otherwise one frame per thread.  The MAPPED instances read
// output channel c from plane map(c) instead of plane c (symgpu_pcm_pack_mapped_*); the unmapped ones are unchanged by that.
#include "pack_kernel.h"

namespace symgpu {
namespace {

__device__ __forceinline__ float clamp_unit(float v) {
    // util.rs:258-266: two selects, so a NaN passes through unchanged.
    float c = v > 1.0f ? 1.0f : v;
    c = c < -1.0f ? -1.0f : c;
    return c;
}

// Rust's float -> int `as`: toward zero, saturating, NaN -> 0; cvt.rzi.s32 does exactly that for i32.
template <int FMT>
struct Conv;
template <>
struct Conv<SYMGPU_FMT_F32> {
    using T = float;
    static __device__ __forceinline__ T of(float s) { return s; }
};
template <>
struct Conv<SYMGPU_FMT_S16> {
    using T = int16_t;
    static __device__ __forceinline__ T of(float s) {
        const int v = __float2int_rz(clamp_unit(s) * 32768.0f);
        return (int16_t)min(max(v, -32768), 32767);
    }
};
template <>
struct Conv<SYMGPU_FMT_S24> {
    using T = int32_t;
    static __device__ __forceinline__ T of(float s) {
        const int v = __float2int_rz(clamp_unit(s) * 8388608.0f);
        return min(max(v, -8388608), 8388607); // clamp_i24, util.rs:230-237
    }
};
template <>
struct Conv<SYMGPU_FMT_S32> {
    using T = int32_t;
    static __device__ __forceinline__ T of(float s) {
        // cvt.rzi.s32.f64 turns a NaN into INT_MIN (the f32 form gives 0), Rust's `as` gives 0.
        const float c = clamp_unit(s);
        return c != c ? 0 : __double2int_rz((double)c * 2147483648.0);
    }
};
template <>
struct Conv<SYMGPU_FMT_U8> {
    using T = uint8_t;
    static __device__ __forceinline__ T of(float s) {
        const int v = __float2int_rz((clamp_unit(s) + 1.0f) * 128.0f);
        return (uint8_t)min(max(v, 0), 255);
    }
};

template <typename T>
struct alignas(sizeof(T) * 8) Vec8 { // four stereo frames
    T v[8];
};

template <bool MAPPED>
__device__ __forceinline__ uint32_t plane_of(uint32_t plane_map, uint32_t c) {
    return MAPPED ? (plane_map >> (4 * c)) & 15u : c;
}

template <int FMT, bool MAPPED>
__global__ void __launch_bounds__(256) pack_kernel(PackArgs a) {
    using C = Conv<FMT>;
    using T = typename C::T;
    T* __restrict__ out = static_cast<T*>(a.out);
    const float* __restrict__ pcm = a.pcm;
    const uint32_t map = a.plane_map;
    for (uint32_t p = blockIdx.x; p < a.n_spans; p += gridDim.x) {
        uint64_t src, dst;
        uint32_t stride, kept;
        if (a.spans) {
            const symgpu_pcm_span sp = a.spans[p];
            uint32_t n = sp.frames > sp.trim_end ? sp.frames - sp.trim_end : 0;
            kept = sp.trim_start >= n ? 0 : n - sp.trim_start;
            src = sp.src + sp.trim_start;
            stride = sp.plane_stride;
            dst = sp.dst_frame;
        } else {
            src = (uint64_t)p * a.channels * a.plane_stride;
            stride = a.plane_stride;
            kept = a.frames;
            dst = (uint64_t)p * a.frames;
        }
        if (a.channels == 2 && ((src | stride | dst) & 3) == 0) {
            const uint64_t s0 = src + (uint64_t)plane_of<MAPPED>(map, 0) * stride, s1 = src + (uint64_t)plane_of<MAPPED>(map, 1) * stride;
            const float4* p0 = reinterpret_cast<const float4*>(pcm + s0);
            const float4* p1 = reinterpret_cast<const float4*>(pcm + s1);
            Vec8<T>* o = reinterpret_cast<Vec8<T>*>(out + dst * 2);
            const uint32_t quads = kept >> 2;
            for (uint32_t q = threadIdx.x; q < quads; q += blockDim.x) {
                const float4 l = __ldg(p0 + q), r = __ldg(p1 + q);
                Vec8<T> w;
                w.v[0] = C::of(l.x); w.v[1] = C::of(r.x);
                w.v[2] = C::of(l.y); w.v[3] = C::of(r.y);
                w.v[4] = C::of(l.z); w.v[5] = C::of(r.z);
                w.v[6] = C::of(l.w); w.v[7] = C::of(r.w);
                o[q] = w;
            }
            for (uint32_t i = (quads << 2) + threadIdx.x; i < kept; i += blockDim.x) {
                out[(dst + i) * 2] = C::of(__ldg(pcm + s0 + i));
                out[(dst + i) * 2 + 1] = C::of(__ldg(pcm + s1 + i));
            }
        } else {
            const uint32_t ch = a.channels;
            for (uint32_t i = threadIdx.x; i < kept; i += blockDim.x) {
                uint32_t m = map; // (shifted per channel: indexing it by (4 * c) makes ptxas spill)
                for (uint32_t c = 0; c < ch; ++c, m >>= 4)
                    out[(dst + i) * ch + c] = C::of(__ldg(pcm + src + (uint64_t)(MAPPED ? m & 15u : c) * stride + i));
            }
        }
    }
}

// Quantised spectra -> f32: value = sign(q) * POW43[|q|] (requantize.rs:23-32, :128, :144), eight lines per
// thread.  q = 0 gives +0.0, as read_huffman_samples does (requantize.rs:131-133).
__global__ void __launch_bounds__(256) dequant_kernel(const int4* __restrict__ q8, float4* __restrict__ out, size_t n8,
                                                      const float* __restrict__ pow43) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
        const int4 w = __ldg(q8 + i);
        const int words[4] = {w.x, w.y, w.z, w.w};
        float v[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int lo = (int)(short)(words[k] & 0xffff), hi = words[k] >> 16;
            const float a = __ldg(pow43 + min(abs(lo), 8207)), b = __ldg(pow43 + min(abs(hi), 8207));
            v[2 * k] = lo < 0 ? -a : a;
            v[2 * k + 1] = hi < 0 ? -b : b;
        }
        out[2 * i] = make_float4(v[0], v[1], v[2], v[3]);
        out[2 * i + 1] = make_float4(v[4], v[5], v[6], v[7]);
    }
}

} // namespace

cudaError_t dequant_launch(const int16_t* q, float* spectra, size_t n, const float* pow43, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    if (n % 8) return cudaErrorInvalidValue;
    const size_t n8 = n / 8;
    const unsigned grid = (unsigned)((n8 + 255) / 256 < 148u * 16u ? (n8 + 255) / 256 : 148u * 16u);
    dequant_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const int4*>(q), reinterpret_cast<float4*>(spectra), n8, pow43);
    return cudaGetLastError();
}

namespace {

template <bool MAPPED>
cudaError_t pack_launch_as(const PackArgs& a, int format, unsigned grid, cudaStream_t stream) {
    switch (format) {
    case SYMGPU_FMT_F32: pack_kernel<SYMGPU_FMT_F32, MAPPED><<<grid, 256, 0, stream>>>(a); break;
    case SYMGPU_FMT_S16: pack_kernel<SYMGPU_FMT_S16, MAPPED><<<grid, 256, 0, stream>>>(a); break;
    case SYMGPU_FMT_S24: pack_kernel<SYMGPU_FMT_S24, MAPPED><<<grid, 256, 0, stream>>>(a); break;
    case SYMGPU_FMT_S32: pack_kernel<SYMGPU_FMT_S32, MAPPED><<<grid, 256, 0, stream>>>(a); break;
    case SYMGPU_FMT_U8: pack_kernel<SYMGPU_FMT_U8, MAPPED><<<grid, 256, 0, stream>>>(a); break;
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

} // namespace

cudaError_t pack_launch(const PackArgs& a, int format, cudaStream_t stream, bool mapped) {
    if (a.n_spans == 0) return cudaSuccess;
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    }
    const unsigned cap = (unsigned)sms * 8;
    const unsigned grid = a.n_spans < cap ? a.n_spans : cap;
    return mapped ? pack_launch_as<true>(a, format, grid, stream) : pack_launch_as<false>(a, format, grid, stream);
}

} // namespace symgpu
