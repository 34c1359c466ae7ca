// Host <-> kernel interface of the FLAC integer restoration (flac_kernel.cu).
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

#include "../../include/symgpu.h"

namespace symgpu {

// Two launches on `stream`: the predictors of all sub-frames, then decorrelation + output scaling per frame.
cudaError_t flac_launch(const symgpu_flac_frame* frames, uint32_t n_frames, const symgpu_flac_subframe* subs, uint32_t n_subs,
                        int32_t* samples, size_t n_samples, cudaStream_t stream);
// The predictors in place on `samples`, then per frame decorrelation + scaling + conversion to `format` (SYMGPU_FMT_*) into
// out[dst[f] ..] (out_samples samples of that format), interleaved; the restored planes are not written back.
cudaError_t flac_decode_launch(const symgpu_flac_frame* frames, uint32_t n_frames, const symgpu_flac_subframe* subs, uint32_t n_subs,
                               int32_t* samples, size_t n_samples, const uint64_t* dst, int format, void* out, size_t out_samples,
                               cudaStream_t stream);

} // namespace symgpu
