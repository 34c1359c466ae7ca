// Host <-> kernel interface of the output stage (pack_kernel.cu).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "../../include/symgpu.h"

namespace symgpu {

struct PackArgs {
    const float* pcm;
    const symgpu_pcm_span* spans; // nullptr: uniform packets (see symgpu_pcm_pack_dev)
    uint32_t n_spans;
    uint32_t channels;
    uint32_t plane_stride;
    uint32_t frames;
    void* out;
    uint32_t plane_map;           // with `mapped`: output channel c reads plane (plane_map >> 4c) & 15
};

// mapped = false: output channel c reads plane c (plane_map unused).
cudaError_t pack_launch(const PackArgs& a, int format, cudaStream_t stream, bool mapped = false);
// spectra[i] = sign(q[i]) * pow43[|q[i]|] for n values (n a multiple of 8, both pointers 16-byte aligned).
cudaError_t dequant_launch(const int16_t* q, float* spectra, size_t n, const float* pow43, cudaStream_t stream);

} // namespace symgpu
