// Hidden widths below 128 (MSHGNN_PLAN_PAD_HIDDEN): the model runs as the 128-wide one whose weights are its zero-padded
// copy.  With zero rows / columns / biases, every padded channel's pre-activation is exactly 0 (ReLU gives 0, its mask bit
// is 0), every product that touches one is exactly 0, and so the real channels - and their gradients - are bit for bit
// those of that 128-wide model.  These two kernels move the parameters and gradients between the caller's layout
// (the model's own width) and the kernels' layout, tensor by tensor through the plan's PadSeg table.
#pragma once
#include "common.cuh"

namespace mshgnn {

constexpr int PAD_BLOCKS_X = 4;      // CTAs per tensor (grid.y = tensors): a 128 x 128 tensor is 16 float4 stores per thread
constexpr int PAD_MAX_GRID_Y = 65535;

__device__ __forceinline__ float pad_at(const PadSeg& s, const float* __restrict__ ext, const int r, const int c) {
    return (r < s.rows && c < s.cols) ? __ldg(ext + s.ext_off + (int64_t)r * s.cols + c) : 0.f;
}

// internal[seg] = zero-padded external[seg] for every tensor: every internal element is written, zeros included, so the
// result does not depend on what an earlier call left in the workspace.  Segments are blockIdx.y, blockIdx.y + gridDim.y, ...
// (a mixed plan's table can hold more segments than grid.y allows).  blockIdx.z = model of a model batch on a plan of one
// model (row z of both, strides ext_n / in_n); a mixed plan's table has absolute offsets and launches z = 1 with strides 0.
__global__ void __launch_bounds__(256)
k_pad_params(const PadSeg* __restrict__ segs, const int n_segs, const float* __restrict__ ext, float* __restrict__ in, const int64_t ext_n,
             const int64_t in_n) {
    ext += blockIdx.z * ext_n;
    in += blockIdx.z * in_n;
    const int stride = gridDim.x * blockDim.x;
    const int t0 = blockIdx.x * blockDim.x + threadIdx.x;
    for (int y = blockIdx.y; y < n_segs; y += gridDim.y) {
        const PadSeg s = segs[y];
        const int n = s.rows_i * s.cols_i;                            // < 2^30 (build_plan)
        float* dst = in + s.int_off;
        if ((s.cols_i & 3) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {     // four consecutive elements share a row: one 16-byte store
            for (int q = t0; q < n / 4; q += stride) {
                const int r = q * 4 / s.cols_i, c = q * 4 - r * s.cols_i;
                reinterpret_cast<float4*>(dst)[q] = make_float4(pad_at(s, ext, r, c), pad_at(s, ext, r, c + 1), pad_at(s, ext, r, c + 2),
                                                                pad_at(s, ext, r, c + 3));
            }
        } else {
            for (int i = t0; i < n; i += stride) {
                const int r = i / s.cols_i, c = i - r * s.cols_i;
                dst[i] = pad_at(s, ext, r, c);
            }
        }
    }
}

// external[seg] = top-left block of internal[seg] for the tensors segs[0 .. n_segs): every external element is written.
// Segments, models and strides as k_pad_params.
__global__ void __launch_bounds__(256)
k_compact_grads(const PadSeg* __restrict__ segs, const int n_segs, const float* __restrict__ in, float* __restrict__ ext, const int64_t in_n,
                const int64_t ext_n) {
    in += blockIdx.z * in_n;
    ext += blockIdx.z * ext_n;
    const int stride = gridDim.x * blockDim.x;
    for (int y = blockIdx.y; y < n_segs; y += gridDim.y) {
        const PadSeg s = segs[y];
        const int n = s.rows * s.cols;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
            const int r = i / s.cols, c = i - r * s.cols;
            ext[s.ext_off + i] = in[s.int_off + (int64_t)r * s.cols_i + c];
        }
    }
}

}  // namespace mshgnn
