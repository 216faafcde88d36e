// Fused step metrics (SURVEY 8f-2): everything Base_Lightning.calculate_losses_step derives from (y_pred, y) besides the
// gradient-carrying loss, in two launches and without a host sync.
//
//  Replaces, for the classification head (gnnLightning.py:L131-151, L285-348; customMetrics.py:L6-54):
//    softmax per foot -> 16-class conversion (product of per-foot probabilities) -> argmax -> MulticlassAccuracy;
//    per-foot argmax -> four BinaryF1Score (the reference: 4 sklearn confusion matrices on the host + a python loop over B);
//    CrossEntropyLossMetric (sum-reduced CE / rows).
//  The 16-class argmax equals "every foot's 2-way argmax" (the joint probability factorises; torch.argmax takes the first
//  maximum, i.e. class 0 on a per-foot tie, which is what the per-foot rule below does too).
//  For the regression heads (L124-130): sum of squared / absolute errors -> MSE, RMSE, L1.
//  COM momentum (gnnLightning_com.py:L70-95): MSE / RMSE over [n, n_base*6], MSE of the lin and ang halves of every base, and
//    CosineSimilarityMetric of the un-standardised lin and ang 3-vectors of base 0.
//  World-frame GRF (gnnLightning.py:L287-311): the body-frame MSE / RMSE / L1, and the same after rotating each foot's force
//    by R(q)^T (q normalised here), optionally on the z components only.
//  Deterministic: per-block partials in fixed order, summed by one final block; no atomics.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mshgnn_b200.h"

namespace mshgnn {

constexpr int MET_SLOTS = 32;
constexpr int MET_BLOCKS = 296;
// slots: classification  0 ce_sum  1 rows  2 graphs_all_feet_right  3 graphs  4+4*leg+{0,1,2,3} tp fp fn tn
//                        20 ce_mean (fp32-rounded like the reference)  21 accuracy  22..25 F1 of leg 0..3
//        regression      0 sse  1 sae  2 n   20 mse  21 rmse  22 l1
//        COM             0 sse  1 n  2 sse_lin  3 sse_ang  4 n_lin (= n_ang)  5 cos_lin sum  6 cos_ang sum  7 rows
//                        20 mse  21 rmse  22 mse_lin  23 mse_ang  24 cos_sim_lin  25 cos_sim_ang  26 avg_cos_sim
//        GRF world frame 0 sse  1 sae  2 n (body frame)  3 sse  4 sae  5 n (world frame)
//                        20 mse  21 rmse  22 l1  23 mse_world  24 rmse_world  25 l1_world
constexpr int MET_CE2 = MSHGNN_LOSS_CE2, MET_COM = MSHGNN_METRIC_COM, MET_GRF_WORLD = MSHGNN_METRIC_GRF_WORLD;

__device__ __forceinline__ double met_label(const void* p, int dtype, int64_t i) {
    if (dtype == 1) return ((const double*)p)[i];
    if (dtype == 2) return (double)((const long long*)p)[i];
    return (double)((const float*)p)[i];
}

// block sum of the 20 per-thread states into this block's partial row (fixed order: warp shuffle, then warps 0..7)
__device__ __forceinline__ void met_block_partial(const double (&a)[20], double (&sh)[8][MET_SLOTS], double* __restrict__ partial) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 20; ++i) {
        double v = a[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) sh[wid][i] = v;
    }
    __syncthreads();
    if (threadIdx.x < 20) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += sh[w][threadIdx.x];
        partial[(int64_t)blockIdx.x * MET_SLOTS + threadIdx.x] = s;
    }
}

__global__ void __launch_bounds__(256)
k_metrics_partial(const int kind, const int feet, const float* __restrict__ out, const void* __restrict__ labels, const int label_dtype,
                  const int64_t n, double* __restrict__ partial) {
    __shared__ double sh[8][MET_SLOTS];
    double a[20];
#pragma unroll
    for (int i = 0; i < 20; ++i) a[i] = 0.0;
    const int64_t stride = (int64_t)gridDim.x * 256;
    if (kind == 1) {
        // n = graphs; out [n*feet, 2] logits, labels [n, feet] in {0,1}
        for (int64_t g = (int64_t)blockIdx.x * 256 + threadIdx.x; g < n; g += stride) {
            bool all_ok = true;
            for (int f = 0; f < feet; ++f) {
                const int64_t r = g * feet + f;
                const float2 l = *reinterpret_cast<const float2*>(out + 2 * r);
                const int y = met_label(labels, label_dtype, r) != 0.0;
                const double l0 = (double)l.x, l1 = (double)l.y;
                const double m = l0 > l1 ? l0 : l1;
                a[0] += m + log(exp(l0 - m) + exp(l1 - m)) - (y ? l1 : l0);
                const int p = l.y > l.x;           // argmax of the 2-way softmax, first maximum on ties
                all_ok = all_ok && (p == y);
                if (f < 4) a[4 + 4 * f + (p ? (y ? 0 : 1) : (y ? 2 : 3))] += 1.0;
            }
            a[1] += (double)feet; a[2] += all_ok ? 1.0 : 0.0; a[3] += 1.0;
        }
    } else {
        for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
            const double d = (double)out[i] - met_label(labels, label_dtype, i);
            a[0] += d * d; a[1] += fabs(d); a[2] += 1.0;
        }
    }
    met_block_partial(a, sh, partial);
}

// torch.nn.functional.cosine_similarity(x1, x2, dim=1, eps=1e-8) of one row of 3-vectors: each vector is divided by its
// norm clamped to eps before the product (so a zero vector gives 0), as ATen's cosine_similarity does
__device__ __forceinline__ double met_cos3(const double* x1, const double* x2) {
    const double n1 = fmax(sqrt(x1[0] * x1[0] + x1[1] * x1[1] + x1[2] * x1[2]), 1e-8);
    const double n2 = fmax(sqrt(x2[0] * x2[0] + x2[1] * x2[1] + x2[2] * x2[2]), 1e-8);
    return (x1[0] / n1) * (x2[0] / n2) + (x1[1] / n1) * (x2[1] / n2) + (x1[2] / n1) * (x2[2] / n2);
}

// n = rows (graphs).  COM: out / labels [n, n_base*6].  GRF world frame: out / labels [n, 12], quaternions [n, 4].
__global__ void __launch_bounds__(256)
k_metrics_partial_ex(const int kind, const mshgnn_metric_args args, const float* __restrict__ out, const void* __restrict__ labels,
                     const int label_dtype, const int64_t n, double* __restrict__ partial) {
    __shared__ double sh[8][MET_SLOTS];
    double a[20];
#pragma unroll
    for (int i = 0; i < 20; ++i) a[i] = 0.0;
    const int64_t stride = (int64_t)gridDim.x * 256;
    if (kind == MET_COM) {
        const int w = args.n_base * 6;
        double mean[6], sd[6];
#pragma unroll
        for (int c = 0; c < 6; ++c) { mean[c] = args.y_mean[c]; sd[c] = args.y_std[c]; }
        for (int64_t g = (int64_t)blockIdx.x * 256 + threadIdx.x; g < n; g += stride) {
            double pu[6], yu[6];
            for (int b = 0; b < args.n_base; ++b) {
#pragma unroll
                for (int c = 0; c < 6; ++c) {
                    const int64_t i = g * w + b * 6 + c;
                    const double p = (double)out[i], y = met_label(labels, label_dtype, i);
                    const double d = p - y;
                    a[0] += d * d;
                    a[c < 3 ? 2 : 3] += d * d;
                    if (b == 0) {
                        // Standarizer.unstandarize: yn * std + mean, rounded twice as torch does (no FMA contraction)
                        pu[c] = __dadd_rn(__dmul_rn(p, sd[c]), mean[c]);
                        yu[c] = __dadd_rn(__dmul_rn(y, sd[c]), mean[c]);
                    }
                }
            }
            a[1] += (double)w; a[4] += (double)(w / 2);
            a[5] += met_cos3(pu, yu); a[6] += met_cos3(pu + 3, yu + 3); a[7] += 1.0;
        }
    } else {
        for (int64_t g = (int64_t)blockIdx.x * 256 + threadIdx.x; g < n; g += stride) {
            double q[4];
#pragma unroll
            for (int c = 0; c < 4; ++c)
                q[c] = args.quat_dtype == MSHGNN_F64 ? ((const double*)args.quat)[g * 4 + c] : (double)((const float*)args.quat)[g * 4 + c];
            const double qn = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
            const double x = q[0] / qn, y = q[1] / qn, z = q[2] / qn, s = q[3] / qn;
            // R(q) of body_frame_to_world_frame, row-major; the world-frame force is R^T f
            const double R[9] = {1 - 2 * (y * y + z * z), 2 * (x * y - z * s), 2 * (x * z + y * s),
                                 2 * (x * y + z * s), 1 - 2 * (x * x + z * z), 2 * (y * z - x * s),
                                 2 * (x * z - y * s), 2 * (y * z + x * s), 1 - 2 * (x * x + y * y)};
#pragma unroll
            for (int f = 0; f < 4; ++f) {
                double p[3], t[3];
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const int64_t i = g * 12 + f * 3 + j;
                    p[j] = (double)out[i]; t[j] = met_label(labels, label_dtype, i);
                    const double d = p[j] - t[j];
                    a[0] += d * d; a[1] += fabs(d);
                }
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    if (args.z_only && c != 2) continue;
                    const double pw = R[c] * p[0] + R[3 + c] * p[1] + R[6 + c] * p[2];
                    const double tw = R[c] * t[0] + R[3 + c] * t[1] + R[6 + c] * t[2];
                    const double d = pw - tw;
                    a[3] += d * d; a[4] += fabs(d);
                }
            }
            a[2] += 12.0; a[5] += args.z_only ? 4.0 : 12.0;
        }
    }
    met_block_partial(a, sh, partial);
}

__global__ void __launch_bounds__(32)
k_metrics_final(const int kind, const double* __restrict__ partial, const int n_blocks, double* __restrict__ batch, double* __restrict__ epoch) {
    __shared__ double s[MET_SLOTS];
    const int t = threadIdx.x;
    double v = 0.0;
    if (t < 20)
        for (int b = 0; b < n_blocks; ++b) v += partial[(int64_t)b * MET_SLOTS + t];
    s[t] = v;
    __syncwarp();
    double d = 0.0;
    auto f1 = [&](int leg) {
        const double tp = s[4 + 4 * leg], fp = s[5 + 4 * leg], fn = s[6 + 4 * leg];
        const double pr = tp / (tp + fp), rc = tp / (tp + fn);
        const double f = 2.0 * (pr * rc) / (pr + rc);
        return f != f ? 0.0 : f;                   // torch.nan_to_num (customMetrics.py:L54)
    };
    if (kind == MET_CE2) {
        if (t == 20) d = (double)((float)s[0] / (float)s[1]);          // summed_loss.float() / total_num (customMetrics.py:L25)
        else if (t == 21) d = s[2] / s[3];
        else if (t >= 22 && t < 26) d = f1(t - 22);
    } else if (kind == MET_COM) {
        if (t == 20) d = s[0] / s[1];
        else if (t == 21) d = sqrt(s[0] / s[1]);
        else if (t == 22) d = s[2] / s[4];
        else if (t == 23) d = s[3] / s[4];
        else if (t == 24) d = s[5] / s[7];
        else if (t == 25) d = s[6] / s[7];
        else if (t == 26) d = (s[5] / s[7] + s[6] / s[7]) / 2;
    } else if (kind == MET_GRF_WORLD) {
        if (t == 20) d = s[0] / s[2];
        else if (t == 21) d = sqrt(s[0] / s[2]);
        else if (t == 22) d = s[1] / s[2];
        else if (t == 23) d = s[3] / s[5];
        else if (t == 24) d = sqrt(s[3] / s[5]);
        else if (t == 25) d = s[4] / s[5];
    } else {
        if (t == 20) d = s[0] / s[2];
        else if (t == 21) d = sqrt(s[0] / s[2]);
        else if (t == 22) d = s[1] / s[2];
    }
    batch[t] = t < 20 ? v : d;
    if (epoch != nullptr && t < 20) epoch[t] += v;
}

}  // namespace mshgnn
