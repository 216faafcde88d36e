// fp32 SIMT kernels of the MS-HGNN hot path (MSHGNN_MODE_FP32): the parity backbone.
//
//  k_rowgemm   : D[128 rows, 128] = sum_chunks A_c[rows, K_c] * Wt_c[K_c, 128]  + fused epilogue
//                (bias, ReLU, positivity mask, residual, ReLU bitmask out, masked second output).
//                Serves the encoder (A = caller's x rows with the +-1 symmetry signs folded into
//                the load: apply_symmetry, hgnn_k4.py:L198-237), every HeteroConv/GraphConv layer
//                (hgnn_k4.py:L170-186), base_transform, and the dX half of the backward pass.
//  k_reducegemm: dW[128, K] = sum_pairs dC[rows,128]^T * A[rows, K]  split over row ranges,
//                + column sums of dC (bias gradients); deterministic two-stage reduction.
//  k_encoder_dx: dx[rows, K] = sign * (dpre0[rows, 128] W_enc[128, K]): the input gradient (mshgnn_input_grad).
//  k_decoder_* : Linear(H, C) on the decoded node type + output signs (hgnn_c2.py:L184-189,
//                hgnn_k4_com.py:L157-165) and its backward.
//  k_loss_*    : MSE / per-row 2-way CE heads (gnnLightning.py:L124-139, customMetrics.py:L6-25).
#pragma once
#include "../../include/mshgnn_b200.h"
#include "common.cuh"

namespace mshgnn {

// node-feature element type of the caller's x tensors, as the kernels carry it ("x_f64" arguments): 0 fp32, 1 fp64, 2 fp16
__device__ __forceinline__ float ld_x(const void* base, int dtype_f64, int64_t idx) {
    if (dtype_f64 == 2) return __half2float(__ldg((const __half*)base + idx));
    return dtype_f64 ? (float)__ldg((const double*)base + idx) : __ldg((const float*)base + idx);
}

// (hi, lo) fp16 image of 4 consecutive values: hi = fp16(v), lo = fp16((v - hi) * 2^11)  (see kernels_tc.cuh)
__device__ __forceinline__ void split_store4(__half* hi, __half* lo, int64_t off, const float (&v)[4]) {
    __half2 h[2], l[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const __half ha = __float2half_rn(v[2 * j]), hb = __float2half_rn(v[2 * j + 1]);
        h[j] = __halves2half2(ha, hb);
        l[j] = __halves2half2(__float2half_rn((v[2 * j] - __half2float(ha)) * LO_SCALE), __float2half_rn((v[2 * j + 1] - __half2float(hb)) * LO_SCALE));
    }
    *reinterpret_cast<uint2*>(hi + off) = *reinterpret_cast<uint2*>(h);
    *reinterpret_cast<uint2*>(lo + off) = *reinterpret_cast<uint2*>(l);
}

// 4 consecutive activations from the fp32 slab, or (tensor-core modes: no fp32 slab) rebuilt from the (hi, lo) images
__device__ __forceinline__ float4 load_h4(const float* slab, const __half* hi, const __half* lo, int64_t off) {
    if (slab) return *reinterpret_cast<const float4*>(slab + off);
    const uint2 a = *reinterpret_cast<const uint2*>(hi + off), b = *reinterpret_cast<const uint2*>(lo + off);
    const float2 a0 = __half22float2(*reinterpret_cast<const __half2*>(&a.x)), a1 = __half22float2(*reinterpret_cast<const __half2*>(&a.y));
    const float2 b0 = __half22float2(*reinterpret_cast<const __half2*>(&b.x)), b1 = __half22float2(*reinterpret_cast<const __half2*>(&b.y));
    const float u = 1.f / LO_SCALE;
    return make_float4(fmaf(b0.x, u, a0.x), fmaf(b0.y, u, a0.y), fmaf(b1.x, u, a1.x), fmaf(b1.y, u, a1.y));
}

// ------------------------------------------------------------------------------------------
// row-GEMM
// ------------------------------------------------------------------------------------------
constexpr int RG_BK = 16;
constexpr int RG_AS = TILE_M + 4;   // padded leading dimension of the transposed A tile

struct RgRegs {
    float a[2][4];
    float4 w[2];
};

__device__ __forceinline__ void rg_load(const Tile& t, const BufTable& bt, int c, int k0, int row0, int64_t B,
                                        int64_t Bp, int x_f64, int tid, RgRegs& r) {
    const Chunk& ch = t.chunks[c];
    const int ak = (tid & 3) * 4;
    const int K = ch.K;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int64_t row = row0 + (tid >> 2) + 64 * h;
        float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
        if (row < B) {
            const int k = k0 + ak;
            if (ch.a_kind == A_SLAB) {
                const float* p = (const float*)bt.p[ch.a_buf] + ((int64_t)ch.a_slot * Bp + row) * H + k;
                const float4 q = *reinterpret_cast<const float4*>(p);
                v0 = q.x; v1 = q.y; v2 = q.z; v3 = q.w;
            } else {
                const int64_t idx = row * (int64_t)ch.lda + ch.a_off + k;
                const void* xb = bt.p[ch.a_buf];
                const float* pf = (const float*)xb + idx;
                if (x_f64 == 0 && k + 3 < K && ((reinterpret_cast<uintptr_t>(pf) & 15) == 0)) {
                    const float4 q = __ldg(reinterpret_cast<const float4*>(pf));
                    v0 = q.x; v1 = q.y; v2 = q.z; v3 = q.w;
                } else {
                    if (k + 0 < K) v0 = ld_x(xb, x_f64, idx + 0);
                    if (k + 1 < K) v1 = ld_x(xb, x_f64, idx + 1);
                    if (k + 2 < K) v2 = ld_x(xb, x_f64, idx + 2);
                    if (k + 3 < K) v3 = ld_x(xb, x_f64, idx + 3);
                }
                if (ch.sign_off >= 0) {
                    const float* s = (const float*)bt.p[2] + ch.sign_off + k;
                    if (k + 0 < K) v0 *= __ldg(s + 0);
                    if (k + 1 < K) v1 *= __ldg(s + 1);
                    if (k + 2 < K) v2 *= __ldg(s + 2);
                    if (k + 3 < K) v3 *= __ldg(s + 3);
                }
            }
        }
        r.a[h][0] = v0; r.a[h][1] = v1; r.a[h][2] = v2; r.a[h][3] = v3;
    }
    const float* W = (const float*)bt.p[ch.w_buf] + ch.w_off;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int k = k0 + (tid >> 5) + 8 * h;
        r.w[h] = (k < K) ? __ldg(reinterpret_cast<const float4*>(W + (int64_t)k * H + (tid & 31) * 4))
                         : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

__global__ void __launch_bounds__(256, 2)
k_rowgemm(const Tile* __restrict__ tiles, const BufTable bt, const int64_t B, const int64_t Bp, const int x_f64) {
    __shared__ Tile t;
    __shared__ __align__(16) float As[RG_BK][RG_AS];
    __shared__ __align__(16) float Ws[RG_BK][H];

    const int tid = threadIdx.x;
    {
        const int* src = reinterpret_cast<const int*>(tiles + blockIdx.y);
        int* dst = reinterpret_cast<int*>(&t);
        for (int i = tid; i < (int)(sizeof(Tile) / 4); i += 256) dst[i] = src[i];
    }
    __syncthreads();

    const int row0 = blockIdx.x * TILE_M;
    const int tx = tid & 15, ty = tid >> 4;
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    int c = 0, k0 = 0;
    RgRegs r;
    const int nch = t.n_chunks;
    if (nch > 0) rg_load(t, bt, 0, 0, row0, B, Bp, x_f64, tid, r);
    bool more = nch > 0;
    while (more) {
        // registers -> shared (A transposed to [k][row])
        {
            const int ak = (tid & 3) * 4;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int rr = (tid >> 2) + 64 * h;
#pragma unroll
                for (int i = 0; i < 4; ++i) As[ak + i][rr] = r.a[h][i];
                *reinterpret_cast<float4*>(&Ws[(tid >> 5) + 8 * h][(tid & 31) * 4]) = r.w[h];
            }
        }
        __syncthreads();
        // advance + prefetch
        k0 += RG_BK;
        if (k0 >= t.chunks[c].K) { ++c; k0 = 0; }
        more = c < nch;
        if (more) rg_load(t, bt, c, k0, row0, B, Bp, x_f64, tid, r);
#pragma unroll
        for (int k = 0; k < RG_BK; ++k) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4*>(&As[k][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Ws[k][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4*>(&Ws[k][64 + tx * 4]);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }

    // ---------------- epilogue ----------------
    float bias[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) bias[j] = 0.f;
    if (t.bias_buf >= 0) {
        const float* bp = (const float*)bt.p[t.bias_buf] + t.bias_off;
        const float4 q0 = __ldg(reinterpret_cast<const float4*>(bp + tx * 4));
        const float4 q1 = __ldg(reinterpret_cast<const float4*>(bp + 64 + tx * 4));
        bias[0] = q0.x; bias[1] = q0.y; bias[2] = q0.z; bias[3] = q0.w;
        bias[4] = q1.x; bias[5] = q1.y; bias[6] = q1.z; bias[7] = q1.w;
    }
    const int lane_shift = (tx & 7) * 4;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int64_t row = row0 + ty * 4 + (i & 3) + (i >> 2) * 64;
        const bool live = row < B;           // warp-uniform per 16-lane half? no: per ty -> handle shuffles outside guards
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            const int col = tx * 4 + 64 * hh;
            float v[4];
            unsigned nib = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float x = acc[i][hh * 4 + j] + bias[hh * 4 + j];
                if (x > 0.f) nib |= 1u << j;
                if (t.relu) x = fmaxf(x, 0.f);
                v[j] = x;
            }
            if (t.mask_out_buf >= 0) {
                unsigned word = nib << lane_shift;
                word |= __shfl_xor_sync(0xffffffffu, word, 1);
                word |= __shfl_xor_sync(0xffffffffu, word, 2);
                word |= __shfl_xor_sync(0xffffffffu, word, 4);
                if (live && (tx & 7) == 0) {
                    unsigned* mp = (unsigned*)bt.p[t.mask_out_buf] + ((int64_t)t.mask_out_slot * Bp + row) * 4 + hh * 2 + (tx >> 3);
                    *mp = word;
                }
            }
            if (!live) continue;
            if (t.posmask_buf >= 0) {
                const unsigned w = *((const unsigned*)bt.p[t.posmask_buf] +
                                     ((int64_t)t.posmask_slot * Bp + row) * 4 + hh * 2 + (tx >> 3));
                const unsigned nb = (w >> lane_shift) & 0xFu;
#pragma unroll
                for (int j = 0; j < 4; ++j) v[j] = ((nb >> j) & 1u) ? v[j] : 0.f;
            }
            if (t.res_buf >= 0) {
                const float4 q = *reinterpret_cast<const float4*>(
                    (const float*)bt.p[t.res_buf] + ((int64_t)t.res_slot * Bp + row) * H + col);
                v[0] += q.x; v[1] += q.y; v[2] += q.z; v[3] += q.w;
            }
            if (t.out_buf >= 0) {
                const int64_t off = ((int64_t)t.out_slot * Bp + row) * H + col;
                *reinterpret_cast<float4*>((float*)bt.p[t.out_buf] + off) = make_float4(v[0], v[1], v[2], v[3]);
            }
            if (t.out2_buf >= 0) {
                if (t.out2_mask_kind == MK_BITS) {
                    const unsigned w = *((const unsigned*)bt.p[t.out2_mask_buf] +
                                         ((int64_t)t.out2_mask_slot * Bp + row) * 4 + hh * 2 + (tx >> 3));
                    const unsigned nb = (w >> lane_shift) & 0xFu;
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[j] = ((nb >> j) & 1u) ? v[j] : 0.f;
                }
                const int64_t off2 = ((int64_t)t.out2_slot * Bp + row) * H + col;
                *reinterpret_cast<float4*>((float*)bt.p[t.out2_buf] + off2) = make_float4(v[0], v[1], v[2], v[3]);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// reduce-over-rows GEMM (weight gradients)
// ------------------------------------------------------------------------------------------
struct RdRegs {
    float4 d[2];
    float4 a[2];
};

__device__ __forceinline__ void rd_load(const RPair& p, const RTask& t, const BufTable& bt, int64_t r0, int64_t r_end,
                                        int64_t Bp, int x_f64, int tid, RdRegs& r) {
    const int col = (tid & 31) * 4;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int64_t row = r0 + (tid >> 5) + 8 * h;
        float4 d = make_float4(0.f, 0.f, 0.f, 0.f), a = d;
        if (row < r_end) {
            d = *reinterpret_cast<const float4*>((const float*)bt.p[p.d_buf] + ((int64_t)p.d_slot * Bp + row) * H + col);
            if (p.a_kind == A_SLAB) {
                a = *reinterpret_cast<const float4*>((const float*)bt.p[p.a_buf] + ((int64_t)p.a_slot * Bp + row) * H + col);
            } else {
                const int k = t.k0 + col;
                const int64_t idx = row * (int64_t)p.lda + p.a_off + k;
                const void* xb = bt.p[p.a_buf];
                const float* pf = (const float*)xb + idx;
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                if (x_f64 == 0 && k + 3 < t.K && ((reinterpret_cast<uintptr_t>(pf) & 15) == 0)) {
                    const float4 q = __ldg(reinterpret_cast<const float4*>(pf));
                    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (k + j < t.K) v[j] = ld_x(xb, x_f64, idx + j);
                }
                if (p.sign_off >= 0) {
                    const float* s = (const float*)bt.p[2] + p.sign_off + k;
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (k + j < t.K) v[j] *= __ldg(s + j);
                }
                a = make_float4(v[0], v[1], v[2], v[3]);
            }
        }
        r.d[h] = d; r.a[h] = a;
    }
}

__global__ void __launch_bounds__(256, 2)
k_reducegemm(const RTask* __restrict__ tasks, const RPair* __restrict__ pairs, const int task0, const BufTable bt,
             const int64_t B, const int64_t Bp, const int x_f64, const int n_splits,
             float* __restrict__ part_w, float* __restrict__ part_b) {
    __shared__ __align__(16) float Ds[RG_BK][H];
    __shared__ __align__(16) float As[RG_BK][H];
    __shared__ RTask t;
    const int tid = threadIdx.x;
    const int task = task0 + blockIdx.x;
    if (tid < (int)(sizeof(RTask) / 4)) reinterpret_cast<int*>(&t)[tid] = reinterpret_cast<const int*>(tasks + task)[tid];
    __syncthreads();

    const int split = blockIdx.y;
    const int64_t rows_per = round_up((B + n_splits - 1) / n_splits, RG_BK);
    const int64_t r_begin = split * rows_per;
    const int64_t r_end = (r_begin + rows_per < B) ? (r_begin + rows_per) : B;
    const int64_t n_steps_pair = (r_end > r_begin) ? (r_end - r_begin + RG_BK - 1) / RG_BK : 0;

    const int tx = tid & 15, ty = tid >> 4;
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    float cs = 0.f;

    // Summation accuracy: a task holds at most RD_MAX_PAIRS pairs and a split at most 512 rows, so no fp32
    // running sum is longer than 2048 terms; the splits are then summed in double (k_reduce_partials).
    float* pw = part_w + ((int64_t)task * n_splits + split) * (H * H);
    const int64_t total = n_steps_pair * t.n_pairs;
    RdRegs r;
    int64_t step = 0;
    if (total > 0) rd_load(pairs[t.pair_begin], t, bt, r_begin, r_end, Bp, x_f64, tid, r);
    while (step < total) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            *reinterpret_cast<float4*>(&Ds[(tid >> 5) + 8 * h][(tid & 31) * 4]) = r.d[h];
            *reinterpret_cast<float4*>(&As[(tid >> 5) + 8 * h][(tid & 31) * 4]) = r.a[h];
        }
        __syncthreads();
        ++step;
        if (step < total) {
            const int pi = (int)(step / n_steps_pair);
            const int64_t r0 = r_begin + (step % n_steps_pair) * RG_BK;
            rd_load(pairs[t.pair_begin + pi], t, bt, r0, r_end, Bp, x_f64, tid, r);
        }
#pragma unroll
        for (int k = 0; k < RG_BK; ++k) {
            const float4 d0 = *reinterpret_cast<const float4*>(&Ds[k][ty * 4]);
            const float4 d1 = *reinterpret_cast<const float4*>(&Ds[k][64 + ty * 4]);
            const float4 a0 = *reinterpret_cast<const float4*>(&As[k][tx * 4]);
            const float4 a1 = *reinterpret_cast<const float4*>(&As[k][64 + tx * 4]);
            const float d[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(d[i], a[j], acc[i][j]);
        }
        if (t.want_colsum && tid < H) {
#pragma unroll
            for (int k = 0; k < RG_BK; ++k) cs += Ds[k][tid];
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int o = ty * 4 + (i & 3) + (i >> 2) * 64;
        *reinterpret_cast<float4*>(pw + o * H + tx * 4) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        *reinterpret_cast<float4*>(pw + o * H + 64 + tx * 4) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
    }
    if (t.want_colsum && tid < H) part_b[((int64_t)task * n_splits + split) * H + tid] = cs;
}

// sum the split partials of a group of tasks into the flat gradient buffer (fixed order => deterministic).  blockIdx.z = model of a
// model batch: its partials start part_slots slots further, its gradients n_params elements further.
__global__ void __launch_bounds__(256)
k_reduce_partials(const OutGroup* __restrict__ groups, const float* __restrict__ part_w,
                  const float* __restrict__ part_b, const __grid_constant__ PartSegs segs,
                  float* __restrict__ grads, const float rscale, const int64_t part_slots, const int64_t n_params) {
    const OutGroup g = groups[blockIdx.x];
    part_w += blockIdx.z * part_slots * (H * H);
    part_b += blockIdx.z * part_slots * H;
    grads += blockIdx.z * n_params;
    if (g.kind == 0) {
        const int per = (H * H) / gridDim.y;
        for (int e = blockIdx.y * per + threadIdx.x; e < (blockIdx.y + 1) * per; e += 256) {
            const int o = e / H, i = e % H;
            if (g.k0 + i >= g.K) continue;
            double sd = 0.0;
            for (int ti = 0; ti < g.n_tasks; ++ti) {
                int64_t slot0; int n_splits;
                part_lookup(segs, g.tasks[ti], slot0, n_splits);
                const float* p = part_w + slot0 * (H * H) + e;
                int sp = 0;
                for (; sp + 16 <= n_splits; sp += 16) {    // 16 independent loads in flight, summed in the fixed order
                    float v[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = __ldg(p + (int64_t)(sp + j) * (H * H));
#pragma unroll
                    for (int j = 0; j < 16; ++j) sd += (double)v[j];
                }
                for (; sp + 8 <= n_splits; sp += 8) {
                    float v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = __ldg(p + (int64_t)(sp + j) * (H * H));
#pragma unroll
                    for (int j = 0; j < 8; ++j) sd += (double)v[j];
                }
                for (; sp < n_splits; ++sp) sd += (double)__ldg(p + (int64_t)sp * (H * H));
            }
            const float s = (float)(sd * (double)g.scale * (double)rscale);
            for (int oi = 0; oi < g.n_outs; ++oi) grads[(int64_t)g.outs[oi] + (int64_t)o * g.K + g.k0 + i] = s;
        }
    } else {
        if (blockIdx.y != 0) return;
        for (int e = threadIdx.x; e < H; e += 256) {
            double sd = 0.0;
            for (int ti = 0; ti < g.n_tasks; ++ti) {
                int64_t slot0; int n_splits;
                part_lookup(segs, g.tasks[ti], slot0, n_splits);
                const float* p = part_b + slot0 * H + e;
                for (int sp = 0; sp < n_splits; ++sp) sd += (double)p[(int64_t)sp * H];
            }
            const float s = (float)(sd * (double)g.scale * (double)rscale);
            for (int oi = 0; oi < g.n_outs; ++oi) grads[(int64_t)g.outs[oi] + e] = s;
        }
    }
}

// ------------------------------------------------------------------------------------------
// derived weights: transposes, per-destination root sums and bias sums
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_derive(const DeriveOp* __restrict__ ops, const float* __restrict__ params, float* __restrict__ derived) {
    const DeriveOp op = ops[blockIdx.y];
    const int n = op.rows * op.cols;
    for (int e = blockIdx.x * 256 + threadIdx.x; e < n; e += gridDim.x * 256) {
        // e indexes the destination
        int r, c;
        if (op.transpose) { c = e / op.rows; r = e % op.rows; } else { r = e / op.cols; c = e % op.cols; }
        float s = 0.f;
        for (int i = 0; i < op.n_src; ++i) s += params[(int64_t)op.src_off[i] + (int64_t)r * op.cols + c];
        derived[(int64_t)op.dst_off + e] = s;
    }
}

// ------------------------------------------------------------------------------------------
// decoder: out[g*n_dec + j, c] = (h[slot_j][g] . Wdec[c] + b[c]) * sign[j*C + c]
// ------------------------------------------------------------------------------------------
// 4 consecutive weights: one 16-byte load where aligned.  Row m of a model batch's [M, n_params] buffer starts 4 m n_params bytes in,
// which is 16-byte aligned only when n_params is a multiple of 4.
__device__ __forceinline__ float4 ld_w4(const float* p) {
    if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) return __ldg(reinterpret_cast<const float4*>(p));
    return make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
}

// CMAX: compile-time bound of the decoder width (2 / 4 / 8): the weight rows are register arrays, and sized for 8 channels they cost the
// 2-channel contact head 48 registers it never uses
template <int CMAX>
__global__ void __launch_bounds__(256)
k_decoder_fwd(const DecoderDesc dd, const float* __restrict__ hslab, const __half* __restrict__ h_hi, const __half* __restrict__ h_lo,
              const float* __restrict__ params, const float* __restrict__ signs, float* __restrict__ out, const int64_t B, const int64_t Bp,
              const int64_t Bm, const int64_t n_params) {
    // blockIdx.y = model of a model batch: its parameters, its row block [y Bm, y Bm + B) of the slabs, its output rows
    params += blockIdx.y * n_params;
    out += blockIdx.y * B * dd.n_dec * dd.C;
    if (hslab) hslab += blockIdx.y * Bm * H;
    if (h_hi) { h_hi += blockIdx.y * Bm * H; h_lo += blockIdx.y * Bm * H; }
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int64_t n_rows = B * dd.n_dec;
    const int64_t stride = (int64_t)gridDim.x * 8;
    float4 w[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
        w[c] = (c < dd.C) ? ld_w4(params + dd.w_off + c * H + lane * 4)
                          : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 2
    for (int64_t row = warp; row < n_rows; row += stride) {
        const int64_t g = row / dd.n_dec;
        const int j = (int)(row % dd.n_dec);
        const float4 h = load_h4(hslab, h_hi, h_lo, ((int64_t)dd.slots[j] * Bp + g) * H + lane * 4);
#pragma unroll
        for (int c = 0; c < CMAX; ++c) {
            if (c >= dd.C) break;
            float s = h.x * w[c].x + h.y * w[c].y + h.z * w[c].z + h.w * w[c].w;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) {
                float v = s + __ldg(params + dd.b_off + c);
                if (dd.sign_off >= 0) v *= __ldg(signs + dd.sign_off + j * dd.C + c);
                out[row * dd.C + c] = v;
            }
        }
    }
}

// backward: dH[slot_j][g][:] = sum_c dout'[c] Wdec[c][:]   (written to dh_buf, masked copy to dc_buf)
//           partial dWdec / db per block -> part[(block*(C*H + C))]
template <int CMAX>
__global__ void __launch_bounds__(256)
k_decoder_bwd(const DecoderDesc dd, const float* __restrict__ hslab, const __half* __restrict__ h_hi, const __half* __restrict__ h_lo,
              const float* __restrict__ params,
              const float* __restrict__ signs, const float* __restrict__ dout,
              float* __restrict__ dh, float* __restrict__ dc, const int mask_kind, const void* __restrict__ mask_buf,
              float* __restrict__ part, const int64_t B, const int64_t Bp, const float gscale,
              __half* __restrict__ dh_hi, __half* __restrict__ dh_lo, __half* __restrict__ dc_hi, __half* __restrict__ dc_lo,
              const int64_t Bm, const int64_t n_params) {
    __shared__ float red[8][CMAX][H + 1];
    __shared__ float redb[8][CMAX];
    // blockIdx.y = model of a model batch (see k_decoder_fwd); its partials are the next gridDim.x blocks
    {
        const int64_t r0 = blockIdx.y * Bm * H;      // the model's first row of every slab / image
        params += blockIdx.y * n_params;
        dout += blockIdx.y * B * dd.n_dec * dd.C;
        part += (int64_t)blockIdx.y * gridDim.x * (DEC_MAXC * H + DEC_MAXC);
        if (hslab) hslab += r0;
        if (h_hi) { h_hi += r0; h_lo += r0; }
        if (dh) dh += r0;
        if (dc) dc += r0;
        if (dh_hi) { dh_hi += r0; dh_lo += r0; }
        if (dc_hi) { dc_hi += r0; dc_lo += r0; }
        if (mask_buf) mask_buf = (const unsigned*)mask_buf + blockIdx.y * Bm * 4;
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t warp = (int64_t)blockIdx.x * 8 + wid;
    const int64_t n_rows = B * dd.n_dec;
    const int64_t stride = (int64_t)gridDim.x * 8;
    float4 w[CMAX], gw[CMAX];
    float gb[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
        w[c] = (c < dd.C) ? ld_w4(params + dd.w_off + c * H + lane * 4)
                          : make_float4(0.f, 0.f, 0.f, 0.f);
        gw[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        gb[c] = 0.f;
    }
#pragma unroll 2
    for (int64_t row = warp; row < n_rows; row += stride) {
        const int64_t g = row / dd.n_dec;
        const int j = (int)(row % dd.n_dec);
        const int64_t off = ((int64_t)dd.slots[j] * Bp + g) * H + lane * 4;
        const float4 h = load_h4(hslab, h_hi, h_lo, off);
        float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int c = 0; c < CMAX; ++c) {
            if (c >= dd.C) break;
            float dv = __ldg(dout + row * dd.C + c) * gscale;
            if (dd.sign_off >= 0) dv *= __ldg(signs + dd.sign_off + j * dd.C + c);
            d.x = fmaf(dv, w[c].x, d.x); d.y = fmaf(dv, w[c].y, d.y);
            d.z = fmaf(dv, w[c].z, d.z); d.w = fmaf(dv, w[c].w, d.w);
            gw[c].x = fmaf(dv, h.x, gw[c].x); gw[c].y = fmaf(dv, h.y, gw[c].y);
            gw[c].z = fmaf(dv, h.z, gw[c].z); gw[c].w = fmaf(dv, h.w, gw[c].w);
            gb[c] += dv;
        }
        if (dh) *reinterpret_cast<float4*>(dh + off) = d;
        if (dh_hi) { const float vv[4] = {d.x, d.y, d.z, d.w}; split_store4(dh_hi, dh_lo, off, vv); }
        if (dc || dc_hi) {
            if (mask_kind == MK_BITS) {
                const unsigned wd = *((const unsigned*)mask_buf + ((int64_t)dd.slots[j] * Bp + g) * 4 + (lane >> 3));
                const unsigned nb = (wd >> ((lane & 7) * 4)) & 0xFu;
                d.x = (nb & 1u) ? d.x : 0.f; d.y = (nb & 2u) ? d.y : 0.f;
                d.z = (nb & 4u) ? d.z : 0.f; d.w = (nb & 8u) ? d.w : 0.f;
            }
            if (dc) *reinterpret_cast<float4*>(dc + off) = d;
            if (dc_hi) { const float vv[4] = {d.x, d.y, d.z, d.w}; split_store4(dc_hi, dc_lo, off, vv); }
        }
    }
    if (dh_hi || dc_hi) {   // rows [B, Bm) of the model's block of the decoded slots' fp16 images stay zero
        const int64_t pad = Bm - B;
        const float z[4] = {0.f, 0.f, 0.f, 0.f};
        for (int64_t r = warp; r < pad * dd.n_dec; r += stride) {
            const int64_t off = ((int64_t)dd.slots[r / pad] * Bp + B + r % pad) * H + lane * 4;
            if (dh_hi) split_store4(dh_hi, dh_lo, off, z);
            if (dc_hi) split_store4(dc_hi, dc_lo, off, z);
        }
    }
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
        if (c >= dd.C) break;                  // only the decoder's C channels carry anything
        red[wid][c][lane * 4 + 0] = gw[c].x; red[wid][c][lane * 4 + 1] = gw[c].y;
        red[wid][c][lane * 4 + 2] = gw[c].z; red[wid][c][lane * 4 + 3] = gw[c].w;
        if (lane == 0) redb[wid][c] = gb[c];   // every lane holds the same gb
    }
    __syncthreads();
    float* pb = part + (int64_t)blockIdx.x * (DEC_MAXC * H + DEC_MAXC);
    for (int e = threadIdx.x; e < dd.C * H; e += 256) {
        const int c = e / H, k = e % H;
        float s = 0.f;
#pragma unroll
        for (int wv = 0; wv < 8; ++wv) s += red[wv][c][k];
        pb[e] = s;
    }
    if ((int)threadIdx.x < dd.C) {
        float s = 0.f;
#pragma unroll
        for (int wv = 0; wv < 8; ++wv) s += redb[wv][threadIdx.x];
        pb[DEC_MAXC * H + threadIdx.x] = s;
    }
}

__global__ void __launch_bounds__(256)
k_decoder_bwd_reduce(const DecoderDesc dd, const float* __restrict__ part, const int n_blocks, float* __restrict__ grads,
                     const float scale, const int64_t n_params) {
    // one CTA per output element: thread t sums the partials of blocks t, t + 256, ... (fixed order), then a fixed tree;
    // blockIdx.y = model of a model batch
    __shared__ float sh[256];
    part += (int64_t)blockIdx.y * n_blocks * (DEC_MAXC * H + DEC_MAXC);
    grads += blockIdx.y * n_params;
    const int e = blockIdx.x;
    const int src = (e < dd.C * H) ? e : (DEC_MAXC * H + (e - dd.C * H));
    float s = 0.f;
    for (int b = threadIdx.x; b < n_blocks; b += 256) s += __ldg(part + (int64_t)b * (DEC_MAXC * H + DEC_MAXC) + src);
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const float r = sh[0] * scale;
        if (e < dd.C * H) grads[dd.w_off + e] = r; else grads[dd.b_off + (e - dd.C * H)] = r;
    }
}

// ------------------------------------------------------------------------------------------
// input gradient of the encoder (MSHGNN_MODE_FP32, mshgnn_input_grad):
//   dx[t][g * nodes + n, k] = sign[slot][k] * sum_c dpre0[slot][g][c] * W_enc[t][c, k]        (hgnn_k4.py:L159-160, L198-237)
// one CTA = 16 graphs x 64 columns of one node slot (blockIdx.y = DxUnit); dead slots write exact zeros and read nothing
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_encoder_dx(const DxUnit* __restrict__ units, const DxOut out, const float* __restrict__ dpre, const float* __restrict__ params,
             const float* __restrict__ signs, const int64_t B, const int64_t Bp) {
    __shared__ float D[16][H + 1];
    __shared__ float W[H][64];
    const DxUnit u = units[blockIdx.y];
    float* dx = out.p[u.type];
    const int64_t g0 = (int64_t)blockIdx.x * 16;
    const int k0 = blockIdx.z * 64, K = u.K;
    if (!dx || k0 >= K || g0 >= B) return;
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    if (u.live) {
        const float* dp = dpre + ((int64_t)u.slot * Bp + g0) * H;      // rows up to Bp exist
        for (int e = tid; e < 16 * H; e += 256) D[e / H][e % H] = dp[e];
        const float* w = params + out.w_off[u.type];
        for (int e = tid; e < H * 64; e += 256) {
            const int c = e / 64, kk = e % 64;
            W[c][kk] = k0 + kk < K ? w[(int64_t)c * K + k0 + kk] : 0.f;
        }
        __syncthreads();
#pragma unroll 4
        for (int c = 0; c < H; ++c) {
            const float d = D[ty][c];
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i] = fmaf(d, W[c][tx + 16 * i], acc[i]);
        }
    }
    const int64_t g = g0 + ty;
    if (g >= B) return;
    float* row = dx + (g * out.nodes[u.type] + u.node) * K;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int k = k0 + tx + 16 * i;
        if (k < K) row[k] = u.live ? (u.sign_off >= 0 ? acc[i] * signs[u.sign_off + k] : acc[i]) : 0.f;
    }
}

// ------------------------------------------------------------------------------------------
// loss heads
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double ld_label(const void* p, int dtype, int64_t i) {
    if (dtype == 1) return ((const double*)p)[i];
    if (dtype == 2) return (double)((const long long*)p)[i];
    return (double)((const float*)p)[i];
}

__device__ __forceinline__ double block_sum(double v, double* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) sh[wid] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += sh[i];
    return s;   // valid in thread 0
}

// MSE: n elements; CE2: n rows of 2 logits.  partial[blockIdx.x] = block sum (double).  blockIdx.y = model of a model batch:
// its n elements / rows follow those of the models before it, its partials start LOSS_PARTIALS further.
__global__ void __launch_bounds__(256)
k_loss_partial(const int kind, const float* __restrict__ out, const void* __restrict__ labels, const int label_dtype,
               const int64_t n, const float dscale, float* __restrict__ dout, double* __restrict__ partial) {
    __shared__ double sh[8];
    double acc = 0.0;
    {
        const int64_t first = blockIdx.y * n;       // the model's first element (MSE) / row (CE2)
        partial += blockIdx.y * LOSS_PARTIALS;
        out += kind == 0 ? first : 2 * first;
        if (dout) dout += kind == 0 ? first : 2 * first;
        labels = (const char*)labels + first * (label_dtype == 0 ? 4 : 8);
    }
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        if (kind == 0) {
            const float d = out[i] - (float)ld_label(labels, label_dtype, i);
            acc += (double)d * (double)d;
            if (dout) dout[i] = 2.f * d * dscale;
        } else {
            const float a = out[2 * i], b = out[2 * i + 1];
            const int y = ld_label(labels, label_dtype, i) != 0.0;
            const float m = fmaxf(a, b);
            const float ea = expf(a - m), eb = expf(b - m);
            const float lse = m + logf(ea + eb);
            acc += (double)(lse - (y ? b : a));
            if (dout) {
                const float inv = 1.f / (ea + eb);
                dout[2 * i] = (ea * inv - (y ? 0.f : 1.f)) * dscale;
                dout[2 * i + 1] = (eb * inv - (y ? 1.f : 0.f)) * dscale;
            }
        }
    }
    const double s = block_sum(acc, sh);
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

__global__ void k_loss_final(const double* __restrict__ partial, const int n_blocks, const double inv_n,
                             const int round_f32, float* __restrict__ loss_out) {
    // one warp: lane l sums the partials l, l + 32, ... (fixed order), then a fixed shuffle tree; blockIdx.x = model
    partial += blockIdx.x * LOSS_PARTIALS;
    loss_out += blockIdx.x;
    double s = 0.0;
    for (int i = threadIdx.x; i < n_blocks; i += 32) s += partial[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    // customMetrics.py:L25: summed_loss.float() / total_num
    if (threadIdx.x == 0) loss_out[0] = round_f32 ? (float)((double)(float)s * inv_n) : (float)(s * inv_n);
}

// ------------------------------------------------------------------------------------------
// optimizers on the flat buffers
// ------------------------------------------------------------------------------------------
// One element of the Adam / SGD updates.  k_adam / k_sgd and their per-model forms call the same function, so the compiler
// contracts the same products into FMAs and model m of a per-model launch gets the bits of a launch on its range alone.
__device__ __forceinline__ void adam_update(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                            const int64_t i, const float lr, const float b1, const float b2, const float eps, const float wd,
                                            const float bc1, const float bc2s) {
    float gi = g[i];
    const float pi = p[i];
    if (wd != 0.f) gi = fmaf(wd, pi, gi);
    const float mi = m[i] + (1.f - b1) * (gi - m[i]);      // torch: exp_avg.lerp_(grad, 1-beta1)
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2s + eps;
    p[i] = pi - (lr / bc1) * (mi / denom);
}

__device__ __forceinline__ void sgd_update(float* __restrict__ p, const float* __restrict__ g, const int64_t i, const float lr) { p[i] -= lr * g[i]; }

__global__ void __launch_bounds__(256)
k_adam(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, const int64_t n,
       const float lr, const float b1, const float b2, const float eps, const float wd, const float bc1, const float bc2s) {
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256)
        adam_update(p, g, m, v, i, lr, b1, b2, eps, wd, bc1, bc2s);
}

__global__ void __launch_bounds__(256)
k_sgd(float* __restrict__ p, const float* __restrict__ g, const int64_t n, const float lr) {
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) sgd_update(p, g, i, lr);
}

// Per-model optimizer table of mshgnn_adam_step_models / mshgnn_sgd_step_models, passed by value: a launch captured in a CUDA
// graph keeps the values it was captured with, like the scalars of k_adam, and no host-to-device copy is needed.
constexpr int OPT_MAX_MODELS = 1023;
struct OptModels {
    int64_t off[OPT_MAX_MODELS + 1];   // model m owns elements [off[m], off[m + 1]) of every buffer
    float lr[OPT_MAX_MODELS];
    float bc1[OPT_MAX_MODELS];         // Adam bias corrections of the model's step (host-computed as mshgnn_adam_step does)
    float bc2s[OPT_MAX_MODELS];
    uint8_t active[OPT_MAX_MODELS];    // 0: the model's elements are not touched
};
static_assert(sizeof(OptModels) + 64 <= 32764, "the per-model optimizer table must fit the kernel-parameter limit");

// grid.y = model; grid.x strides over that model's range
__global__ void __launch_bounds__(256)
k_adam_models(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, const __grid_constant__ OptModels t,
              const float b1, const float b2, const float eps, const float wd) {
    const int mo = blockIdx.y;
    if (!t.active[mo]) return;
    const float lr = t.lr[mo], bc1 = t.bc1[mo], bc2s = t.bc2s[mo];
    const int64_t end = t.off[mo + 1];
    for (int64_t i = t.off[mo] + (int64_t)blockIdx.x * 256 + threadIdx.x; i < end; i += (int64_t)gridDim.x * 256)
        adam_update(p, g, m, v, i, lr, b1, b2, eps, wd, bc1, bc2s);
}

__global__ void __launch_bounds__(256)
k_sgd_models(float* __restrict__ p, const float* __restrict__ g, const __grid_constant__ OptModels t) {
    const int mo = blockIdx.y;
    if (!t.active[mo]) return;
    const float lr = t.lr[mo];
    const int64_t end = t.off[mo + 1];
    for (int64_t i = t.off[mo] + (int64_t)blockIdx.x * 256 + threadIdx.x; i < end; i += (int64_t)gridDim.x * 256) sgd_update(p, g, i, lr);
}

// ------------------------------------------------------------------------------------------
// edge_index validation (SURVEY 3.4 batching layout; modules.py "validate_edges")
// ------------------------------------------------------------------------------------------
//  The kernels never read edge_index: the morphology template is compiled into the plan.  What has to hold is that the
//  caller's edge_index_dict IS that template tiled over the batch, bit-exactly (PyG Batch.from_data_list: graph g's edges
//  are the template's plus g * nodes_per_graph).  One launch checks every edge type; a mismatch raises `flag` (pinned host
//  memory or device memory), which the host reads without synchronising.
struct EdgeCheck {
    int n_etypes;
    int E[MSHGNN_MAX_EDGE_TYPES];              // edges per graph
    int n_src[MSHGNN_MAX_EDGE_TYPES], n_dst[MSHGNN_MAX_EDGE_TYPES];
    int tpl_off[MSHGNN_MAX_EDGE_TYPES];        // offset of [src E | dst E] in the template table
    const long long* ei[MSHGNN_MAX_EDGE_TYPES];   // [2][E * B] int64, row-major
};
__global__ void __launch_bounds__(256)
k_check_edges(const EdgeCheck ec, const int* __restrict__ tpl, const long long B, int* __restrict__ flag) {
    const int e = blockIdx.y;
    const int E = ec.E[e];
    const long long n = (long long)E * B;
    const long long* src = ec.ei[e];
    const long long* dst = src + n;
    const int* ts = tpl + ec.tpl_off[e];
    const int* td = ts + E;
    bool bad = false;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
        const long long g = i / E;
        const int j = (int)(i - g * E);
        bad |= __ldg(src + i) != (long long)ts[j] + g * ec.n_src[e];
        bad |= __ldg(dst + i) != (long long)td[j] + g * ec.n_dst[e];
    }
    if (bad) *reinterpret_cast<volatile int*>(flag) = 1 + e;
}

}  // namespace mshgnn
