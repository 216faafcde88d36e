// Input gradient of the encoder on tcgen05 (mshgnn_input_grad, tensor-core modes):
//
//   dx[t][g * nodes + n, k] = sign[slot][k] * sum_c dpre0[slot][g][c] * W_enc[t][c, k]        (slot = slot of node n of type t)
//
//  the transpose of the encoder forward (hgnn_k4.py:L159-160, L198-237).  dpre0 (the gradient at the encoder pre-activation, scaled
//  by the backward's power-of-two G) is in the workspace as (hi, lo) fp16 images when the backward ends; the encoder weight image
//  [n_types*128][kmax] (x 2^8) that the forward prologue wrote is still there (a region of its own in ws_layout).  No row is permuted:
//  every feature row feeds exactly one node slot.
//  One CTA = one (node slot, row tile of 128 graphs); it walks the 64-column blocks of the slot's in-width:
//    * warp 0: TMA of the slot's dpre0 tile (hi, lo: K-major, 128 channels = two 64-channel SWIZZLE_128B boxes, loaded once and used
//      by every column block) and of the weight blocks (MN-major: box 64 columns x 64 channels, two per block, 2-stage ring);
//    * warp 1: TMEM owner + MMA issuer: D[128 graphs, 64 columns] += A[128 x 128] B[128 x 64], 3 MMAs per K step in MODE_TC
//      (hi*hi + lo*hi + hi*lo), 1 in MODE_TC_1X; two 64-column fp32 accumulators, so block j + 1 is multiplied while j is drained;
//    * warps 2..5 (one thread per graph row): tcgen05.ld, x sign x 1/(G 2^8) (powers of two: exact), into a 128B-swizzled fp32
//      staging tile (two 32-column halves, two tiles in rotation), then one TMA store per half through a 3-D tensor map over the
//      caller's dx[t] (dims K, nodes, B; box 32 x 1 x 128): columns >= K and graphs >= B are clipped by the hardware.  Widths whose
//      rows are not a multiple of 16 bytes cannot have a tensor map; there the 128 threads copy the staged tile out with coalesced
//      plain stores.
//  A dead slot (need[0][slot] == 0) has no dpre0: its rows are written as exact zeros and nothing is read.
#pragma once
#include "kernels_tc.cuh"

namespace mshgnn {

constexpr int DX_THREADS = 192;
constexpr int DX_A_BYTES = 2 * ENC_TILE_BYTES;               // 128 graphs x 128 channels fp16 (two 64-channel boxes)
constexpr int DX_W_BYTES = ENC_TILE_BYTES;                   // 128 channels x 64 columns fp16 (two 64 x 64 boxes)
constexpr int DX_STG_BYTES = 2 * ENC_TILE_BYTES;             // 128 graphs x 64 fp32 (two 32-column halves)
constexpr int DX_OFF_W = 2 * DX_A_BYTES;                     // after A hi, A lo
constexpr int DX_OFF_STG = DX_OFF_W + 2 * 2 * DX_W_BYTES;    // after 2 stages x (W hi, W lo)
constexpr int DX_OFF_BAR = DX_OFF_STG + 2 * DX_STG_BYTES;
constexpr int DX_SMEM_BYTES = DX_OFF_BAR + 128;              // 192 KB + barriers; no static shared memory: the window starts 1024-aligned
constexpr uint32_t DX_TMEM_COLS = 128;                       // two 64-column accumulators
// kind::f16, fp16 x fp16 -> fp32, A K-major (dpre0 rows), B MN-major (weight image rows are the hidden channels), M = 128, N = 64
constexpr uint32_t DX_IDESC = (1u << 4) | (1u << 16) | ((64u >> 3) << 17) | ((128u >> 4) << 24);

struct alignas(64) DxMaps {
    CUtensorMap a;               // workspace images, box 64 x 128, SWIZZLE_128B
    CUtensorMap w_hi, w_lo;      // encoder weight images, box 64 columns x 64 channels, SWIZZLE_128B
    CUtensorMap x[4];            // dx[t] as (K, nodes, B) fp32, box 32 x 1 x 128, SWIZZLE_128B (DxOut::tma bit t)
};

__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
                 "r"(src), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void tma_store_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }

__global__ void __launch_bounds__(DX_THREADS, 1)
k_tc_encoder_dx(const __grid_constant__ DxMaps maps, const DxUnit* __restrict__ units, const DxOut out, const float* __restrict__ signs,
                const int dc_hi_row, const int dc_lo_row /*first workspace rows of the dpre0 images*/, const int64_t B, const int64_t Bp,
                const int split, const float scale) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const DxUnit u = units[blockIdx.y];
    float* dx = out.p[u.type];
    const int64_t row0 = (int64_t)blockIdx.x * TILE_M;
    if (!dx || row0 >= B) return;
    const int K = u.K, nodes = out.nodes[u.type];
    if (!u.live) {
        const int64_t rows = B - row0 < TILE_M ? B - row0 : TILE_M;
        for (int64_t e = tid; e < rows * K; e += DX_THREADS) {
            const int64_t r = e / K;
            dx[((row0 + r) * nodes + u.node) * K + (e - r * K)] = 0.f;
        }
        return;
    }
    const uint32_t sb = smem_u32(smem_raw);
    if (sb & 1023u) __trap();                                // the swizzled tiles need the 1024-byte alignment
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + DX_OFF_BAR);
    const uint32_t a_full = smem_u32(bars), w_full0 = smem_u32(bars + 1), w_empty0 = smem_u32(bars + 3), acc_full0 = smem_u32(bars + 5),
                   acc_free0 = smem_u32(bars + 7);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);
    if (tid == 0) {
        mbar_init(a_full, 1);
        for (int s = 0; s < 2; ++s) {
            mbar_init(w_full0 + 8 * s, 1); mbar_init(w_empty0 + 8 * s, 1);
            mbar_init(acc_full0 + 8 * s, 1); mbar_init(acc_free0 + 8 * s, 128);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(tmem_slot), DX_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int n_kb = u.n_kb;

    if (warp == 0) {
        if (lane == 0) {
            // ---------------- TMA: the dpre0 tile once, then the weight blocks through a 2-stage ring ----------------
            const int arow = (int)((int64_t)u.slot * Bp + row0);
            mbar_expect_tx(a_full, split ? 2 * DX_A_BYTES : DX_A_BYTES);
            tma_load_2d(sb, &maps.a, a_full, 0, dc_hi_row + arow);
            tma_load_2d(sb + ENC_TILE_BYTES, &maps.a, a_full, 64, dc_hi_row + arow);
            if (split) {
                tma_load_2d(sb + DX_A_BYTES, &maps.a, a_full, 0, dc_lo_row + arow);
                tma_load_2d(sb + DX_A_BYTES + ENC_TILE_BYTES, &maps.a, a_full, 64, dc_lo_row + arow);
            }
            const int wrow = u.type * H;
            for (int j = 0; j < n_kb; ++j) {
                const int s = j & 1;
                mbar_wait(w_empty0 + 8 * s, (uint32_t)((j >> 1) & 1) ^ 1u);
                const uint32_t st = sb + DX_OFF_W + (uint32_t)s * 2 * DX_W_BYTES, fb = w_full0 + 8 * s;
                mbar_expect_tx(fb, split ? 2 * DX_W_BYTES : DX_W_BYTES);
                tma_load_2d(st, &maps.w_hi, fb, j * 64, wrow);
                tma_load_2d(st + DX_W_BYTES / 2, &maps.w_hi, fb, j * 64, wrow + 64);
                if (split) {
                    tma_load_2d(st + DX_W_BYTES, &maps.w_lo, fb, j * 64, wrow);
                    tma_load_2d(st + DX_W_BYTES + DX_W_BYTES / 2, &maps.w_lo, fb, j * 64, wrow + 64);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // ---------------- MMA issuer: accumulator j & 1 for column block j ----------------
            mbar_wait(a_full, 0);
            tc_fence_after();
            for (int j = 0; j < n_kb; ++j) {
                const int s = j & 1;
                mbar_wait(acc_free0 + 8 * s, (uint32_t)((j >> 1) & 1) ^ 1u);       // the epilogue has drained block j - 2
                mbar_wait(w_full0 + 8 * s, (uint32_t)((j >> 1) & 1));
                tc_fence_after();
                const uint32_t st = sb + DX_OFF_W + (uint32_t)s * 2 * DX_W_BYTES;
                const uint64_t w_hi = smem_desc_mn_sw128(st), w_lo = smem_desc_mn_sw128(st + DX_W_BYTES);
                const uint32_t acc = tmem_base + (uint32_t)s * 64u;
#pragma unroll
                for (int ks = 0; ks < H / 16; ++ks) {
                    const uint32_t abox = sb + (uint32_t)(ks >> 2) * ENC_TILE_BYTES;
                    const uint64_t a_hi = smem_desc_sw128(abox) + (uint64_t)((ks & 3) * 2);                 // 16 channels = 32 bytes
                    const uint64_t a_lo = smem_desc_sw128(abox + DX_A_BYTES) + (uint64_t)((ks & 3) * 2);
                    const uint64_t wadv = (uint64_t)(ks * (2048 >> 4));                                     // 16 channels = two 8-row groups
                    umma_f16(acc, a_hi, w_hi + wadv, DX_IDESC, ks ? 1u : 0u);
                    if (split) {
                        umma_f16(acc, a_lo, w_hi + wadv, DX_IDESC, 1u);
                        umma_f16(acc, a_hi, w_lo + wadv, DX_IDESC, 1u);
                    }
                }
                umma_commit(w_empty0 + 8 * s);
                umma_commit(acc_full0 + 8 * s);
            }
        }
    } else {
        // ---------------- epilogue: thread = graph row r of the tile (TMEM lane quarter = warp % 4) ----------------
        const int q = warp & 3;
        const int r = q * 32 + lane;
        const bool leader = warp == 2 && lane == 0;
        const bool tma = (out.tma >> u.type) & 1;
        const float* sg = u.sign_off >= 0 ? signs + u.sign_off : nullptr;
        for (int j = 0; j < n_kb; ++j) {
            const int b = j & 1;
            mbar_wait(acc_full0 + 8 * b, (uint32_t)((j >> 1) & 1));
            tc_fence_after();
            uint32_t raw[2][32];
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)b * 64u, raw[0]);
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)b * 64u + 32u, raw[1]);
            tmem_ld_wait();
            tc_fence_before();
            mbar_arrive(acc_free0 + 8 * b);
            if (leader) tma_store_wait_read1();              // the store issued from this staging tile two blocks ago has read it
            epi_bar_sync();
            const uint32_t stg = sb + DX_OFF_STG + (uint32_t)b * DX_STG_BYTES;
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const int k = j * 64 + h * 32 + c * 4;
                    float f[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) f[i] = (sg && k + i < K) ? __ldg(sg + k + i) * scale : scale;
                    uint4 v;
                    v.x = __float_as_uint(__uint_as_float(raw[h][4 * c]) * f[0]);
                    v.y = __float_as_uint(__uint_as_float(raw[h][4 * c + 1]) * f[1]);
                    v.z = __float_as_uint(__uint_as_float(raw[h][4 * c + 2]) * f[2]);
                    v.w = __float_as_uint(__uint_as_float(raw[h][4 * c + 3]) * f[3]);
                    sts128(stg + (uint32_t)(h * ENC_TILE_BYTES + r * 128 + ((c ^ (r & 7)) << 4)), v);
                }
            fence_proxy_async_smem();
            epi_bar_sync();
            if (tma) {
                if (leader) {
                    tma_store_3d(&maps.x[u.type], stg, j * 64, u.node, (int)row0);
                    tma_store_3d(&maps.x[u.type], stg + ENC_TILE_BYTES, j * 64 + 32, u.node, (int)row0);
                    tma_store_commit();
                }
            } else {
                // rows that are not a multiple of 16 bytes: consecutive threads store consecutive columns of one graph row
                const int cols = K - j * 64 < 64 ? K - j * 64 : 64;
                for (int e = tid - 64; e < TILE_M * cols; e += 128) {
                    const int rr = e / cols, cc = e - rr * cols;
                    if (row0 + rr >= B) break;
                    const uint32_t a = stg + (uint32_t)((cc >> 5) * ENC_TILE_BYTES + rr * 128 + ((((cc & 31) >> 2) ^ (rr & 7)) << 4) + (cc & 3) * 4);
                    float v;
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
                    dx[((row0 + rr) * nodes + u.node) * K + j * 64 + cc] = v;
                }
            }
        }
        if (leader) tma_store_wait_all();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, DX_TMEM_COLS);
    }
}

}  // namespace mshgnn
