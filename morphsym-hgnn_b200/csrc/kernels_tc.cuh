// tcgen05 tensor-core kernels of the MS-HGNN hot path (MSHGNN_MODE_TC / MSHGNN_MODE_TC_1X), sm_100a only.
//
//  k_tc_rowgemm : the same tile/chunk program as k_rowgemm (kernels_simt.cuh) for slab inputs:
//        D[128 graphs, 128] = sum_chunks A_c[128, 128] * W_c[128, 128]^T + fused epilogue.
//     * operands are fp16; every activation / weight value v is stored as a pair (hi, lo) with
//       hi = fp16(v), lo = fp16(v - hi)  (~22 significant bits).  MODE_TC issues three MMAs per chunk
//       (hi*hi + lo*hi + hi*lo, fp32 accumulation in TMEM) which keeps forward pre-activations at fp32
//       accuracy - required because ReLU makes the gradient discontinuous in the forward numerics
//       (DESIGN.md "precision").  MODE_TC_1X issues hi*hi only.
//     * TMA (cp.async.bulk.tensor, SWIZZLE_128B) stages the slot tile picked by the gather table and the
//       weight tile straight into the UMMA shared-memory layout: the morphology gather never touches a
//       register.  One elected thread issues tcgen05.mma; the accumulator lives in TMEM; four epilogue
//       warps read it back with tcgen05.ld (one thread per graph row) and apply bias / ReLU / mask /
//       residual, then write the fp32 slab plus its (hi, lo) fp16 images for the next layer's TMA.
//  warp roles: 0 = TMA producer, 1 = MMA issuer + TMEM owner, 2..5 = epilogue.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace mshgnn {

constexpr int TC_STAGES = 3;
constexpr int TC_KB = 32;                          // K columns per pipeline stage of the row-GEMM (one 64B-swizzled block)
constexpr int TC_TILE_BYTES = 128 * TC_KB * 2;     // 128 rows x 32 fp16 = 8 KB
constexpr int TC_STAGE_BYTES = 4 * TC_TILE_BYTES;  // A_hi, A_lo, W_hi, W_lo = 32 KB
constexpr int TC_SMEM_BYTES = TC_STAGES * TC_STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;   // 2 CTAs per SM
constexpr int TC_THREADS = 192;
constexpr float TC_W_SCALE = 256.f;                // weights are stored as fp16 pairs of (w * 2^8)
constexpr float TC_W_UNSCALE = 1.f / 256.f;
// The low halves are stored unscaled: lo = fp16(v - hi).  |lo| <= 2^-11 |v|, so lo is a normal fp16 (pair error 2^-22 |v|)
// for |v| >= 2^-3 and a subnormal one below that (pair error <= 2^-25 absolute).  Every slab the kernels carry is O(1) by
// construction (z-scored inputs, ReLU features, gradients pre-multiplied by G ~ #output rows), so the absolute floor sits
// seven decades under the tensor norms - and the three products hi*hi + lo*hi + hi*lo share ONE fp32 accumulator in
// TMEM (128 columns per 128x128 tile), which is what lets a CTA keep two row tiles x two accumulator sets resident.
constexpr float TC_LO_SCALE = LO_SCALE;
constexpr float TC_LO_UNSCALE = 1.f / LO_SCALE;
constexpr uint32_t TC_TMEM_COLS = 128;

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128B-swizzled shared-memory operand: 8-row groups 1024 B apart (SBO), descriptor version 1.
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr) {
    const uint32_t lo = ((saddr & 0x3FFFFu) >> 4) | (1u << 16);
    const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
    return ((uint64_t)hi << 32) | lo;
}
// K-major, 64B-swizzled operand (32 fp16 of K per row): 8-row groups 512 B apart, layout type 4 (SWIZZLE_64B).
__device__ __forceinline__ uint64_t smem_desc_sw64(uint32_t saddr) {
    const uint32_t lo = ((saddr & 0x3FFFFu) >> 4) | (1u << 16);
    const uint32_t hi = (512u >> 4) | (1u << 14) | (4u << 29);
    return ((uint64_t)hi << 32) | lo;
}
// kind::f16, A = B = fp16, D = fp32, both K-major, M = 128, N = 128
constexpr uint32_t TC_IDESC = (1u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24);

// first 256-byte row of each fp16 image, relative to the workspace base: one TMA map over the whole workspace
// ([total/256 rows][128 fp16]) then reaches every activation / gradient / weight image.
struct BufRows {
    int hi[MAX_BUFS];
    int lo[MAX_BUFS];
    int w_hi, w_lo;              // 128x128 weight images (row = w16_row of the chunk)
};

struct alignas(64) TcMaps {
    CUtensorMap k;               // box 32 columns x 128 rows, SWIZZLE_64B : MMA operand K blocks (activations and weights)
    CUtensorMap o;               // box 64 columns x 128 rows, SWIZZLE_128B: epilogue tiles (residual in, results out)
};

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
                 "r"(src), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// 8 consecutive values -> 16 bytes of the hi image and 16 bytes of the lo image (packed conversions)
__device__ __forceinline__ void split8(const float* v, uint4& hi, uint4& lo) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float a = v[2 * j], b = v[2 * j + 1];
        const __half2 hh = __floats2half2_rn(a, b);
        const float2 g = __half22float2(hh);
        const __half2 ll = __floats2half2_rn((a - g.x) * TC_LO_SCALE, (b - g.y) * TC_LO_SCALE);
        h[j] = *reinterpret_cast<const uint32_t*>(&hh);
        l[j] = *reinterpret_cast<const uint32_t*>(&ll);
    }
    hi = make_uint4(h[0], h[1], h[2], h[3]);
    lo = make_uint4(l[0], l[1], l[2], l[3]);
}
__device__ __forceinline__ void join8_add(float* v, const uint4 hi, const uint4 lo) {
    const uint32_t h[4] = {hi.x, hi.y, hi.z, hi.w}, l[4] = {lo.x, lo.y, lo.z, lo.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&h[j]));
        const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&l[j]));
        v[2 * j] += fmaf(b.x, TC_LO_UNSCALE, a.x);
        v[2 * j + 1] += fmaf(b.y, TC_LO_UNSCALE, a.y);
    }
}

// Epilogue shared by the row-GEMM kernels and the encoder.  Epilogue warps own one TMEM lane quarter each (one thread per
// graph row); a GROUP of four warps covers the 128 rows.  With two groups each takes one 64-column half of the tile, with
// one group it walks both halves.  accumulators (D0 + D1 * 2^-11) -> bias / ReLU / stored mask / residual -> (hi, lo) fp16
// pairs written into 128B-swizzled staging tiles in shared memory -> TMA stores.  The residual tile arrives the same way
// (TMA load into the staging tiles, combined in place), so no thread ever touches a global activation row directly: every
// HBM/L2 transaction of the activation stream is a full-line bulk transfer.  A masked second output (dc = dh (*) ReLU mask)
// is produced by clearing the masked-off fp16 lanes of the staged tile in place after the first store has been read.
struct EpiSmem {
    uint32_t stg;        // 64 KB: [column half][hi | lo] tiles of 128 rows x 64 fp16 (16 KB each)
    uint32_t bias;       // 512 B: bias of the current tile
    uint32_t res_bar;    // mbarriers (one per group, 8 bytes apart): residual tiles landed
    uint32_t accum_bar;  // mbarrier: accumulator complete (non-persistent kernels: operand pipeline drained, too)
    uint32_t free_bar;   // persistent kernel: mbarrier every epilogue thread arrives on once the accumulator is drained (0: none)
    uint32_t acc_parity, res_parity;
    int persistent;      // staging is dedicated memory: the residual is fetched before the accumulator is waited for
    int n_groups;        // 1 or 2
};

__device__ __forceinline__ void group_bar_sync(const int g) { asm volatile("bar.sync %0, 128;" ::"r"(g + 1) : "memory"); }

// clears the fp16 lanes of a 16-byte chunk whose mask bit is off (bits of `m`, lowest = first lane)
__device__ __forceinline__ uint4 mask8(const uint4 v, const uint32_t m) {
    uint4 r;
    r.x = v.x & (((m & 1u) ? 0xFFFFu : 0u) | ((m & 2u) ? 0xFFFF0000u : 0u));
    r.y = v.y & (((m & 4u) ? 0xFFFFu : 0u) | ((m & 8u) ? 0xFFFF0000u : 0u));
    r.z = v.z & (((m & 16u) ? 0xFFFFu : 0u) | ((m & 32u) ? 0xFFFF0000u : 0u));
    r.w = v.w & (((m & 64u) ? 0xFFFFu : 0u) | ((m & 128u) ? 0xFFFF0000u : 0u));
    return r;
}

__device__ __forceinline__ void tc_epilogue(const Tile& t, const BufTable& bt, const BufRows& br, const CUtensorMap* map_o,
                                            const uint32_t tmem_base, const int row0, const int64_t B, const int64_t Bp,
                                            const int split, const int warp /*CTA warp index, epilogue warps start at 2*/,
                                            const int lane, const EpiSmem es) {
    const int q = warp & 3;                        // TMEM lane quarter this warp may access (hardware rule: warp index mod 4)
    const int grp = es.n_groups == 2 ? ((warp - 2) >> 2) : 0;
    const int h0 = es.n_groups == 2 ? grp : 0, h1 = es.n_groups == 2 ? grp + 1 : 2;    // column halves of this group
    const bool leader = ((warp - 2) & 3) == 0 && lane == 0;                                // one per group
    const int rl = q * 32 + lane;                  // row inside the tile
    const int64_t row = (int64_t)row0 + rl;
    const bool live = row < B;
    const uint32_t rsw = (uint32_t)(rl & 7);
    const uint32_t rbase = (uint32_t)rl * 128u;
    const uint32_t res_bar = es.res_bar + 8u * grp;
    const bool has_out = t.out_buf >= 0, has_out2 = t.out2_buf >= 0, has_res = t.res_buf >= 0;
    const bool want_mask = t.relu || t.mask_out_buf >= 0;

    auto fetch_residual = [&]() {
        const int r_hi = br.hi[t.res_buf] + (int)((int64_t)t.res_slot * Bp) + row0, r_lo = br.lo[t.res_buf] + (int)((int64_t)t.res_slot * Bp) + row0;
        mbar_expect_tx(res_bar, (uint32_t)(h1 - h0) * 2u * 16384u);
        for (int half = h0; half < h1; ++half) {
            tma_load_2d(es.stg + half * 32768, map_o, res_bar, half * 64, r_hi);
            tma_load_2d(es.stg + half * 32768 + 16384, map_o, res_bar, half * 64, r_lo);
        }
    };
    if (es.persistent) {
        // the staging tiles still feed the previous item's TMA stores: wait until those have been read, then (residual
        // tiles) fetch early so that their latency hides behind the MMAs of this item
        if (leader) {
            tma_store_wait_read();
            if (has_res) fetch_residual();
        }
    }
    // bias of this group's columns -> shared memory (read back as broadcasts)
    if (rl < 64 * (h1 - h0)) {
        const int c = h0 * 64 + rl;
        const float bv = t.bias_buf >= 0 ? __ldg((const float*)bt.p[t.bias_buf] + t.bias_off + c) : 0.f;
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(es.bias + 4u * c), "f"(bv) : "memory");
    }
    uint4 pm = make_uint4(~0u, ~0u, ~0u, ~0u), m2 = make_uint4(~0u, ~0u, ~0u, ~0u);
    if (live && t.posmask_buf >= 0) pm = __ldg(reinterpret_cast<const uint4*>(bt.p[t.posmask_buf]) + (int64_t)t.posmask_slot * Bp + row);
    if (live && has_out2 && t.out2_mask_kind == MK_BITS)
        m2 = __ldg(reinterpret_cast<const uint4*>(bt.p[t.out2_mask_buf]) + (int64_t)t.out2_mask_slot * Bp + row);
    const uint32_t pmw[4] = {pm.x, pm.y, pm.z, pm.w}, m2w[4] = {m2.x, m2.y, m2.z, m2.w};
    uint32_t mw[4] = {0u, 0u, 0u, 0u};
    group_bar_sync(grp);

    mbar_wait(es.accum_bar, es.acc_parity);
    tc_fence_after();
    if (has_res) {
        if (leader && !es.persistent) fetch_residual();
        mbar_wait(res_bar, es.res_parity);
    }
#pragma unroll 1
    for (int half = h0; half < h1; ++half) {
#pragma unroll 1
        for (int c2 = 0; c2 < 2; ++c2) {
            const int cc = half * 2 + c2;
            uint32_t raw[32];
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + cc * 32, raw);
            tmem_ld_wait();
            if (cc == 2 * h1 - 1 && es.free_bar) {       // last read of this accumulator by this thread: hand it back
                tc_fence_before();
                mbar_arrive(es.free_bar);
            }
            float v[32];
            unsigned mask = 0;
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
                float4 b4;
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b4.x), "=f"(b4.y), "=f"(b4.z), "=f"(b4.w) : "r"(es.bias + 4u * (cc * 32 + j4 * 4)));
                const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int j = j4 * 4 + e;
                    float x = fmaf(__uint_as_float(raw[j]), TC_W_UNSCALE, bb[e]);
                    if (want_mask && x > 0.f) mask |= 1u << j;
                    if (t.relu) x = fmaxf(x, 0.f);
                    v[j] = x;
                }
            }
            mw[cc] = mask;
            if (t.posmask_buf >= 0) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = ((pmw[cc] >> j) & 1u) ? v[j] : 0.f;
            }
            const uint32_t tile = es.stg + (uint32_t)half * 32768u + rbase;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const uint32_t a = tile + ((((uint32_t)(c2 * 4 + g)) ^ rsw) << 4);
                if (has_res) join8_add(v + g * 8, lds128(a), lds128(a + 16384));
                if (has_out || has_out2) {
                    uint4 hi, lo;
                    split8(v + g * 8, hi, lo);
                    if (!has_out) { hi = mask8(hi, m2w[cc] >> (g * 8)); lo = mask8(lo, m2w[cc] >> (g * 8)); }
                    if (!live) { hi = make_uint4(0u, 0u, 0u, 0u); lo = hi; }     // rows [B, Bp) of every image stay zero
                    sts128(a, hi);
                    sts128(a + 16384, lo);
                }
            }
        }
        fence_proxy_async_smem();
        group_bar_sync(grp);
        if (leader) {
            const int ob = has_out ? t.out_buf : t.out2_buf, os = has_out ? t.out_slot : t.out2_slot;
            if (ob >= 0) {
                const int o = (int)((int64_t)os * Bp) + row0;
                tma_store_2d(map_o, es.stg + (uint32_t)half * 32768u, half * 64, br.hi[ob] + o);
                tma_store_2d(map_o, es.stg + (uint32_t)half * 32768u + 16384u, half * 64, br.lo[ob] + o);
                tma_store_commit();
            }
        }
    }
    if (has_out && has_out2) {
        // second output = first output with the masked-off lanes cleared, made in place once the first store has read the tile
        if (leader) tma_store_wait_read();
        group_bar_sync(grp);
        for (int half = h0; half < h1; ++half) {
            const uint32_t tile = es.stg + (uint32_t)half * 32768u + rbase;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const uint32_t a = tile + ((((uint32_t)c) ^ rsw) << 4);
                const uint32_t m = m2w[half * 2 + (c >> 2)] >> ((c & 3) * 8);
                sts128(a, mask8(lds128(a), m));
                sts128(a + 16384, mask8(lds128(a + 16384), m));
            }
        }
        fence_proxy_async_smem();
        group_bar_sync(grp);
        if (leader) {
            const int o = (int)((int64_t)t.out2_slot * Bp) + row0;
            for (int half = h0; half < h1; ++half) {
                tma_store_2d(map_o, es.stg + (uint32_t)half * 32768u, half * 64, br.hi[t.out2_buf] + o);
                tma_store_2d(map_o, es.stg + (uint32_t)half * 32768u + 16384u, half * 64, br.lo[t.out2_buf] + o);
            }
            tma_store_commit();
        }
    }
    if (live && t.mask_out_buf >= 0) {
        uint32_t* mp = reinterpret_cast<uint32_t*>(bt.p[t.mask_out_buf]) + ((int64_t)t.mask_out_slot * Bp + row) * 4;
        if (h1 - h0 == 2) *reinterpret_cast<uint4*>(mp) = make_uint4(mw[0], mw[1], mw[2], mw[3]);
        else *reinterpret_cast<uint2*>(mp + 2 * h0) = make_uint2(mw[2 * h0], mw[2 * h0 + 1]);
    }
    if (leader && !es.persistent) tma_store_wait_all();
}

// Epilogue of the persistent kernel: ONE group of four warps (one TMEM lane quarter each) drains a whole 128 x 128
// accumulator through its private 32 KB staging pair (hi | lo tiles of 128 rows x 64 fp16), one column half after the
// other.  The two groups of a CTA work on ALTERNATE items (group g always owns accumulator set g), so the latency chain
// of one item - residual tiles in by TMA, accumulator read-back, TMA stores that must have read the staging before it is
// reused - overlaps the arithmetic of the other group instead of stalling all eight warps at once (ncu: with both groups
// on the same item the epilogue warps, not the MMA or the operand stream, paced the kernel).
__device__ __forceinline__ void tc_epilogue_alt(const Tile& t, const BufTable& bt, const BufRows& br, const CUtensorMap* map_o,
                                                const uint32_t tmem_acc, const int row0, const int64_t B, const int64_t Bp,
                                                const int split, const int warp, const int lane, const int grp, const EpiSmem es,
                                                uint32_t& res_count) {
    const int q = warp & 3;                        // TMEM lane quarter this warp may access (hardware rule: warp index mod 4)
    const bool leader = ((warp - 2) & 3) == 0 && lane == 0;
    const int rl = q * 32 + lane;                  // row inside the tile
    const int64_t row = (int64_t)row0 + rl;
    const bool live = row < B;
    const uint32_t rsw = (uint32_t)(rl & 7);
    const uint32_t tile = es.stg + (uint32_t)rl * 128u;
    const bool has_out = t.out_buf >= 0, has_out2 = t.out2_buf >= 0, has_res = t.res_buf >= 0;
    const bool want_mask = t.relu || t.mask_out_buf >= 0;

    auto fetch_residual = [&](const int half) {
        const int r_hi = br.hi[t.res_buf] + (int)((int64_t)t.res_slot * Bp) + row0, r_lo = br.lo[t.res_buf] + (int)((int64_t)t.res_slot * Bp) + row0;
        mbar_expect_tx(es.res_bar, 2u * 16384u);
        tma_load_2d(es.stg, map_o, es.res_bar, half * 64, r_hi);
        tma_load_2d(es.stg + 16384, map_o, es.res_bar, half * 64, r_lo);
    };
    // the staging tiles may still feed this group's previous TMA stores: wait until those have been read, then fetch the
    // residual of the first column half early so that its latency hides behind the MMAs of this item
    if (leader) {
        tma_store_wait_read();
        if (has_res) fetch_residual(0);
    }
    {
        const float bv = t.bias_buf >= 0 ? __ldg((const float*)bt.p[t.bias_buf] + t.bias_off + rl) : 0.f;
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(es.bias + 4u * rl), "f"(bv) : "memory");
    }
    uint4 pm = make_uint4(~0u, ~0u, ~0u, ~0u), m2 = make_uint4(~0u, ~0u, ~0u, ~0u);
    if (live && t.posmask_buf >= 0) pm = __ldg(reinterpret_cast<const uint4*>(bt.p[t.posmask_buf]) + (int64_t)t.posmask_slot * Bp + row);
    if (live && has_out2 && t.out2_mask_kind == MK_BITS)
        m2 = __ldg(reinterpret_cast<const uint4*>(bt.p[t.out2_mask_buf]) + (int64_t)t.out2_mask_slot * Bp + row);
    const uint32_t pmw[4] = {pm.x, pm.y, pm.z, pm.w}, m2w[4] = {m2.x, m2.y, m2.z, m2.w};
    uint32_t mw[4] = {0u, 0u, 0u, 0u};
    group_bar_sync(grp);

    mbar_wait(es.accum_bar, es.acc_parity);
    tc_fence_after();
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
        if (half == 1) {
            if (leader) {
                tma_store_wait_read();
                if (has_res) fetch_residual(1);
            }
            group_bar_sync(grp);
        }
        if (has_res) {
            mbar_wait(es.res_bar, res_count & 1u);
            ++res_count;
        }
#pragma unroll 1
        for (int c2 = 0; c2 < 2; ++c2) {
            const int cc = half * 2 + c2;
            uint32_t raw[32];
            tmem_ld32(tmem_acc + ((uint32_t)(q * 32) << 16) + cc * 32, raw);
            tmem_ld_wait();
            if (cc == 3) {                         // last read of this accumulator by this thread: hand it back
                tc_fence_before();
                mbar_arrive(es.free_bar);
            }
            float v[32];
            unsigned mask = 0;
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
                float4 b4;
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b4.x), "=f"(b4.y), "=f"(b4.z), "=f"(b4.w) : "r"(es.bias + 4u * (cc * 32 + j4 * 4)));
                const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int j = j4 * 4 + e;
                    float x = fmaf(__uint_as_float(raw[j]), TC_W_UNSCALE, bb[e]);
                    if (want_mask && x > 0.f) mask |= 1u << j;
                    if (t.relu) x = fmaxf(x, 0.f);
                    v[j] = x;
                }
            }
            mw[cc] = mask;
            if (t.posmask_buf >= 0) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = ((pmw[cc] >> j) & 1u) ? v[j] : 0.f;
            }
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const uint32_t a = tile + ((((uint32_t)(c2 * 4 + g)) ^ rsw) << 4);
                if (has_res) join8_add(v + g * 8, lds128(a), lds128(a + 16384));
                if (has_out || has_out2) {
                    uint4 hi, lo;
                    split8(v + g * 8, hi, lo);
                    if (!has_out) { hi = mask8(hi, m2w[cc] >> (g * 8)); lo = mask8(lo, m2w[cc] >> (g * 8)); }
                    if (!live) { hi = make_uint4(0u, 0u, 0u, 0u); lo = hi; }     // rows [B, Bp) of every image stay zero
                    sts128(a, hi);
                    sts128(a + 16384, lo);
                }
            }
        }
        fence_proxy_async_smem();
        group_bar_sync(grp);
        if (leader) {
            const int ob = has_out ? t.out_buf : t.out2_buf, os = has_out ? t.out_slot : t.out2_slot;
            if (ob >= 0) {
                const int o = (int)((int64_t)os * Bp) + row0;
                tma_store_2d(map_o, es.stg, half * 64, br.hi[ob] + o);
                tma_store_2d(map_o, es.stg + 16384u, half * 64, br.lo[ob] + o);
                tma_store_commit();
            }
        }
        if (has_out && has_out2) {
            // second output = first output with the masked-off lanes cleared, made in place once the first store has read the tile
            if (leader) tma_store_wait_read();
            group_bar_sync(grp);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const uint32_t a = tile + ((((uint32_t)c) ^ rsw) << 4);
                const uint32_t m = m2w[half * 2 + (c >> 2)] >> ((c & 3) * 8);
                sts128(a, mask8(lds128(a), m));
                sts128(a + 16384, mask8(lds128(a + 16384), m));
            }
            fence_proxy_async_smem();
            group_bar_sync(grp);
            if (leader) {
                const int o = (int)((int64_t)t.out2_slot * Bp) + row0;
                tma_store_2d(map_o, es.stg, half * 64, br.hi[t.out2_buf] + o);
                tma_store_2d(map_o, es.stg + 16384u, half * 64, br.lo[t.out2_buf] + o);
                tma_store_commit();
            }
        }
    }
    if (live && t.mask_out_buf >= 0) {
        uint32_t* mp = reinterpret_cast<uint32_t*>(bt.p[t.mask_out_buf]) + ((int64_t)t.mask_out_slot * Bp + row) * 4;
        *reinterpret_cast<uint4*>(mp) = make_uint4(mw[0], mw[1], mw[2], mw[3]);
    }
}

// Epilogue of the persistent kernel, 16 warps: FOUR groups of four warps; group g drains the 32-column quarter g of the
// accumulator (one tcgen05.ld.32x32b.x32 per thread) through a private 16 KB staging pair (hi | lo tiles of 128 rows x
// 32 fp16, 64 B rows, SWIZZLE_64B - the same box shape as the operand K blocks, so the operand tensor map serves the
// residual loads and the image stores).  Ablation runs (DESIGN 3.1) showed the 8-warp epilogue alone - no loads, no MMAs -
// taking 63-70 % of the kernel time at ~22 instructions per element with two warps per scheduler; four warps per scheduler
// hide each other's dependent-issue and shared-memory latency.
__device__ __forceinline__ void tc_epilogue_q(const Tile& t, const BufTable& bt, const BufRows& br, const CUtensorMap* map_k,
                                              const uint32_t tmem_acc, const int row0, const int64_t B, const int64_t Bp,
                                              const int warp, const int lane, const int grp, const EpiSmem es, uint32_t& res_count) {
    const int q = warp & 3;                        // TMEM lane quarter this warp may access (hardware rule: warp index mod 4)
    const bool leader = q == 2 && lane == 0;       // first warp of the group (warps 2 + 4g .. 5 + 4g): warp index = 2 mod 4
    const int rl = q * 32 + lane;                  // row inside the tile
    const int64_t row = (int64_t)row0 + rl;
    const bool live = row < B;
    const uint32_t rsw = (uint32_t)((rl >> 1) & 3);     // SWIZZLE_64B: 16-byte chunk index ^= address bits [7, 9)
    const uint32_t tile = es.stg + (uint32_t)rl * 64u;
    const bool has_out = t.out_buf >= 0, has_out2 = t.out2_buf >= 0, has_res = t.res_buf >= 0;
    const bool want_mask = t.relu || t.mask_out_buf >= 0;
    const int col0 = grp * 32;

    if (leader) {
        // the staging tiles may still feed this group's previous TMA stores
        tma_store_wait_read();
        if (has_res) {
            const int r_hi = br.hi[t.res_buf] + (int)((int64_t)t.res_slot * Bp) + row0, r_lo = br.lo[t.res_buf] + (int)((int64_t)t.res_slot * Bp) + row0;
            mbar_expect_tx(es.res_bar, 2u * 8192u);
            tma_load_2d(es.stg, map_k, es.res_bar, col0, r_hi);
            tma_load_2d(es.stg + 8192, map_k, es.res_bar, col0, r_lo);
        }
    }
    if (rl < 32) {
        const float bv = t.bias_buf >= 0 ? __ldg((const float*)bt.p[t.bias_buf] + t.bias_off + col0 + rl) : 0.f;
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(es.bias + 4u * rl), "f"(bv) : "memory");
    }
    uint32_t pm = ~0u, m2 = ~0u;
    if (live && t.posmask_buf >= 0) pm = __ldg(reinterpret_cast<const uint32_t*>(bt.p[t.posmask_buf]) + ((int64_t)t.posmask_slot * Bp + row) * 4 + grp);
    if (live && has_out2 && t.out2_mask_kind == MK_BITS)
        m2 = __ldg(reinterpret_cast<const uint32_t*>(bt.p[t.out2_mask_buf]) + ((int64_t)t.out2_mask_slot * Bp + row) * 4 + grp);
    group_bar_sync(grp);

    mbar_wait(es.accum_bar, es.acc_parity);
    tc_fence_after();
    uint32_t raw[32];
    tmem_ld32(tmem_acc + ((uint32_t)(q * 32) << 16) + col0, raw);
    tmem_ld_wait();
    tc_fence_before();
    mbar_arrive(es.free_bar);                      // this thread's part of the accumulator is in registers
    if (has_res) {
        mbar_wait(es.res_bar, res_count & 1u);
        ++res_count;
    }
    float v[32];
    unsigned mask = 0;
#pragma unroll
    for (int j4 = 0; j4 < 8; ++j4) {
        float4 b4;
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b4.x), "=f"(b4.y), "=f"(b4.z), "=f"(b4.w) : "r"(es.bias + 16u * j4));
        const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int j = j4 * 4 + e;
            float x = fmaf(__uint_as_float(raw[j]), TC_W_UNSCALE, bb[e]);
            if (want_mask && x > 0.f) mask |= 1u << j;
            if (t.relu) x = fmaxf(x, 0.f);
            v[j] = x;
        }
    }
    if (t.posmask_buf >= 0) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = ((pm >> j) & 1u) ? v[j] : 0.f;
    }
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        const uint32_t a = tile + ((((uint32_t)g) ^ rsw) << 4);
        if (has_res) join8_add(v + g * 8, lds128(a), lds128(a + 8192));
        if (has_out || has_out2) {
            uint4 hi, lo;
            split8(v + g * 8, hi, lo);
            if (!has_out) { hi = mask8(hi, m2 >> (g * 8)); lo = mask8(lo, m2 >> (g * 8)); }
            if (!live) { hi = make_uint4(0u, 0u, 0u, 0u); lo = hi; }     // rows [B, Bp) of every image stay zero
            sts128(a, hi);
            sts128(a + 8192, lo);
        }
    }
    fence_proxy_async_smem();
    group_bar_sync(grp);
    if (leader) {
        const int ob = has_out ? t.out_buf : t.out2_buf, os = has_out ? t.out_slot : t.out2_slot;
        if (ob >= 0) {
            const int o = (int)((int64_t)os * Bp) + row0;
            tma_store_2d(map_k, es.stg, col0, br.hi[ob] + o);
            tma_store_2d(map_k, es.stg + 8192u, col0, br.lo[ob] + o);
            tma_store_commit();
        }
    }
    if (has_out && has_out2) {
        // second output = first output with the masked-off lanes cleared, made in place once the first store has read the tile
        if (leader) tma_store_wait_read();
        group_bar_sync(grp);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const uint32_t a = tile + ((((uint32_t)c) ^ rsw) << 4);
            const uint32_t m = m2 >> (c * 8);
            sts128(a, mask8(lds128(a), m));
            sts128(a + 8192, mask8(lds128(a + 8192), m));
        }
        fence_proxy_async_smem();
        group_bar_sync(grp);
        if (leader) {
            const int o = (int)((int64_t)t.out2_slot * Bp) + row0;
            tma_store_2d(map_k, es.stg, col0, br.hi[t.out2_buf] + o);
            tma_store_2d(map_k, es.stg + 8192u, col0, br.lo[t.out2_buf] + o);
            tma_store_commit();
        }
    }
    if (live && t.mask_out_buf >= 0)
        *(reinterpret_cast<uint32_t*>(bt.p[t.mask_out_buf]) + ((int64_t)t.mask_out_slot * Bp + row) * 4 + grp) = mask;
}

// ------------------------------------------------------------------------------------------
// row-GEMM on tcgen05
// ------------------------------------------------------------------------------------------
//  Two CTAs share an SM (96 KB of operand pipeline and 256 TMEM columns each): while one CTA drains its accumulator
//  through the epilogue the other one keeps the tensor pipe and the L2->SMEM stream busy.
//  grid = (tiles of the launch, row tiles): CTAs that run together read the same 128 graphs, so every source slot
//  tile is fetched from HBM once and re-read from L2 by the other destination slots that gather it.
__global__ void __launch_bounds__(TC_THREADS, 2)
k_tc_rowgemm(const __grid_constant__ TcMaps maps, const Tile* __restrict__ tiles, const BufTable bt, const BufRows br,
             const int64_t B, const int64_t Bp, const int split) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ Tile t;
    __shared__ __align__(16) float bias_s[H];
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TC_STAGES * TC_STAGE_BYTES);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + TC_STAGES), accum_bar = smem_u32(bars + 2 * TC_STAGES),
                   res_bar = smem_u32(bars + 2 * TC_STAGES + 1);
    const uint32_t smem_base = smem_u32(smem);

    {
        const int* src = reinterpret_cast<const int*>(tiles + blockIdx.x);
        int* dst = reinterpret_cast<int*>(&t);
        for (int i = tid; i < (int)(sizeof(Tile) / 4); i += TC_THREADS) dst[i] = src[i];
    }
    if (tid == 0) {
        for (int s = 0; s < TC_STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        mbar_init(accum_bar, 1);
        mbar_init(res_bar, 1);
        mbar_init(res_bar + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(&tmem_base_s), TC_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    const int row0 = blockIdx.y * TILE_M;
    const int n_steps = t.n_chunks * (H / TC_KB);

    if (warp == 0) {
        if (lane == 0) {
            const uint32_t tx_bytes = split ? 4 * TC_TILE_BYTES : 2 * TC_TILE_BYTES;
            for (int i = 0; i < n_steps; ++i) {
                const int s = i % TC_STAGES;
                mbar_wait(empty0 + 8 * s, ((i / TC_STAGES) & 1) ^ 1);
                const Chunk& ch = t.chunks[i / (H / TC_KB)];
                const int kcol = (i % (H / TC_KB)) * TC_KB;
                const int arow = (int)((int64_t)ch.a_slot * Bp) + row0;
                const uint32_t st = smem_base + s * TC_STAGE_BYTES;
                const uint32_t fb = full0 + 8 * s;
                mbar_expect_tx(fb, tx_bytes);
                tma_load_2d(st, &maps.k, fb, kcol, br.hi[ch.a_buf] + arow);
                tma_load_2d(st + 2 * TC_TILE_BYTES, &maps.k, fb, kcol, br.w_hi + ch.w16_row);
                if (split) {
                    tma_load_2d(st + TC_TILE_BYTES, &maps.k, fb, kcol, br.lo[ch.a_buf] + arow);
                    tma_load_2d(st + 3 * TC_TILE_BYTES, &maps.k, fb, kcol, br.w_lo + ch.w16_row);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            for (int i = 0; i < n_steps; ++i) {
                const int s = i % TC_STAGES;
                mbar_wait(full0 + 8 * s, (i / TC_STAGES) & 1);
                tc_fence_after();
                const uint32_t st = smem_base + s * TC_STAGE_BYTES;
                const uint64_t a_hi = smem_desc_sw64(st), a_lo = smem_desc_sw64(st + TC_TILE_BYTES);
                const uint64_t w_hi = smem_desc_sw64(st + 2 * TC_TILE_BYTES), w_lo = smem_desc_sw64(st + 3 * TC_TILE_BYTES);
#pragma unroll
                for (int ks = 0; ks < TC_KB / 16; ++ks) {
                    const uint64_t adv = (uint64_t)(ks * 2);      // +32 bytes (16 fp16) along K inside the swizzle atom
                    umma_f16(tmem_base, a_hi + adv, w_hi + adv, TC_IDESC, (i | ks) ? 1u : 0u);             // D0 += hi * hi
                    if (split) {
                        umma_f16(tmem_base, a_lo + adv, w_hi + adv, TC_IDESC, 1u);                         // D0 += lo * hi
                        umma_f16(tmem_base, a_hi + adv, w_lo + adv, TC_IDESC, 1u);                         // D0 += hi * lo
                    }
                }
                umma_commit(empty0 + 8 * s);          // frees the stage once these MMAs have read it
            }
            umma_commit(accum_bar);                   // accumulator complete, every stage drained
        }
        __syncwarp();
    } else {
        EpiSmem es;
        es.stg = smem_base; es.bias = smem_u32(bias_s); es.res_bar = res_bar; es.accum_bar = accum_bar;
        es.free_bar = 0; es.acc_parity = 0; es.res_parity = 0; es.persistent = 0; es.n_groups = 1;
        tc_epilogue(t, bt, br, &maps.o, tmem_base, row0, B, Bp, split, warp, lane, es);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TC_TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------
// persistent row-GEMM: one CTA per SM walks the (row tile, output tile) items of a launch
// ------------------------------------------------------------------------------------------
//  Three roles run decoupled, linked by mbarriers only: warp 0 streams operand K blocks by TMA (3-stage ring that keeps
//  running across items), warp 1 issues the MMAs into one of TWO accumulator sets in TMEM (2 x 256 columns), warps 2..5
//  drain the other set through the epilogue (dedicated staging tiles, residual prefetched).  So the tensor pipe never
//  waits for an epilogue, and tile prologues (barrier init, TMEM allocation, descriptor fetch) are paid once per SM.
//  Item i = blockIdx.x + k * gridDim.x  ->  row tile i / n_tiles, output tile i % n_tiles: CTAs that run together work
//  on the same few row tiles, so gathered source tiles are re-read from L2, not HBM.
constexpr int PK_MAX_TILES = 32;
constexpr int PK_STAGES = 4;
constexpr int PK_THREADS = 576;                                           // TMA warp, MMA warp, 16 epilogue warps
constexpr int PK_PIPE_BYTES = PK_STAGES * TC_STAGE_BYTES;                 // 128 KB operand ring
constexpr int PK_SMEM_BYTES = PK_PIPE_BYTES + 65536 + 1024 /*align*/ + 256 /*barriers*/;
constexpr uint32_t PK_TMEM_COLS = 256;

__global__ void __launch_bounds__(PK_THREADS, 1)
k_tc_rowgemm_persistent(const __grid_constant__ TcMaps maps, const Tile* __restrict__ tiles, const int n_tiles, const int n_items,
                        const BufTable bt, const BufRows br, const int64_t B, const int64_t Bp, const int split) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ Tile ts[PK_MAX_TILES];
    __shared__ __align__(16) float bias_s[4][32];         // one quarter per epilogue group
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + PK_PIPE_BYTES + 65536);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + PK_STAGES), acc_full0 = smem_u32(bars + 2 * PK_STAGES),
                   acc_free0 = smem_u32(bars + 2 * PK_STAGES + 2), res_bar = smem_u32(bars + 2 * PK_STAGES + 4);   // 4 residual barriers
    const uint32_t smem_base = smem_u32(smem);

    {
        const int* src = reinterpret_cast<const int*>(tiles);
        int* dst = reinterpret_cast<int*>(ts);
        for (int i = tid; i < n_tiles * (int)(sizeof(Tile) / 4); i += PK_THREADS) dst[i] = src[i];
    }
    if (tid == 0) {
        for (int s = 0; s < PK_STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        // acc_free: every epilogue thread (16 warps) arrives once per item
        for (int a = 0; a < 2; ++a) { mbar_init(acc_full0 + 8 * a, 1); mbar_init(acc_free0 + 8 * a, 512); }
        for (int g = 0; g < 4; ++g) mbar_init(res_bar + 8 * g, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(&tmem_base_s), PK_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    constexpr int SPC = H / TC_KB;                 // pipeline steps per chunk
    // Programmatic dependent launch: everything above (tile table, barriers, TMEM) ran while the previous kernel of the
    // stream was still draining; from here on this grid reads what that kernel wrote.  Our own dependents may be scheduled
    // as soon as every CTA of this grid has passed this point (they start on an SM when its CTA has exited).
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (warp == 0) {
        if (lane == 0) {
            const uint32_t tx_bytes = split ? 4 * TC_TILE_BYTES : 2 * TC_TILE_BYTES;
            uint32_t g = 0;                        // pipeline step counter, runs across items
            for (int i = blockIdx.x; i < n_items; i += gridDim.x) {
                const Tile& t = ts[i % n_tiles];
                const int row0 = (i / n_tiles) * TILE_M;
                const int n_steps = t.n_chunks * SPC;
                for (int j = 0; j < n_steps; ++j, ++g) {
                    const uint32_t s = g % PK_STAGES;
                    mbar_wait(empty0 + 8 * s, ((g / PK_STAGES) & 1) ^ 1);
                    const Chunk& ch = t.chunks[j / SPC];
                    const int kcol = (j % SPC) * TC_KB;
                    const int arow = (int)((int64_t)ch.a_slot * Bp) + row0;
                    const uint32_t st = smem_base + s * TC_STAGE_BYTES;
                    const uint32_t fb = full0 + 8 * s;
                    mbar_expect_tx(fb, tx_bytes);
                    tma_load_2d(st, &maps.k, fb, kcol, br.hi[ch.a_buf] + arow);
                    tma_load_2d(st + 2 * TC_TILE_BYTES, &maps.k, fb, kcol, br.w_hi + ch.w16_row);
                    if (split) {
                        tma_load_2d(st + TC_TILE_BYTES, &maps.k, fb, kcol, br.lo[ch.a_buf] + arow);
                        tma_load_2d(st + 3 * TC_TILE_BYTES, &maps.k, fb, kcol, br.w_lo + ch.w16_row);
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            uint32_t g = 0, k = 0;
            for (int i = blockIdx.x; i < n_items; i += gridDim.x, ++k) {
                const int n_steps = ts[i % n_tiles].n_chunks * SPC;
                const uint32_t a = k & 1;
                mbar_wait(acc_free0 + 8 * a, ((k >> 1) & 1) ^ 1);      // the epilogue has drained this accumulator set
                tc_fence_after();
                const uint32_t d0 = tmem_base + a * 128;
                for (int j = 0; j < n_steps; ++j, ++g) {
                    const uint32_t s = g % PK_STAGES;
                    mbar_wait(full0 + 8 * s, (g / PK_STAGES) & 1);
                    tc_fence_after();
                    const uint32_t st = smem_base + s * TC_STAGE_BYTES;
                    const uint64_t a_hi = smem_desc_sw64(st), a_lo = smem_desc_sw64(st + TC_TILE_BYTES);
                    const uint64_t w_hi = smem_desc_sw64(st + 2 * TC_TILE_BYTES), w_lo = smem_desc_sw64(st + 3 * TC_TILE_BYTES);
#pragma unroll
                    for (int ks = 0; ks < TC_KB / 16; ++ks) {
                        const uint64_t adv = (uint64_t)(ks * 2);
                        umma_f16(d0, a_hi + adv, w_hi + adv, TC_IDESC, (j | ks) ? 1u : 0u);
                        if (split) {
                            umma_f16(d0, a_lo + adv, w_hi + adv, TC_IDESC, 1u);
                            umma_f16(d0, a_hi + adv, w_lo + adv, TC_IDESC, 1u);
                        }
                    }
                    umma_commit(empty0 + 8 * s);
                }
                umma_commit(acc_full0 + 8 * a);
            }
        }
        __syncwarp();
    } else {
        // group g (warps 2 + 4g .. 5 + 4g) drains column quarter g of every item
        const int grp = (warp - 2) >> 2;
        EpiSmem es;
        es.stg = smem_base + PK_PIPE_BYTES + grp * 16384; es.bias = smem_u32(bias_s[grp]); es.res_bar = res_bar + 8 * grp;
        es.persistent = 1; es.n_groups = 4; es.res_parity = 0;
        uint32_t k = 0, n_res = 0;
        for (int i = blockIdx.x; i < n_items; i += gridDim.x, ++k) {
            const uint32_t a = k & 1;
            es.accum_bar = acc_full0 + 8 * a; es.free_bar = acc_free0 + 8 * a;
            es.acc_parity = (k >> 1) & 1;
            tc_epilogue_q(ts[i % n_tiles], bt, br, &maps.k, tmem_base + a * 128, (i / n_tiles) * TILE_M, B, Bp, warp, lane, grp, es, n_res);
        }
        if (((warp - 2) & 3) == 0 && lane == 0) tma_store_wait_all();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, PK_TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------
// persistent row-GEMM, two row tiles per item ("pair" kernel): every weight K block staged in shared memory feeds TWO
// 128-row accumulators, so the L2 -> SMEM operand stream per 128x128x128 product drops from 128 KB to 96 KB.  With the
// 16-warp epilogue the operand stream is the longest leg of an item (352 KB at the ~84 GB/s an SM gets of the chip-wide
// L2 cap = 4.2 us against 2.2 us of MMAs); the weights are the only operand neighbouring row tiles share.
//  Item i -> row pair i / n_tiles (rows [256 p, 256 p + 256)), output tile i % n_tiles.  Stage = [A0_hi, A0_lo, A1_hi,
//  A1_lo, W_hi, W_lo] x 8 KB, 3 stages.  TMEM: 2 accumulator sets x 2 row tiles x 128 columns = 512.  Each epilogue
//  group drains its column quarter of the two row tiles one after the other.
// ------------------------------------------------------------------------------------------
constexpr int PP_STAGES = 3;
constexpr int PP_STAGE_BYTES = 6 * TC_TILE_BYTES;                          // 48 KB
constexpr int PP_PIPE_BYTES = PP_STAGES * PP_STAGE_BYTES;                  // 144 KB operand ring
constexpr int PP_SMEM_BYTES = PP_PIPE_BYTES + 65536 + 1024 /*align*/ + 256 /*barriers*/;
constexpr uint32_t PP_TMEM_COLS = 512;

__global__ void __launch_bounds__(PK_THREADS, 1)
k_tc_rowgemm_pair(const __grid_constant__ TcMaps maps, const Tile* __restrict__ tiles, const int n_tiles, const int n_items,
                        const BufTable bt, const BufRows br, const int64_t B, const int64_t Bp, const int split) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ Tile ts[PK_MAX_TILES];
    __shared__ __align__(16) float bias_s[4][32];         // one quarter per epilogue group
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + PP_PIPE_BYTES + 65536);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + PP_STAGES), acc_full0 = smem_u32(bars + 2 * PP_STAGES),
                   acc_free0 = smem_u32(bars + 2 * PP_STAGES + 2), res_bar = smem_u32(bars + 2 * PP_STAGES + 4);   // 4 residual barriers
    const uint32_t smem_base = smem_u32(smem);

    {
        const int* src = reinterpret_cast<const int*>(tiles);
        int* dst = reinterpret_cast<int*>(ts);
        for (int i = tid; i < n_tiles * (int)(sizeof(Tile) / 4); i += PK_THREADS) dst[i] = src[i];
    }
    if (tid == 0) {
        for (int s = 0; s < PP_STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        // acc_free: every epilogue thread (16 warps) arrives once per row tile of the item (two row tiles per item)
        for (int a = 0; a < 2; ++a) { mbar_init(acc_full0 + 8 * a, 1); mbar_init(acc_free0 + 8 * a, 1024); }
        for (int g = 0; g < 4; ++g) mbar_init(res_bar + 8 * g, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(&tmem_base_s), PP_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    constexpr int SPC = H / TC_KB;                 // pipeline steps per chunk
    const int last_tile_row = (int)Bp - TILE_M;    // first row of the last 128-row tile
    // Programmatic dependent launch: everything above (tile table, barriers, TMEM) ran while the previous kernel of the
    // stream was still draining; from here on this grid reads what that kernel wrote.  Our own dependents may be scheduled
    // as soon as every CTA of this grid has passed this point (they start on an SM when its CTA has exited).
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (warp == 0) {
        if (lane == 0) {
            uint32_t g = 0;                        // pipeline step counter, runs across items
            for (int i = blockIdx.x; i < n_items; i += gridDim.x) {
                const Tile& t = ts[i % n_tiles];
                const int row0 = (i / n_tiles) * (2 * TILE_M);
                const bool two = row0 + TILE_M <= last_tile_row;
                const uint32_t tx_bytes = (uint32_t)((split ? 2 : 1) * (two ? 3 : 2) * TC_TILE_BYTES);
                const int n_steps = t.n_chunks * SPC;
                for (int j = 0; j < n_steps; ++j, ++g) {
                    const uint32_t s = g % PP_STAGES;
                    mbar_wait(empty0 + 8 * s, ((g / PP_STAGES) & 1) ^ 1);
                    const Chunk& ch = t.chunks[j / SPC];
                    const int kcol = (j % SPC) * TC_KB;
                    const int arow = (int)((int64_t)ch.a_slot * Bp) + row0;
                    const uint32_t st = smem_base + s * PP_STAGE_BYTES;
                    const uint32_t fb = full0 + 8 * s;
                    mbar_expect_tx(fb, tx_bytes);
                    tma_load_2d(st, &maps.k, fb, kcol, br.hi[ch.a_buf] + arow);
                    if (two) tma_load_2d(st + 2 * TC_TILE_BYTES, &maps.k, fb, kcol, br.hi[ch.a_buf] + arow + TILE_M);
                    tma_load_2d(st + 4 * TC_TILE_BYTES, &maps.k, fb, kcol, br.w_hi + ch.w16_row);
                    if (split) {
                        tma_load_2d(st + TC_TILE_BYTES, &maps.k, fb, kcol, br.lo[ch.a_buf] + arow);
                        if (two) tma_load_2d(st + 3 * TC_TILE_BYTES, &maps.k, fb, kcol, br.lo[ch.a_buf] + arow + TILE_M);
                        tma_load_2d(st + 5 * TC_TILE_BYTES, &maps.k, fb, kcol, br.w_lo + ch.w16_row);
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            uint32_t g = 0, k = 0;
            for (int i = blockIdx.x; i < n_items; i += gridDim.x, ++k) {
                const int n_steps = ts[i % n_tiles].n_chunks * SPC;
                const bool two = (i / n_tiles) * (2 * TILE_M) + TILE_M <= last_tile_row;
                const uint32_t a = k & 1;
                mbar_wait(acc_free0 + 8 * a, ((k >> 1) & 1) ^ 1);      // the epilogue has drained this accumulator set
                tc_fence_after();
                const uint32_t d0 = tmem_base + a * 256, d1 = d0 + 128;
                for (int j = 0; j < n_steps; ++j, ++g) {
                    const uint32_t s = g % PP_STAGES;
                    mbar_wait(full0 + 8 * s, (g / PP_STAGES) & 1);
                    tc_fence_after();
                    const uint32_t st = smem_base + s * PP_STAGE_BYTES;
                    const uint64_t a0_hi = smem_desc_sw64(st), a0_lo = smem_desc_sw64(st + TC_TILE_BYTES);
                    const uint64_t a1_hi = smem_desc_sw64(st + 2 * TC_TILE_BYTES), a1_lo = smem_desc_sw64(st + 3 * TC_TILE_BYTES);
                    const uint64_t w_hi = smem_desc_sw64(st + 4 * TC_TILE_BYTES), w_lo = smem_desc_sw64(st + 5 * TC_TILE_BYTES);
#pragma unroll
                    for (int ks = 0; ks < TC_KB / 16; ++ks) {
                        const uint64_t adv = (uint64_t)(ks * 2);
                        const uint32_t acc = (j | ks) ? 1u : 0u;
                        umma_f16(d0, a0_hi + adv, w_hi + adv, TC_IDESC, acc);
                        if (two) umma_f16(d1, a1_hi + adv, w_hi + adv, TC_IDESC, acc);
                        if (split) {
                            umma_f16(d0, a0_lo + adv, w_hi + adv, TC_IDESC, 1u);
                            if (two) umma_f16(d1, a1_lo + adv, w_hi + adv, TC_IDESC, 1u);
                            umma_f16(d0, a0_hi + adv, w_lo + adv, TC_IDESC, 1u);
                            if (two) umma_f16(d1, a1_hi + adv, w_lo + adv, TC_IDESC, 1u);
                        }
                    }
                    umma_commit(empty0 + 8 * s);
                }
                umma_commit(acc_full0 + 8 * a);
            }
        }
        __syncwarp();
    } else {
        // group g (warps 2 + 4g .. 5 + 4g) drains column quarter g of every item
        const int grp = (warp - 2) >> 2;
        EpiSmem es;
        es.stg = smem_base + PP_PIPE_BYTES + grp * 16384; es.bias = smem_u32(bias_s[grp]); es.res_bar = res_bar + 8 * grp;
        es.persistent = 1; es.n_groups = 4; es.res_parity = 0;
        uint32_t k = 0, n_res = 0;
        for (int i = blockIdx.x; i < n_items; i += gridDim.x, ++k) {
            const uint32_t a = k & 1;
            const int row0 = (i / n_tiles) * (2 * TILE_M);
            const bool two = row0 + TILE_M <= last_tile_row;
            es.accum_bar = acc_full0 + 8 * a; es.free_bar = acc_free0 + 8 * a;
            es.acc_parity = (k >> 1) & 1;
            tc_epilogue_q(ts[i % n_tiles], bt, br, &maps.k, tmem_base + a * 256, row0, B, Bp, warp, lane, grp, es, n_res);
            if (two) tc_epilogue_q(ts[i % n_tiles], bt, br, &maps.k, tmem_base + a * 256 + 128, row0 + TILE_M, B, Bp, warp, lane, grp, es, n_res);
            else mbar_arrive(es.free_bar);         // keeps the arrival count of the set at 1024
        }
        if (((warp - 2) & 3) == 0 && lane == 0) tma_store_wait_all();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, PP_TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------
// reduce-over-rows GEMM on tcgen05 (weight gradients):  dW[128 out, 128 in] = sum_pairs dC[rows,128]^T * A[rows,128]
// ------------------------------------------------------------------------------------------
//  The reduction dimension is the graph-row dimension, so both MMA operands are "MN-major": the fp16 images are
//  [row][feature] and a TMA box of 64 features x 64 rows (SWIZZLE_128B) is exactly the canonical MN-major SW128 atom
//  sequence (8 rows x 128 B per atom, SBO = 1024 B between 8-row groups, LBO = 8192 B between the two 64-feature
//  halves).  No transposed copy of any activation is ever made.
//  Bias gradients (column sums of dC) ride on the same operand: one extra N=16 MMA against an all-ones B tile.
//  Accumulators (TMEM columns): D0 [0,128) hi*hi, D1 [128,256) cross terms (x 2^11), D2 [256,272) colsum hi,
//  D3 [288,304) colsum lo (x 2^11).  One CTA = one task (<= 4 pairs) x one row split; fp32 partials go to part_w /
//  part_b and are summed in double by k_reduce_partials (deterministic, no atomics).
constexpr int BUF_PARAMS_ID = 0, BUF_DERIVED_ID = 1;     // plan.cuh BUF_PARAMS, BUF_DERIVED
constexpr int BUF_DC1_ID = 80;     // plan.cuh BUF_DCL0 - 1: dpre of the encoder (dc_{-1}), written by the layer-0 dX tiles

constexpr int DW_STAGES = 3;
constexpr int DW_KB = 64;                              // graph rows (MMA K) per pipeline stage
constexpr int DW_IMG_BYTES = DW_KB * H * 2;            // 64 rows x 128 fp16 = two 64x64 boxes
constexpr int DW_STAGE_BYTES = 4 * DW_IMG_BYTES;       // dC_hi, dC_lo, A_hi, A_lo
constexpr int DW_ONES_BYTES = 2048;
constexpr int DW_SMEM_BYTES = DW_STAGES * DW_STAGE_BYTES + DW_ONES_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
constexpr uint32_t DW_TMEM_COLS = 256;
constexpr int DW_MAX_PAIRS = 4;

// MN-major, 128B-swizzled operand of 128 (MN) x 16 (K) fp16: LBO = 8192 B (next 64 MN elements), SBO = 1024 B (next 8 K rows)
__device__ __forceinline__ uint64_t smem_desc_mn_sw128(uint32_t saddr) {
    const uint32_t lo = ((saddr & 0x3FFFFu) >> 4) | ((uint32_t)(DW_IMG_BYTES / 2 >> 4) << 16);
    const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
    return ((uint64_t)hi << 32) | lo;
}
// kind::f16, fp16 x fp16 -> fp32, A and B MN-major, M = 128, N = 128
constexpr uint32_t DW_IDESC = (1u << 4) | (1u << 15) | (1u << 16) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
// column sums: A MN-major (dC), B K-major (all ones), M = 128, N = 16
constexpr uint32_t DW_IDESC_CS = (1u << 4) | (1u << 15) | ((16u >> 3) << 17) | ((128u >> 4) << 24);

__global__ void __launch_bounds__(TC_THREADS, 1)
k_tc_reducegemm(const __grid_constant__ CUtensorMap map, const RTask* __restrict__ tasks, const RPair* __restrict__ pairs,
                const int task0, const BufRows br, const int64_t B, const int64_t Bp, const int rows_per, const int slot0 /*first partial slot of this launch*/,
                const int split, float* __restrict__ part_w, float* __restrict__ part_b, const int64_t Bm, const int n_splits, const int64_t part_slots) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ RTask t;
    __shared__ RPair prs[DW_MAX_PAIRS];
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* ones = smem + DW_STAGES * DW_STAGE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(ones + DW_ONES_BYTES);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + DW_STAGES), accum_bar = smem_u32(bars + 2 * DW_STAGES);
    const uint32_t smem_base = smem_u32(smem);

    const int task = task0 + blockIdx.x;
    if (tid < (int)(sizeof(RTask) / 4)) reinterpret_cast<int*>(&t)[tid] = reinterpret_cast<const int*>(tasks + task)[tid];
    for (int i = tid; i < DW_ONES_BYTES / 4; i += TC_THREADS) reinterpret_cast<uint32_t*>(ones)[i] = 0x3C003C00u;   // fp16 1.0 pairs
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");        // the ones tile is read by the MMA (async proxy)
    if (tid == 0) {
        for (int s = 0; s < DW_STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        mbar_init(accum_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(&tmem_base_s), DW_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    {
        const int np = t.n_pairs < DW_MAX_PAIRS ? t.n_pairs : DW_MAX_PAIRS;
        const int* src = reinterpret_cast<const int*>(pairs + t.pair_begin);
        int* dst = reinterpret_cast<int*>(prs);
        for (int i = tid; i < np * (int)(sizeof(RPair) / 4); i += TC_THREADS) dst[i] = src[i];
    }
    __syncthreads();
    const uint32_t tmem_base = tmem_base_s;

    // blockIdx.y = model x row split: model m reduces its rows [m Bm, m Bm + B) in the splits of a single-model call, into its own partials
    const int mdl = blockIdx.y / n_splits, sp = blockIdx.y - mdl * n_splits;
    const int64_t r_first = (int64_t)mdl * Bm;
    const int64_t r_begin = r_first + (int64_t)sp * rows_per;
    const int64_t r_end = (r_begin + rows_per < r_first + B) ? (r_begin + rows_per) : r_first + B;
    const int n_kb = r_end > r_begin ? (int)((r_end - r_begin + DW_KB - 1) / DW_KB) : 0;
    const int n_pairs = t.n_pairs < DW_MAX_PAIRS ? t.n_pairs : DW_MAX_PAIRS;
    const int n_steps = n_kb * n_pairs;
    const int want_cs = t.want_colsum;

    if (warp == 0) {
        if (lane == 0) {
            const uint32_t tx_bytes = split ? 4 * DW_IMG_BYTES : 2 * DW_IMG_BYTES;
            for (int i = 0; i < n_steps; ++i) {
                const int s = i % DW_STAGES;
                mbar_wait(empty0 + 8 * s, ((i / DW_STAGES) & 1) ^ 1);
                const RPair& pr = prs[i / n_kb];
                const int r0 = (int)(r_begin + (int64_t)(i % n_kb) * DW_KB);
                const int d_off = (int)((int64_t)pr.d_slot * Bp) + r0, a_off = (int)((int64_t)pr.a_slot * Bp) + r0;
                const uint32_t st = smem_base + s * DW_STAGE_BYTES;
                const uint32_t fb = full0 + 8 * s;
                mbar_expect_tx(fb, tx_bytes);
                tma_load_2d(st, &map, fb, 0, br.hi[pr.d_buf] + d_off);
                tma_load_2d(st + DW_IMG_BYTES / 2, &map, fb, 64, br.hi[pr.d_buf] + d_off);
                tma_load_2d(st + 2 * DW_IMG_BYTES, &map, fb, 0, br.hi[pr.a_buf] + a_off);
                tma_load_2d(st + 2 * DW_IMG_BYTES + DW_IMG_BYTES / 2, &map, fb, 64, br.hi[pr.a_buf] + a_off);
                if (split) {
                    tma_load_2d(st + DW_IMG_BYTES, &map, fb, 0, br.lo[pr.d_buf] + d_off);
                    tma_load_2d(st + DW_IMG_BYTES + DW_IMG_BYTES / 2, &map, fb, 64, br.lo[pr.d_buf] + d_off);
                    tma_load_2d(st + 3 * DW_IMG_BYTES, &map, fb, 0, br.lo[pr.a_buf] + a_off);
                    tma_load_2d(st + 3 * DW_IMG_BYTES + DW_IMG_BYTES / 2, &map, fb, 64, br.lo[pr.a_buf] + a_off);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint64_t ones_desc = smem_desc_sw128(smem_u32(ones));
            for (int i = 0; i < n_steps; ++i) {
                const int s = i % DW_STAGES;
                mbar_wait(full0 + 8 * s, (i / DW_STAGES) & 1);
                tc_fence_after();
                const uint32_t st = smem_base + s * DW_STAGE_BYTES;
                const uint64_t d_hi = smem_desc_mn_sw128(st), d_lo = smem_desc_mn_sw128(st + DW_IMG_BYTES);
                const uint64_t a_hi = smem_desc_mn_sw128(st + 2 * DW_IMG_BYTES), a_lo = smem_desc_mn_sw128(st + 3 * DW_IMG_BYTES);
#pragma unroll
                for (int ks = 0; ks < DW_KB / 16; ++ks) {
                    const uint64_t adv = (uint64_t)(ks * (2048 >> 4));          // 16 rows = two 8-row groups of 1024 B
                    const uint32_t acc = (i | ks) ? 1u : 0u;
                    umma_f16(tmem_base, d_hi + adv, a_hi + adv, DW_IDESC, acc);                       // D0 += dC_hi^T A_hi
                    if (split) {
                        umma_f16(tmem_base, d_lo + adv, a_hi + adv, DW_IDESC, 1u);                    // D0 += dC_lo^T A_hi
                        umma_f16(tmem_base, d_hi + adv, a_lo + adv, DW_IDESC, 1u);                    // D0 += dC_hi^T A_lo
                    }
                    if (want_cs) {
                        umma_f16(tmem_base + 128, d_hi + adv, ones_desc, DW_IDESC_CS, acc);           // D2 += dC_hi^T 1
                        if (split) umma_f16(tmem_base + 128, d_lo + adv, ones_desc, DW_IDESC_CS, 1u); // D2 += dC_lo^T 1
                    }
                }
                umma_commit(empty0 + 8 * s);
            }
            umma_commit(accum_bar);
        }
        __syncwarp();
    } else {
        // ---------------- epilogue: one thread per output feature (TMEM lane) ----------------
        mbar_wait(accum_bar, 0);
        tc_fence_after();
        const int q = warp & 3;
        const int o = q * 32 + lane;
        const int64_t slot = mdl * part_slots + slot0 + (int64_t)blockIdx.x * n_splits + sp;
        float* pw = part_w + slot * (H * H) + (int64_t)o * H;
#pragma unroll 1
        for (int cc = 0; cc < 4; ++cc) {
            uint32_t raw[32];
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + cc * 32, raw);
            tmem_ld_wait();
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = n_steps ? __uint_as_float(raw[j]) : 0.f;
            float4* dst = reinterpret_cast<float4*>(pw + cc * 32);
#pragma unroll
            for (int j = 0; j < 8; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        }
        if (want_cs) {
            uint32_t raw[32];
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + 128, raw);
            tmem_ld_wait();
            part_b[slot * H + o] = n_steps ? __uint_as_float(raw[0]) : 0.f;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, DW_TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------
// encoder on tcgen05:  h0[slot] = relu((x[slot] * sign[slot]) W_enc[type]^T + b)          (hgnn_k4.py:L159-160, L198-237)
// ------------------------------------------------------------------------------------------
//  The caller's fp32 (or fp64) feature rows are the only HBM stream of the whole model.  Eight loader warps read them
//  with 128-bit coalesced loads (all loads of a K block are issued before the first one is consumed, and the next block
//  of the group is already in flight while the current one is converted), fold the +-1 symmetry signs in, split every
//  value into the (hi, lo) fp16 pair and write it straight into the 128B-swizzled K-major UMMA operand layout in shared
//  memory; the weight tiles come by TMA from the padded fp16 weight image [n_types*128][enc_kmax].  Two loader groups
//  alternate K blocks.  warp roles: 0 = TMA (weights), 1 = MMA issuer, 2..9 = loaders, 2..5 = epilogue.
constexpr int ENC_THREADS = 320;
constexpr int ENC_LOADER_WARPS = 4;               // per group
constexpr int ENC_STAGES = 3;
constexpr int ENC_SETS = 3;                       // rotating register sets of the loaders (a fourth one spills at 168 registers and measured slower)
constexpr int ENC_TILE_BYTES = 128 * 128;         // 128 rows x 64 fp16 (one 128B-swizzled K block)
constexpr int ENC_STAGE_BYTES = 4 * ENC_TILE_BYTES;   // A_hi, A_lo, W_hi, W_lo = 64 KB
constexpr int ENC_SMEM_BYTES = ENC_STAGES * ENC_STAGE_BYTES + 1024 + 256;

struct alignas(64) EncMaps {
    CUtensorMap w_hi, w_lo;      // encoder weight images, box 64 x 128, SWIZZLE_128B
    CUtensorMap o;               // workspace images, box 64 x 128, SWIZZLE_128B (epilogue stores)
};


// 4 consecutive values of one row, times their column factors f (+-1 sign, 0 outside [0, K)) -> 8 bytes in the hi tile
// and 8 bytes in the lo tile.  hi = fp16(v f), lo = fp16((v f - hi) * 2^11) with packed conversions: 18 ALU ops per 4 values.
__device__ __forceinline__ void split_to_smem(uint32_t hi_addr, uint32_t lo_addr, const float4 v, const float4 f) {
    const float ax = v.x * f.x, ay = v.y * f.y, az = v.z * f.z, aw = v.w * f.w;
    const __half2 h01 = __floats2half2_rn(ax, ay), h23 = __floats2half2_rn(az, aw);
    const float2 g01 = __half22float2(h01), g23 = __half22float2(h23);
    const __half2 l01 = __floats2half2_rn((ax - g01.x) * TC_LO_SCALE, (ay - g01.y) * TC_LO_SCALE);
    const __half2 l23 = __floats2half2_rn((az - g23.x) * TC_LO_SCALE, (aw - g23.y) * TC_LO_SCALE);
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(hi_addr), "r"(*reinterpret_cast<const uint32_t*>(&h01)), "r"(*reinterpret_cast<const uint32_t*>(&h23)) : "memory");
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(lo_addr), "r"(*reinterpret_cast<const uint32_t*>(&l01)), "r"(*reinterpret_cast<const uint32_t*>(&l23)) : "memory");
}

// How the rows of one node of one type are addressed inside the caller's x tensor [B * nodes, K] (row-major).
struct XRows {
    const void* base;
    int64_t lda;          // elements between the same node of consecutive graphs
    int a_off;            // element offset of the node inside a graph's block
    int K;
    int f64;              // element type: 0 fp32, 1 fp64, 2 fp16 (kernels_simt.cuh: ld_x)
    int vec;              // widest aligned vector: fp32 / fp16 4 / 2 / 1 elements, fp64 2 / 1 elements
};
__device__ __forceinline__ XRows make_xrows(const void* base, int f64, int64_t lda, int a_off, int K) {
    XRows x;
    x.base = base; x.lda = lda; x.a_off = a_off; x.K = K; x.f64 = f64;
    const uintptr_t p = reinterpret_cast<uintptr_t>(base);
    const bool even = ((lda | a_off | K) & 1) == 0, quad = ((lda | a_off | K) & 3) == 0;
    if (f64 == 1) x.vec = (even && (p & 15) == 0) ? 2 : 1;
    else if (f64 == 2) x.vec = (quad && (p & 7) == 0) ? 4 : ((even && (p & 3) == 0) ? 2 : 1);
    else x.vec = (quad && (p & 15) == 0) ? 4 : ((even && (p & 7) == 0) ? 2 : 1);
    return x;
}

// Column factors of the 4 values a thread handles in a K block: the +-1 symmetry sign, 0 outside [0, K).
__device__ __forceinline__ float4 x_factors(const float* __restrict__ signs, const int sign_off, const int k, const int K) {
    float4 f;
    f.x = k < K ? 1.f : 0.f; f.y = k + 1 < K ? 1.f : 0.f; f.z = k + 2 < K ? 1.f : 0.f; f.w = k + 3 < K ? 1.f : 0.f;
    if (sign_off >= 0) {
        const float* sp = signs + sign_off;
        const int kc = k < K ? k : 0;
        f.x *= __ldg(sp + kc); f.y *= __ldg(sp + min(kc + 1, K - 1)); f.z *= __ldg(sp + min(kc + 2, K - 1)); f.w *= __ldg(sp + min(kc + 3, K - 1));
    }
    return f;
}

// The same factors from a per-CTA shared-memory table (fac[k] = sign or 0, staged once in the prologue).  Used by the encoder
// weight gradient, whose CTAs loop over many row blocks (-5 %).  The forward kernels keep x_factors(): there the staging is a
// dependent global round trip in front of every (short-lived) CTA and measured 15 % slower.
__device__ __forceinline__ float4 col_factors(const uint32_t fac_addr, const float* __restrict__ signs, const int sign_off, const int k, const int K) {
    if (!fac_addr) return x_factors(signs, sign_off, k, K);
    float4 f;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(f.x), "=f"(f.y), "=f"(f.z), "=f"(f.w) : "r"(fac_addr + 4u * (uint32_t)k));
    return f;
}
// fac[k] for k in [0, n_cols): +-1 symmetry sign (1 without a sign vector) for k < K, 0 beyond
__device__ __forceinline__ void stage_factors(float* fac, const float* __restrict__ signs, const int sign_off, const int k0, const int K,
                                              const int n_cols, const int tid, const int n_threads) {
    for (int c = tid; c < n_cols; c += n_threads) {
        const int k = k0 + c;
        fac[c] = k < K ? (sign_off >= 0 ? __ldg(signs + sign_off + k) : 1.f) : 0.f;
    }
}

// v[it] = x[min(row_first + RS*it, row_last)][k .. k+3] (columns clamped into [0, K)).  Every load is issued unconditionally
// on a clamped (always valid) address, so all N loads are in flight together; columns outside [0, K) are zeroed later by
// their factor, rows beyond the batch alias the last row and only ever meet zero partners (dead accumulator rows in
// the forward pass, zero dC rows in the weight gradient).
template <int N, int RS = 8>
__device__ __forceinline__ void load_x_block(float4 (&v)[N], const XRows& x, const int64_t row_first, const int64_t row_last, const int k) {
    const int K = x.K;
    const int kc = k < K ? k : 0;
    const int c1 = min(kc + 1, K - 1), c2 = min(kc + 2, K - 1), c3 = min(kc + 3, K - 1);
    if (x.f64 == 2) {
        // fp16 features (MSHGNN_F16): 8-byte loads of four halves; the split to (hi, lo) images downstream is then exact (lo = 0)
        const __half* b = (const __half*)x.base + x.a_off;
        if (x.vec == 4) {
#pragma unroll
            for (int it = 0; it < N; ++it) {
                const int64_t r = min(row_first + it * RS, row_last);
                const uint2 q = __ldg(reinterpret_cast<const uint2*>(b + r * x.lda + kc));
                const float2 lo2 = __half22float2(*reinterpret_cast<const __half2*>(&q.x)), hi2 = __half22float2(*reinterpret_cast<const __half2*>(&q.y));
                v[it] = make_float4(lo2.x, lo2.y, hi2.x, hi2.y);
            }
        } else if (x.vec == 2) {
            const int kd = min(kc + 2, K - 2);
#pragma unroll
            for (int it = 0; it < N; ++it) {
                const int64_t r = min(row_first + it * RS, row_last);
                const float2 p = __half22float2(__ldg(reinterpret_cast<const __half2*>(b + r * x.lda + kc)));
                const float2 q = __half22float2(__ldg(reinterpret_cast<const __half2*>(b + r * x.lda + kd)));
                v[it] = make_float4(p.x, p.y, q.x, q.y);
            }
        } else {
#pragma unroll
            for (int it = 0; it < N; ++it) {
                const __half* pr = b + min(row_first + it * RS, row_last) * x.lda;
                v[it] = make_float4(__half2float(__ldg(pr + kc)), __half2float(__ldg(pr + c1)), __half2float(__ldg(pr + c2)), __half2float(__ldg(pr + c3)));
            }
        }
    } else if (!x.f64) {
        const float* b = (const float*)x.base + x.a_off;
        if (x.vec == 4) {
#pragma unroll
            for (int it = 0; it < N; ++it) {
                const int64_t r = min(row_first + it * RS, row_last);
                v[it] = __ldg(reinterpret_cast<const float4*>(b + r * x.lda + kc));
            }
        } else if (x.vec == 2) {
            const int kd = min(kc + 2, K - 2);
#pragma unroll
            for (int it = 0; it < N; ++it) {
                const int64_t r = min(row_first + it * RS, row_last);
                const float2 p = __ldg(reinterpret_cast<const float2*>(b + r * x.lda + kc));
                const float2 q = __ldg(reinterpret_cast<const float2*>(b + r * x.lda + kd));
                v[it] = make_float4(p.x, p.y, q.x, q.y);
            }
        } else {
#pragma unroll
            for (int it = 0; it < N; ++it) {
                const float* pr = b + min(row_first + it * RS, row_last) * x.lda;
                v[it] = make_float4(__ldg(pr + kc), __ldg(pr + c1), __ldg(pr + c2), __ldg(pr + c3));
            }
        }
    } else {
        const double* b = (const double*)x.base + x.a_off;
        if (x.vec == 2) {
            const int kd = min(kc + 2, K - 2);
#pragma unroll
            for (int it = 0; it < N; ++it) {
                const int64_t r = min(row_first + it * RS, row_last);
                const double2 p = __ldg(reinterpret_cast<const double2*>(b + r * x.lda + kc));
                const double2 q = __ldg(reinterpret_cast<const double2*>(b + r * x.lda + kd));
                v[it] = make_float4((float)p.x, (float)p.y, (float)q.x, (float)q.y);
            }
        } else {
#pragma unroll
            for (int it = 0; it < N; ++it) {
                const double* pr = b + min(row_first + it * RS, row_last) * x.lda;
                v[it] = make_float4((float)__ldg(pr + kc), (float)__ldg(pr + c1), (float)__ldg(pr + c2), (float)__ldg(pr + c3));
            }
        }
    }
}

__device__ __forceinline__ int kb_count(const int g, const int n_kb) { return n_kb > g ? (n_kb - g + 1) / 2 : 0; }   // K blocks g, g+2, ...

__global__ void __launch_bounds__(ENC_THREADS, 1)
k_tc_encoder(const __grid_constant__ EncMaps maps, const Tile* __restrict__ tiles, const BufTable bt, const BufRows br,
             const int64_t B, const int64_t Bp, const int x_f64, const int split) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ Tile t;
    __shared__ __align__(16) float bias_s[H];
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + ENC_STAGES * ENC_STAGE_BYTES);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + ENC_STAGES), accum_bar = smem_u32(bars + 2 * ENC_STAGES),
                   res_bar = smem_u32(bars + 2 * ENC_STAGES + 1);
    const uint32_t smem_base = smem_u32(smem);
    {
        const int* src = reinterpret_cast<const int*>(tiles + blockIdx.y);
        int* dst = reinterpret_cast<int*>(&t);
        for (int i = tid; i < (int)(sizeof(Tile) / 4); i += ENC_THREADS) dst[i] = src[i];
    }
    if (tid == 0) {
        for (int s = 0; s < ENC_STAGES; ++s) { mbar_init(full0 + 8 * s, 1 + ENC_LOADER_WARPS); mbar_init(empty0 + 8 * s, 1); }
        mbar_init(accum_bar, 1);
        mbar_init(res_bar, 1);
        mbar_init(res_bar + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(&tmem_base_s), TC_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    const int row0 = blockIdx.x * TILE_M;
    const int K = t.chunks[0].K;
    const int n_kb = (K + 63) / 64;

    if (warp == 0) {
        if (lane == 0) {
            const uint32_t tx_bytes = split ? 2 * ENC_TILE_BYTES : ENC_TILE_BYTES;
            const int wrow = t.chunks[0].w16_row;
            for (int i = 0; i < n_kb; ++i) {
                const int s = i % ENC_STAGES;
                mbar_wait(empty0 + 8 * s, ((i / ENC_STAGES) & 1) ^ 1);
                const uint32_t st = smem_base + s * ENC_STAGE_BYTES;
                const uint32_t fb = full0 + 8 * s;
                mbar_expect_tx(fb, tx_bytes);
                tma_load_2d(st + 2 * ENC_TILE_BYTES, &maps.w_hi, fb, i * 64, wrow);
                if (split) tma_load_2d(st + 3 * ENC_TILE_BYTES, &maps.w_lo, fb, i * 64, wrow);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            for (int i = 0; i < n_kb; ++i) {
                const int s = i % ENC_STAGES;
                mbar_wait(full0 + 8 * s, (i / ENC_STAGES) & 1);
                tc_fence_after();
                const uint32_t st = smem_base + s * ENC_STAGE_BYTES;
                const uint64_t a_hi = smem_desc_sw128(st), a_lo = smem_desc_sw128(st + ENC_TILE_BYTES);
                const uint64_t w_hi = smem_desc_sw128(st + 2 * ENC_TILE_BYTES), w_lo = smem_desc_sw128(st + 3 * ENC_TILE_BYTES);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    const uint64_t adv = (uint64_t)(ks * 2);
                    umma_f16(tmem_base, a_hi + adv, w_hi + adv, TC_IDESC, (i | ks) ? 1u : 0u);
                    if (split) {
                        umma_f16(tmem_base, a_lo + adv, w_hi + adv, TC_IDESC, 1u);
                        umma_f16(tmem_base, a_hi + adv, w_lo + adv, TC_IDESC, 1u);
                    }
                }
                umma_commit(empty0 + 8 * s);
            }
            umma_commit(accum_bar);
        }
        __syncwarp();
    } else {
        // ---------------- loaders: group g takes the K blocks kb = g (mod 2) ----------------
        const int g = (warp - 2) / ENC_LOADER_WARPS;
        const int gt = tid - 64 - g * (ENC_LOADER_WARPS * 32);
        const Chunk& ch = t.chunks[0];
        const XRows xr = make_xrows(bt.p[ch.a_buf], x_f64, ch.lda, ch.a_off, K);
        const float* signs = (const float*)bt.p[2];
        const int kq = gt & 15;                                   // which 4-column group of the 64-column block
        const int rsub = gt >> 4;                                 // 0..7
        const int64_t row_first = (int64_t)row0 + rsub;
        // Work units of 64 rows x 64 columns (half a K block); ENC_SETS register sets rotate so that the loads of units
        // n + 1 .. n + ENC_SETS - 1 are in flight while unit n is converted and written to shared memory.
        const int n_units = kb_count(g, n_kb) * 2;
        float4 v[ENC_SETS][8];
        auto load = [&](float4 (&v)[8], const int n) {
            if (n < n_units) load_x_block<8>(v, xr, row_first + (n & 1) * 64, B - 1, (g + 2 * (n >> 1)) * 64 + kq * 4);
        };
        auto convert = [&](const float4 (&v)[8], const int n) {
            if (n >= n_units) return;
            const int kb = g + 2 * (n >> 1), half = n & 1;
            const float4 f = x_factors(signs, ch.sign_off, kb * 64 + kq * 4, K);
            const int s = kb % ENC_STAGES;
            if (!half) mbar_wait(empty0 + 8 * s, ((kb / ENC_STAGES) & 1) ^ 1);
            const uint32_t st = smem_base + s * ENC_STAGE_BYTES;
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int r = half * 64 + it * 8 + rsub;
                const uint32_t off = (uint32_t)(r * 128 + ((((kq >> 1) ^ (r & 7))) << 4) + ((kq & 1) << 3));
                split_to_smem(st + off, st + ENC_TILE_BYTES + off, v[it], f);
            }
            if (half) {
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(full0 + 8 * s);
            }
        };
#pragma unroll
        for (int j = 0; j < ENC_SETS - 1; ++j) load(v[j], j);
        for (int n = 0; n < n_units; n += ENC_SETS) {
#pragma unroll
            for (int j = 0; j < ENC_SETS; ++j) {
                load(v[(j + ENC_SETS - 1) % ENC_SETS], n + j + ENC_SETS - 1);
                convert(v[j], n + j);
            }
        }
        {
            // ---------------- epilogue: warps 2..5 take columns 0..63, warps 6..9 columns 64..127 ----------------
            EpiSmem es;
            es.stg = smem_base; es.bias = smem_u32(bias_s); es.res_bar = res_bar; es.accum_bar = accum_bar;
            es.free_bar = 0; es.acc_parity = 0; es.res_parity = 0; es.persistent = 0; es.n_groups = 2;
            tc_epilogue(t, bt, br, &maps.o, tmem_base, row0, B, Bp, split, warp, lane, es);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TC_TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------
// encoder, two row tiles per CTA (model batches, inputs the persistent kernel cannot read, option "encoder" = 2)
// ------------------------------------------------------------------------------------------
//  ncu of k_tc_encoder: 46.7 M L2->SM read sectors (1.49 GB) for 708 MB of features - a 128-row x 64-column fp32 block
//  of x is 32 KB and so is the (hi, lo) weight K block it meets, i.e. every CTA pulls as many weight bytes out of L2 as
//  feature bytes.  Here a CTA owns TWO row tiles (256 graphs of one node slot): every weight stage is used by both, the
//  weight stream halves (L2->SM bytes -25 %) and the fixed per-CTA cost is paid once per 256 rows.  Measured on one box,
//  alternating runs: 0.359-0.365 ms against 0.372-0.378 ms for k_tc_encoder (DESIGN 3.1a lists what did NOT help: two
//  CTAs per SM, a fourth register set, staged or prefetched sign factors - the kernel is bound by the latency of the
//  strided 256-byte row fragments, not by L2 bytes, issue slots or per-CTA overhead).
//  Stage = A0_hi, A0_lo, A1_hi, A1_lo, W_hi, W_lo = 96 KB, two stages (loader group g fills row tile g), accumulators of the
//  two tiles in TMEM columns [0,128) and [128,256); the epilogue drains them one after the other through the drained ring.
constexpr int ENCP_STAGES = 2;
constexpr int ENCP_STAGE_BYTES = 6 * ENC_TILE_BYTES;          // 96 KB
constexpr int ENCP_SMEM_BYTES = ENCP_STAGES * ENCP_STAGE_BYTES + 1024 + 256;
constexpr uint32_t ENCP_TMEM_COLS = 256;
constexpr int ENC_PF_BYTES = 1536;                      // first L2 prefetch request per feature row

__global__ void __launch_bounds__(ENC_THREADS, 1)
k_tc_encoder_pair(const __grid_constant__ EncMaps maps, const Tile* __restrict__ tiles, const BufTable bt, const BufRows br,
                  const int64_t B, const int64_t Bp, const int x_f64, const int split, const int enc_prefetch, const int64_t Bm,
                  const int enc_rows /*weight-image rows of one model*/, const int64_t n_params) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ Tile t;
    __shared__ __align__(16) float bias_s[H];
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + ENCP_STAGES * ENCP_STAGE_BYTES);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + ENCP_STAGES), accum_bar = smem_u32(bars + 2 * ENCP_STAGES),
                   res_bar = smem_u32(bars + 2 * ENCP_STAGES + 1);
    const uint32_t smem_base = smem_u32(smem);
    // model of a model batch: blockIdx.x walks the row-tile pairs of model 0's block [0, Bm), then model 1's, ...  Its tile reads
    // that model's weight-image rows and bias; its graphs are rows [mdl B, mdl B + B) of the caller's feature tensors.
    const int pairs_m = (int)((Bm / TILE_M + 1) / 2);
    const int mdl = blockIdx.x / pairs_m;
    const int64_t m_row0 = (int64_t)mdl * Bm;
    {
        const int* src = reinterpret_cast<const int*>(tiles + blockIdx.y);
        int* dst = reinterpret_cast<int*>(&t);
        for (int i = tid; i < (int)(sizeof(Tile) / 4); i += ENC_THREADS)
            dst[i] = src[i] + (i == (int)(offsetof(Tile, bias_off) / 4) ? mdl * (int)n_params : 0)
                            + (i == (int)((offsetof(Tile, chunks) + offsetof(Chunk, w16_row)) / 4) ? mdl * enc_rows : 0);
    }
    const int row0 = (int)(m_row0 + (int64_t)(blockIdx.x - mdl * pairs_m) * (2 * TILE_M));
    const int n_tiles = (int64_t)row0 + TILE_M < m_row0 + Bm ? 2 : 1;     // Bm is a multiple of 128, not of 256
    const int64_t B_end = m_row0 + B;                                    // rows [B_end, m_row0 + Bm) are padding
    if (tid == 0) {
        // a stage is full when the weight TMA and the four loader warps of every live row tile have arrived
        for (int s = 0; s < ENCP_STAGES; ++s) { mbar_init(full0 + 8 * s, 1 + ENC_LOADER_WARPS * n_tiles); mbar_init(empty0 + 8 * s, 1); }
        mbar_init(accum_bar, 1);
        mbar_init(res_bar, 1);
        mbar_init(res_bar + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(&tmem_base_s), ENCP_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    const int K = t.chunks[0].K;
    const int n_kb = (K + 63) / 64;

    if (warp == 0) {
        // Optional (enc_prefetch; the host passes 0) L2 prefetch of this CTA's feature rows as WHOLE-ROW bulk requests (one per
        // graph row, up to 1.5 KB at a time).  Hypothesis tested in round 2: the loaders read the rows as 256-byte fragments, 14 KB
        // apart, K block by K block, and DRAM serves that pattern badly (the weight-gradient kernel reads the same rows in 768-byte
        // fragments at 3.8 TB/s).  Measured: 0.346 -> 0.388 ms, i.e. WORSE - fragment size is not what limits this kernel.
        const Chunk& ch0 = t.chunks[0];
        const bool pf_ok = enc_prefetch && !x_f64 && ((ch0.lda | ch0.a_off | K) & 3) == 0 && (reinterpret_cast<uintptr_t>(bt.p[ch0.a_buf]) & 15) == 0;
        const float* xb = (const float*)bt.p[ch0.a_buf] + ch0.a_off;
        const int row_bytes = K * 4;
        auto prefetch_rows = [&](const int byte0, const int byte1, const int l0, const int lstep) {
            if (byte1 <= byte0) return;
            for (int r = l0; r < n_tiles * TILE_M; r += lstep) {
                const int64_t row = (int64_t)row0 + r;
                if (row >= B_end) break;
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(reinterpret_cast<const char*>(xb + (row - m_row0 + mdl * B) * ch0.lda) + byte0), "r"(byte1 - byte0) : "memory");
            }
        };
        if (pf_ok) prefetch_rows(0, row_bytes < ENC_PF_BYTES ? row_bytes : ENC_PF_BYTES, lane, 32);
        if (lane == 0) {
            const uint32_t tx_bytes = split ? 2 * ENC_TILE_BYTES : ENC_TILE_BYTES;
            const int wrow = t.chunks[0].w16_row;
            for (int i = 0; i < n_kb; ++i) {
                const int s = i % ENCP_STAGES;
                mbar_wait(empty0 + 8 * s, ((i / ENCP_STAGES) & 1) ^ 1);
                const uint32_t st = smem_base + s * ENCP_STAGE_BYTES;
                const uint32_t fb = full0 + 8 * s;
                mbar_expect_tx(fb, tx_bytes);
                tma_load_2d(st + 4 * ENC_TILE_BYTES, &maps.w_hi, fb, i * 64, wrow);
                if (split) tma_load_2d(st + 5 * ENC_TILE_BYTES, &maps.w_lo, fb, i * 64, wrow);
                if (i == 1 && pf_ok) prefetch_rows(ENC_PF_BYTES, row_bytes, 0, 1);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            for (int i = 0; i < n_kb; ++i) {
                const int s = i % ENCP_STAGES;
                mbar_wait(full0 + 8 * s, (i / ENCP_STAGES) & 1);
                tc_fence_after();
                const uint32_t st = smem_base + s * ENCP_STAGE_BYTES;
                const uint64_t w_hi = smem_desc_sw128(st + 4 * ENC_TILE_BYTES), w_lo = smem_desc_sw128(st + 5 * ENC_TILE_BYTES);
                for (int tl = 0; tl < n_tiles; ++tl) {
                    const uint64_t a_hi = smem_desc_sw128(st + (2 * tl) * ENC_TILE_BYTES), a_lo = smem_desc_sw128(st + (2 * tl + 1) * ENC_TILE_BYTES);
                    const uint32_t acc = tmem_base + (uint32_t)tl * 128u;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint64_t adv = (uint64_t)(ks * 2);
                        umma_f16(acc, a_hi + adv, w_hi + adv, TC_IDESC, (i | ks) ? 1u : 0u);
                        if (split) {
                            umma_f16(acc, a_lo + adv, w_hi + adv, TC_IDESC, 1u);
                            umma_f16(acc, a_hi + adv, w_lo + adv, TC_IDESC, 1u);
                        }
                    }
                }
                umma_commit(empty0 + 8 * s);
            }
            umma_commit(accum_bar);
        }
        __syncwarp();
    } else {
        // ---------------- loaders: group g fills row tile g of EVERY K block; stages alternate ----------------
        //  (with the K blocks split between the groups a group always refilled the stage the MMA warp was still reading:
        //  6.5 % of the warp samples sat in that empty-barrier wait; now both groups write stage kb + 1 while stage kb is consumed)
        const int g = (warp - 2) / ENC_LOADER_WARPS;
        const int gt = tid - 64 - g * (ENC_LOADER_WARPS * 32);
        const Chunk& ch = t.chunks[0];
        // workspace row r of this model is the caller's graph r - mdl (Bm - B): shift the base by that many graphs
        const int esz = x_f64 == 1 ? 8 : (x_f64 == 2 ? 2 : 4);
        const XRows xr = make_xrows((const char*)bt.p[ch.a_buf] - (int64_t)mdl * (Bm - B) * ch.lda * esz, x_f64, ch.lda, ch.a_off, K);
        const float* signs = (const float*)bt.p[2];
        const int kq = gt & 15;                                   // which 4-column group of the 64-column block
        const int rsub = gt >> 4;                                 // 0..7
        const int64_t row_first = (int64_t)row0 + g * TILE_M + rsub;
        // Work units of 64 rows x 64 columns (half a K block of this group's row tile); ENC_SETS register sets rotate so that
        // the loads of units n + 1 .. n + ENC_SETS - 1 are in flight while unit n is converted and written to shared memory.
        const int n_units = g < n_tiles ? n_kb * 2 : 0;
        float4 v[ENC_SETS][8];
        auto load = [&](float4 (&v)[8], const int n) {
            if (n < n_units) load_x_block<8>(v, xr, row_first + (n & 1) * 64, B_end - 1, (n >> 1) * 64 + kq * 4);
        };
        auto convert = [&](const float4 (&v)[8], const int n) {
            if (n >= n_units) return;
            const int kb = n >> 1, half = n & 1;
            const float4 f = x_factors(signs, ch.sign_off, kb * 64 + kq * 4, K);
            const int s = kb % ENCP_STAGES;
            if (!half) mbar_wait(empty0 + 8 * s, ((kb / ENCP_STAGES) & 1) ^ 1);
            const uint32_t st = smem_base + s * ENCP_STAGE_BYTES + (uint32_t)g * (2 * ENC_TILE_BYTES);
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int r = half * 64 + it * 8 + rsub;
                const uint32_t off = (uint32_t)(r * 128 + ((((kq >> 1) ^ (r & 7))) << 4) + ((kq & 1) << 3));
                split_to_smem(st + off, st + ENC_TILE_BYTES + off, v[it], f);
            }
            if (half) {
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(full0 + 8 * s);
            }
        };
#pragma unroll
        for (int j = 0; j < ENC_SETS - 1; ++j) load(v[j], j);
        for (int n = 0; n < n_units; n += ENC_SETS) {
#pragma unroll
            for (int j = 0; j < ENC_SETS; ++j) {
                load(v[(j + ENC_SETS - 1) % ENC_SETS], n + j + ENC_SETS - 1);
                convert(v[j], n + j);
            }
        }
        // ---------------- epilogue: warps 2..5 take columns 0..63, warps 6..9 columns 64..127, tile after tile ----------------
        for (int tl = 0; tl < n_tiles; ++tl) {
            EpiSmem es;
            es.stg = smem_base + (uint32_t)tl * 65536u; es.bias = smem_u32(bias_s); es.res_bar = res_bar; es.accum_bar = accum_bar;
            es.free_bar = 0; es.acc_parity = 0; es.res_parity = 0; es.persistent = 0; es.n_groups = 2;
            tc_epilogue(t, bt, br, &maps.o, tmem_base + (uint32_t)tl * 128u, row0 + tl * TILE_M, B_end, Bp, split, warp, lane, es);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, ENCP_TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------
// encoder weight gradient on tcgen05:  dW_enc[t][:, k0 : k0+64*nkb] = sum_slots dpre[slot]^T (x[slot] * sign[slot])
// ------------------------------------------------------------------------------------------
//  M = 128 output features (dpre images, MN-major via TMA like k_tc_reducegemm), N = 64*nkb input columns (the loaders
//  write the split x rows as 64-column MN-major blocks, LBO = 8192 B), K = graph rows.  x is read exactly once per step
//  over all units.  Accumulators: D0 [0,192) hi*hi, D1 [192,384) cross (x 2^11), D2 [384,400) / D3 [416,432) bias sums.
// caller's feature tensors as (K, nodes, B) fp32 tensors, box 64 columns x 1 node x 64 graphs (no swizzle): one request lands the
// 256-byte fragments of a 64-column block of 64 consecutive graphs of one node slot (see kernels_enc.cuh for why the feature rows
// are kept off the register scoreboards)
struct alignas(64) EncXMaps {
    CUtensorMap x[4];
};
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

constexpr int EDW_STAGES = 2;
constexpr int EDW_DC_BYTES = DW_IMG_BYTES;                 // 64 rows x 128 features fp16
constexpr int EDW_X_BYTES = 3 * 64 * 128;                  // up to three 64-row x 64-column blocks
constexpr int EDW_STAGE_BYTES = 2 * EDW_DC_BYTES + 2 * EDW_X_BYTES;     // dC_hi, dC_lo, X_hi, X_lo = 80 KB
constexpr int EDW_SMEM_BYTES = EDW_STAGES * EDW_STAGE_BYTES + DW_ONES_BYTES + 1024 + 256;
constexpr int EDW_NMAX = 192;

//  XT = true (fp32 features with 16-byte rows): the x rows of a step arrive by TMA as raw fp32 in the X operand area of the stage
//  (64 rows x 64 columns x 4 B per block = the 16 KB its hi + lo images take) and the loader group converts them in place.
template <bool XT>
__global__ void __launch_bounds__(ENC_THREADS, 1)
k_tc_encoder_dw(const __grid_constant__ CUtensorMap map, const __grid_constant__ EncXMaps xmaps, const int x_buf0, const EncDwUnit* __restrict__ units,
                const BufTable bt, const BufRows br,
                const int64_t B, const int64_t Bp, const int rows_per, const int n_splits, const int x_f64, const int split,
                float* __restrict__ part_w, float* __restrict__ part_b, const int64_t Bm) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ EncDwUnit u;
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(16) float fac_s[4][EDW_NMAX];     // per-slot column factors of this unit's columns (see col_factors)

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* ones = smem + EDW_STAGES * EDW_STAGE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(ones + DW_ONES_BYTES);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + EDW_STAGES), accum_bar = smem_u32(bars + 2 * EDW_STAGES),
                   landed0 = smem_u32(bars + 2 * EDW_STAGES + 1);
    const uint32_t smem_base = smem_u32(smem);

    if (tid < (int)(sizeof(EncDwUnit) / 4)) reinterpret_cast<int*>(&u)[tid] = reinterpret_cast<const int*>(units + blockIdx.x)[tid];
    {
        const EncDwUnit* gu = units + blockIdx.x;
        const int g_slots = __ldg(&gu->n_slots), g_k0 = __ldg(&gu->k0), g_K = __ldg(&gu->K), g_cols = __ldg(&gu->nkb) * 64;
        for (int j = 0; j < g_slots; ++j) stage_factors(fac_s[j], (const float*)bt.p[2], __ldg(&gu->sign_off[j]), g_k0, g_K, g_cols, tid, ENC_THREADS);
    }
    for (int i = tid; i < DW_ONES_BYTES / 4; i += ENC_THREADS) reinterpret_cast<uint32_t*>(ones)[i] = 0x3C003C00u;
    fence_proxy_async_smem();
    if (tid == 0) {
        for (int s = 0; s < EDW_STAGES; ++s) { mbar_init(full0 + 8 * s, 1 + ENC_LOADER_WARPS); mbar_init(empty0 + 8 * s, 1); mbar_init(landed0 + 8 * s, 1); }
        mbar_init(accum_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(&tmem_base_s), DW_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    // blockIdx.y = model x row split (as in k_tc_reducegemm); partials of model m follow those of every unit of model m - 1
    const int mdl = blockIdx.y / n_splits, sp = blockIdx.y - mdl * n_splits;
    const int64_t r_first = (int64_t)mdl * Bm;
    const int64_t r_begin = r_first + (int64_t)sp * rows_per;
    const int64_t r_end = (r_begin + rows_per < r_first + B) ? (r_begin + rows_per) : r_first + B;
    const int n_rb = r_end > r_begin ? (int)((r_end - r_begin + DW_KB - 1) / DW_KB) : 0;
    const int n_steps = n_rb * u.n_slots;
    const int nkb = u.nkb;
    const int want_cs = u.want_colsum;
    const uint32_t idesc = (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(nkb * 64 >> 3) << 17) | ((128u >> 4) << 24);

    if (warp == 0) {
        if (lane == 0) {
            const uint32_t tx_bytes = split ? 2 * EDW_DC_BYTES : EDW_DC_BYTES;
            for (int i = 0; i < n_steps; ++i) {
                const int s = i % EDW_STAGES;
                mbar_wait(empty0 + 8 * s, ((i / EDW_STAGES) & 1) ^ 1);
                const int r0 = (int)(r_begin + (int64_t)(i % n_rb) * DW_KB);
                const int d_off = (int)((int64_t)u.d_slot[i / n_rb] * Bp) + r0;
                const uint32_t st = smem_base + s * EDW_STAGE_BYTES;
                const uint32_t fb = full0 + 8 * s;
                mbar_expect_tx(fb, tx_bytes);
                tma_load_2d(st, &map, fb, 0, br.hi[BUF_DC1_ID] + d_off);
                tma_load_2d(st + EDW_DC_BYTES / 2, &map, fb, 64, br.hi[BUF_DC1_ID] + d_off);
                if (split) {
                    tma_load_2d(st + EDW_DC_BYTES, &map, fb, 0, br.lo[BUF_DC1_ID] + d_off);
                    tma_load_2d(st + EDW_DC_BYTES + EDW_DC_BYTES / 2, &map, fb, 64, br.lo[BUF_DC1_ID] + d_off);
                }
                if (XT) {
                    // raw x rows of the step: graphs >= B and columns >= K arrive as zeros
                    const int j = i / n_rb;
                    const uint32_t lb = landed0 + 8 * s;
                    mbar_expect_tx(lb, (uint32_t)nkb * 16384u);
                    const CUtensorMap* xm = &xmaps.x[u.x_buf - x_buf0];
                    const int node = u.a_off[j] / u.K;
                    for (int jb = 0; jb < nkb; ++jb) tma_load_3d(st + 2 * EDW_DC_BYTES + jb * 16384, xm, lb, u.k0 + jb * 64, node, r0);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint64_t ones_desc = smem_desc_sw128(smem_u32(ones));
            for (int i = 0; i < n_steps; ++i) {
                const int s = i % EDW_STAGES;
                mbar_wait(full0 + 8 * s, (i / EDW_STAGES) & 1);
                tc_fence_after();
                const uint32_t st = smem_base + s * EDW_STAGE_BYTES;
                const uint64_t d_hi = smem_desc_mn_sw128(st), d_lo = smem_desc_mn_sw128(st + EDW_DC_BYTES);
                const uint64_t x_hi = smem_desc_mn_sw128(st + 2 * EDW_DC_BYTES), x_lo = smem_desc_mn_sw128(st + 2 * EDW_DC_BYTES + EDW_X_BYTES);
#pragma unroll
                for (int ks = 0; ks < DW_KB / 16; ++ks) {
                    const uint64_t adv = (uint64_t)(ks * (2048 >> 4));
                    const uint32_t acc = (i | ks) ? 1u : 0u;
                    umma_f16(tmem_base, d_hi + adv, x_hi + adv, idesc, acc);
                    if (split) {
                        umma_f16(tmem_base, d_lo + adv, x_hi + adv, idesc, 1u);
                        umma_f16(tmem_base, d_hi + adv, x_lo + adv, idesc, 1u);
                    }
                    if (want_cs) {
                        umma_f16(tmem_base + EDW_NMAX, d_hi + adv, ones_desc, DW_IDESC_CS, acc);
                        if (split) umma_f16(tmem_base + EDW_NMAX, d_lo + adv, ones_desc, DW_IDESC_CS, 1u);
                    }
                }
                umma_commit(empty0 + 8 * s);
            }
            umma_commit(accum_bar);
        }
        __syncwarp();
    } else {
        // ---------------- loaders: group g takes the steps i = g (mod 2) ----------------
        const int g = (warp - 2) / ENC_LOADER_WARPS;
        const int gt = tid - 64 - g * (ENC_LOADER_WARPS * 32);
        const float* signs = (const float*)bt.p[2];
        const int kq = gt & 15, rsub = gt >> 4;
        const int esz = x_f64 == 1 ? 8 : (x_f64 == 2 ? 2 : 4);
        const char* xbase = (const char*)bt.p[u.x_buf] - (int64_t)mdl * (Bm - B) * u.lda * esz;     // workspace row r -> caller's graph r - mdl (Bm - B)
        for (int i = g; i < n_steps; i += 2) {
            const int s = i % EDW_STAGES;
            const int j = i / n_rb;
            const XRows xr = make_xrows(xbase, x_f64, u.lda, u.a_off[j], u.K);
            const int64_t r0 = r_begin + (int64_t)(i % n_rb) * DW_KB + rsub;
            const uint32_t st = smem_base + s * EDW_STAGE_BYTES + 2 * EDW_DC_BYTES;
            float4 v[3][8];
            if (XT) {
                mbar_wait(landed0 + 8 * s, (i / EDW_STAGES) & 1);
#pragma unroll
                for (int jb = 0; jb < 3; ++jb)
                    if (jb < nkb) {
#pragma unroll
                        for (int it = 0; it < 8; ++it) {
                            const int r = it * 8 + rsub;
                            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[jb][it].x), "=f"(v[jb][it].y), "=f"(v[jb][it].z), "=f"(v[jb][it].w)
                                         : "r"(st + (uint32_t)(jb * 16384 + r * 256 + kq * 16)));
                        }
                    }
                asm volatile("bar.sync %0, 128;" ::"r"(2 + g) : "memory");       // every raw row of the step is in registers: the images may overwrite them
            } else {
#pragma unroll
                for (int jb = 0; jb < 3; ++jb)
                    if (jb < nkb) load_x_block<8>(v[jb], xr, r0, r_first + B - 1, u.k0 + jb * 64 + kq * 4);
                mbar_wait(empty0 + 8 * s, ((i / EDW_STAGES) & 1) ^ 1);
            }
#pragma unroll
            for (int jb = 0; jb < 3; ++jb)
                if (jb < nkb) {
                    const float4 f = col_factors(smem_u32(fac_s[j]), signs, u.sign_off[j], jb * 64 + kq * 4, u.K);
#pragma unroll
                    for (int it = 0; it < 8; ++it) {
                        const int r = it * 8 + rsub;
                        const uint32_t off = (uint32_t)(jb * 8192 + r * 128 + ((((kq >> 1) ^ (r & 7))) << 4) + ((kq & 1) << 3));
                        split_to_smem(st + off, st + EDW_X_BYTES + off, v[jb][it], f);
                    }
                }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(full0 + 8 * s);
        }
        if (warp < 6) {
            // ---------------- epilogue: one thread per output feature ----------------
            mbar_wait(accum_bar, 0);
            tc_fence_after();
            const int q = warp & 3;
            const int o = q * 32 + lane;
            const int64_t slot = ((int64_t)mdl * gridDim.x + blockIdx.x) * n_splits + sp;
            float* pw = part_w + slot * (H * EDW_NMAX) + (int64_t)o * EDW_NMAX;
            for (int cc = 0; cc < nkb * 2; ++cc) {
                uint32_t raw[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + cc * 32, raw);
                tmem_ld_wait();
                float4* dst = reinterpret_cast<float4*>(pw + cc * 32);
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                    float x[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        x[e] = n_steps ? __uint_as_float(raw[4 * jj + e]) : 0.f;
                    }
                    dst[jj] = make_float4(x[0], x[1], x[2], x[3]);
                }
            }
            if (want_cs) {
                uint32_t raw[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + EDW_NMAX, raw);
                tmem_ld_wait();
                part_b[slot * H + o] = n_steps ? __uint_as_float(raw[0]) : 0.f;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, DW_TMEM_COLS);
    }
}

// sum the encoder partials of one (type, 192-column range) group into the flat gradient buffer (fixed order, double)
__global__ void __launch_bounds__(256)
k_reduce_enc(const EncDwGroup* __restrict__ groups, const float* __restrict__ part_w, const float* __restrict__ part_b,
             const int n_splits, float* __restrict__ grads, const float rscale, const int n_units, const int64_t n_params) {
    const EncDwGroup g = groups[blockIdx.x];
    // blockIdx.z = model of a model batch
    part_w += (int64_t)blockIdx.z * n_units * n_splits * (H * EDW_NMAX);
    part_b += (int64_t)blockIdx.z * n_units * n_splits * H;
    grads += blockIdx.z * n_params;
    const int n = H * g.width;
    for (int e = blockIdx.y * 256 + threadIdx.x; e < n; e += gridDim.y * 256) {
        const int o = e / g.width, i = e % g.width;
        double sd = 0.0;
        const float* p = part_w + (int64_t)g.first * n_splits * (H * EDW_NMAX) + (int64_t)o * EDW_NMAX + i;
        const int n_part = g.count * n_splits;
        int us = 0;
        for (; us + 8 <= n_part; us += 8) {          // 8 independent loads in flight, summed in the fixed order
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = __ldg(p + (int64_t)(us + j) * (H * EDW_NMAX));
#pragma unroll
            for (int j = 0; j < 8; ++j) sd += (double)v[j];
        }
        for (; us < n_part; ++us) sd += (double)__ldg(p + (int64_t)us * (H * EDW_NMAX));
        grads[(int64_t)g.w_off + (int64_t)o * g.K + g.k0 + i] = (float)(sd * (double)rscale);
    }
    if (g.b_off >= 0 && blockIdx.y == 0)
        for (int o = threadIdx.x; o < H; o += 256) {
            double sd = 0.0;
            const float* p = part_b + (int64_t)g.first * n_splits * H + o;
            for (int us = 0; us < g.count * n_splits; ++us) sd += (double)p[(int64_t)us * H];
            grads[(int64_t)g.b_off + o] = (float)(sd * (double)rscale);
        }
}

// fp16 (hi, lo) image of the encoder weights: [n_types*128][kmax], zero padded beyond each type's in-width (blockIdx.y = type)
struct EncImgDesc {
    int n_types;
    int K[4];
    int64_t w_off[4];
};
__global__ void __launch_bounds__(256)
k_derive_enc16(const float* __restrict__ params, const EncImgDesc ed, const int kmax, __half* __restrict__ w_hi, __half* __restrict__ w_lo) {
    const int t = blockIdx.y, K = ed.K[t], row0 = t * H;
    const int64_t w_off = ed.w_off[t];
    for (int e = blockIdx.x * 256 + threadIdx.x; e < H * kmax; e += gridDim.x * 256) {
        const int o = e / kmax, k = e % kmax;
        const float s = k < K ? params[w_off + (int64_t)o * K + k] * TC_W_SCALE : 0.f;
        const __half h = __float2half_rn(s);
        w_hi[(int64_t)(row0 + o) * kmax + k] = h;
        w_lo[(int64_t)(row0 + o) * kmax + k] = __float2half_rn((s - __half2float(h)) * TC_LO_SCALE);
    }
}

// ------------------------------------------------------------------------------------------
// fp16 (hi, lo) images of the weights the tensor-core kernels read: W (forward) and W^T (backward dX)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_derive16(const Derive16Op* __restrict__ ops, const float* __restrict__ params, __half* __restrict__ w_hi, __half* __restrict__ w_lo) {
    const Derive16Op op = ops[blockIdx.y];
    for (int e = blockIdx.x * 256 + threadIdx.x; e < H * H; e += gridDim.x * 256) {
        const int r = e / H, c = e % H;
        const int src = op.transpose ? (c * H + r) : e;
        float s = 0.f;
        for (int i = 0; i < op.n_src; ++i) s += params[(int64_t)op.src_off[i] + src];
        s *= TC_W_SCALE;
        const __half h = __float2half_rn(s);
        w_hi[(int64_t)op.dst_row * H + e] = h;
        w_lo[(int64_t)op.dst_row * H + e] = __float2half_rn((s - __half2float(h)) * TC_LO_SCALE);
    }
}

// ------------------------------------------------------------------------------------------
// One launch for everything the tensor-core forward needs before its first GEMM (was k_derive + k_derive16 + k_derive_enc16 + a
// memset: four launches of 5-16 us each, a quarter of the fixed tail of a 2048-graph step): blocks [0, n_bias) the derived bias
// sums, [n_bias, + 8 n16) the (hi, lo) images of the 128x128 weights, [.., + 64 n_types) the encoder weight image, the rest zero the
// completion counters of the stack kernel.
// ------------------------------------------------------------------------------------------
struct FwdPrologue {
    const DeriveOp* ops; int n_bias;
    const Derive16Op* ops16; int n16;
    EncImgDesc ed; int kmax;
    uint32_t* zero; int64_t zero_words; int zero_blocks;
    uint32_t* enc_sync;          // work counter of k_tc_encoder_stream
    int64_t n_params, n_derived; // per-model strides of a model batch (blockIdx.y = model); the weight images of a model are n16 x 128
};                               // rows, its encoder images ed.n_types x 128 rows
__global__ void __launch_bounds__(256)
k_fwd_prologue(const FwdPrologue a, const float* __restrict__ params, float* __restrict__ derived, __half* __restrict__ w_hi, __half* __restrict__ w_lo,
               __half* __restrict__ e_hi, __half* __restrict__ e_lo) {
    int b = blockIdx.x;
    const int mdl = blockIdx.y;
    params += mdl * a.n_params;
    derived += mdl * a.n_derived;
    w_hi += (int64_t)mdl * a.n16 * H * H; w_lo += (int64_t)mdl * a.n16 * H * H;
    e_hi += (int64_t)mdl * a.ed.n_types * H * a.kmax; e_lo += (int64_t)mdl * a.ed.n_types * H * a.kmax;
    if (b == 0 && mdl == 0 && threadIdx.x == 0 && a.enc_sync) *a.enc_sync = 0u;
    if (b < a.n_bias) {
        const DeriveOp op = a.ops[b];
        const int n = op.rows * op.cols;
        for (int e = threadIdx.x; e < n; e += 256) {
            int r, c;
            if (op.transpose) { c = e / op.rows; r = e % op.rows; } else { r = e / op.cols; c = e % op.cols; }
            float s = 0.f;
            for (int i = 0; i < op.n_src; ++i) s += params[(int64_t)op.src_off[i] + (int64_t)r * op.cols + c];
            derived[(int64_t)op.dst_off + e] = s;
        }
        return;
    }
    b -= a.n_bias;
    if (b < 8 * a.n16) {
        const Derive16Op op = a.ops16[b >> 3];
        for (int e = (b & 7) * 256 + threadIdx.x; e < H * H; e += 8 * 256) {
            const int r = e / H, c = e % H;
            const int src = op.transpose ? (c * H + r) : e;
            float s = 0.f;
            for (int i = 0; i < op.n_src; ++i) s += params[(int64_t)op.src_off[i] + src];
            s *= TC_W_SCALE;
            const __half h = __float2half_rn(s);
            w_hi[(int64_t)op.dst_row * H + e] = h;
            w_lo[(int64_t)op.dst_row * H + e] = __float2half_rn((s - __half2float(h)) * TC_LO_SCALE);
        }
        return;
    }
    b -= 8 * a.n16;
    if (b < 64 * a.ed.n_types) {
        const int t = b >> 6, K = a.ed.K[t], row0 = t * H;
        const int64_t w_off = a.ed.w_off[t];
        for (int e = (b & 63) * 256 + threadIdx.x; e < H * a.kmax; e += 64 * 256) {
            const int o = e / a.kmax, k = e % a.kmax;
            const float s = k < K ? params[w_off + (int64_t)o * K + k] * TC_W_SCALE : 0.f;
            const __half h = __float2half_rn(s);
            e_hi[(int64_t)(row0 + o) * a.kmax + k] = h;
            e_lo[(int64_t)(row0 + o) * a.kmax + k] = __float2half_rn((s - __half2float(h)) * TC_LO_SCALE);
        }
        return;
    }
    b -= 64 * a.ed.n_types;
    if (mdl) return;
    for (int64_t i = (int64_t)b * 256 + threadIdx.x; i < a.zero_words; i += (int64_t)a.zero_blocks * 256) a.zero[i] = 0u;
}

// backward prologue: zero the flat gradient buffer (dead branches keep exact zeros) and the stack kernel's completion counters
__global__ void __launch_bounds__(256)
k_bwd_prologue(float4* __restrict__ grads4, const int64_t n4, float* __restrict__ grads_tail, const int n_tail, uint32_t* __restrict__ zero, const int64_t zero_words) {
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n4; i += stride) grads4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < zero_words; i += stride) zero[i] = 0u;
    if (blockIdx.x == 0 && (int)threadIdx.x < n_tail) grads_tail[threadIdx.x] = 0.f;
}

}  // namespace mshgnn
