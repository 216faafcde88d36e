// Persistent, warp-specialised encoder (default of the tensor-core modes since round 2 for fp32 feature tensors with 16-byte aligned
// rows; option "encoder" = 2 / 1 selects the one-item-per-CTA kernels of kernels_tc.cuh, which also serve fp64 / fp16 / unaligned inputs).
//
//   h0[slot] = relu((x[slot] * sign[slot]) W_enc[type]^T + b)                    (hgnn_k4.py:L159-160, L198-237)
//
//  The caller's feature rows are the only mandatory HBM stream of the model (43.2 KB per graph for the K4 Mini Cheetah model).
//  k_tc_encoder_pair reads them at 30 % of the measured copy bandwidth.  What held it there (round-2 measurements, DESIGN 3.3):
//  its loader warps keep three register sets of 16-byte loads in flight - in the source.  In the SASS all sets share ONE scoreboard
//  (the packed fp16 conversions of the (hi, lo) split are variable-latency instructions and take the other five), and a scoreboard
//  wait is "every load counted on it has returned": waiting for the oldest set waits for the youngest too, so each thread exposes
//  one full DRAM latency (~2 us loaded) per 64-row block with a single set in flight.  A persistent variant of the same loader
//  (one CTA per SM, dedicated epilogue warps, double-buffered accumulators) measured SLOWER (0.44 against 0.37 ms), and with the
//  conversion and the MMAs switched off its loads alone still took 0.30 ms: the loads were the limit, not what surrounds them.
//  Here the feature rows never pass through a scoreboard:
//    * a 3-D tensor map over every feature tensor x[B * nodes, K] (dims K, nodes, B; box 64 columns x 1 node x 128 graphs) lets
//      ONE TMA request fetch the 128 row fragments of 256 bytes of a (row tile, K block): 32 KB of raw fp32 land in the 32 KB of
//      the operand stage that will hold the tile's (hi, lo) fp16 images, columns >= K and graphs >= B arrive as zeros.
//      Completion is a transaction count on an mbarrier per (stage, row tile) - ordered, per stage, no register is tied up while
//      the bytes are in flight (64 KB per stage and SM).  (128 separate cp.async.bulk row copies per tile were measured first:
//      0.43 ms, the copy engine's request rate - ~36 cycles per 256-byte copy - became the limit);
//    * eight converter warps (two groups of 128 threads, one per row tile) wait for the landing barrier, read the raw tile into
//      registers (16 x 16 bytes per thread), meet on a named barrier, and write the signed (hi, lo) split IN PLACE in the
//      128B-swizzled K-major UMMA layout;
//    * warp 0 = scheduler (items = node slot in descending-K order x pair of 128-row tiles - single tiles when pairs would leave an SM
//      fewer than four items, launch_tc_encoder - drawn from a global counter and published through a small shared-memory queue every
//      role walks) + feature / weight-tile TMA, warp 1 = MMA issuer;
//    * warps 12..15 only ever drain accumulators (tc_epilogue_alt, a private 32 KB staging pair, TMA stores); the accumulators
//      are double-buffered in TMEM (2 items x 2 row tiles x 128 columns = all 512 columns), so the MMAs of item n + 1 run while
//      item n is converted to (hi, lo) images and stored.
//  Shared memory: 2 stages x (A0_hi, A0_lo, A1_hi, A1_lo, W_hi, W_lo) 96 KB + 32 KB epilogue staging + 2.3 KB control = the whole
//  227 KB; the kernel has no static shared memory, so the dynamic window starts 1024-aligned.
#pragma once
#include "kernels_tc.cuh"

namespace mshgnn {

constexpr int ENQ_THREADS = 512;
constexpr int ENQ_STAGES = 2;
constexpr int ENQ_STAGE_BYTES = 6 * ENC_TILE_BYTES;          // 96 KB
constexpr int ENQ_STG_BYTES = 2 * ENC_TILE_BYTES;            // 32 KB: (hi | lo) tiles of 128 rows x 64 fp16
constexpr int ENQ_TILE_REGION = ENQ_STAGES * ENQ_STAGE_BYTES + ENQ_STG_BYTES;
constexpr int ENQ_SMEM_BYTES = 232448;                       // 227 KB, the per-CTA maximum of sm_100
constexpr int ENQ_MAX_SLOTS = 32;
constexpr int ENQ_ITEM_Q = 4;
constexpr uint32_t ENQ_TMEM_COLS = 512;
constexpr int ENQ_CONV_WARP0 = 4, ENQ_EPI_WARP0 = 12;
constexpr int ENQ_ITEM_CONSUMERS = 1 + 8 + 4;                // MMA thread, converter warps, epilogue warps

struct EnqSlot {
    int xt, node, K, sign_off, w16_row, n_kb, tile, pad;     // xt: feature tensor (node type) of the slot, node: its node inside a graph
};

struct alignas(64) EnqMaps {
    CUtensorMap w_hi, w_lo;      // encoder weight images, box 64 x 128, SWIZZLE_128B
    CUtensorMap o;               // workspace images, box 64 x 128, SWIZZLE_128B (epilogue stores)
    CUtensorMap x[4];             // caller's feature tensors as (K, nodes, B) fp32, box 64 x 1 x 128, no swizzle
};

struct alignas(16) EnqCtl {
    float bias[H];
    EnqSlot slots[ENQ_MAX_SLOTS];                            // descending K: the long items are drawn first
    uint64_t full[ENQ_STAGES], empty[ENQ_STAGES], landed[ENQ_STAGES][2], acc_full[2], acc_free[2], item_full[ENQ_ITEM_Q], item_empty[ENQ_ITEM_Q], res_bar;
    int items[ENQ_ITEM_Q];
    uint32_t tmem_base;
    int pad[3];
    Tile t;                                                  // tile of the item the epilogue warps work on
};
static_assert(ENQ_TILE_REGION + sizeof(EnqCtl) <= ENQ_SMEM_BYTES, "encoder control block does not fit behind the tiles");

// host-side test of what the tensor maps need: fp32 rows of a 16-byte multiple on a 16-byte aligned base (and whole 4-column sign groups)
inline bool enq_rows_ok(const void* base, int K, int sign_off) {
    return (reinterpret_cast<uintptr_t>(base) & 15) == 0 && (K & 3) == 0 && K >= 4 && (sign_off < 0 || (sign_off & 3) == 0);
}

__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap* map, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// entry m of the item queue (every role reads the same sequence); warps release with one arrival
__device__ __forceinline__ int enq_take(EnqCtl& ctl, const int m, const bool whole_warp, const int lane) {
    const int q = m % ENQ_ITEM_Q;
    mbar_wait(smem_u32(&ctl.item_full[q]), (uint32_t)(m / ENQ_ITEM_Q) & 1u);
    const int id = *reinterpret_cast<volatile int*>(&ctl.items[q]);
    if (whole_warp) __syncwarp();
    if (!whole_warp || lane == 0) mbar_arrive(smem_u32(&ctl.item_empty[q]));
    return id;
}

__global__ void __launch_bounds__(ENQ_THREADS, 1)
k_tc_encoder_stream(const __grid_constant__ EnqMaps maps, const Tile* __restrict__ tiles, const int n_slots, const int x_buf0 /*buffer id of the first feature tensor*/, const BufTable bt, const BufRows br,
                    const int64_t B, const int64_t Bp, const int split, uint32_t* __restrict__ counter, const int tpi /*row tiles per item: 1 or 2*/, const int pf /*L2 prefetch distance in K blocks, 0 = off*/,
                    const int dbg /*measurement switches: 1 no conversion, 2 no MMAs, 4 no weight loads (results are wrong when set; the host passes 0)*/) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const uint32_t smem_base = smem_u32(smem_raw);
    EnqCtl& ctl = *reinterpret_cast<EnqCtl*>(smem_raw + ENQ_TILE_REGION);
    const uint32_t full0 = smem_u32(&ctl.full[0]), empty0 = smem_u32(&ctl.empty[0]), landed0 = smem_u32(&ctl.landed[0][0]),
                   acc_full0 = smem_u32(&ctl.acc_full[0]), acc_free0 = smem_u32(&ctl.acc_free[0]);
    const int n_pairs = (int)((Bp / TILE_M + tpi - 1) / tpi);        // items per node slot: tpi (1 or 2) row tiles each
    const int item_rows = tpi * TILE_M;
    const int n_items = n_slots * n_pairs;

    if (smem_base & 1023u) __trap();                         // the swizzled tiles need the 1024-byte alignment (no static shared memory in this kernel)
    {
        // slot table in descending-K order (stable): rank by counting
        int* keys = reinterpret_cast<int*>(ctl.bias);
        Chunk ch;
        if (tid < n_slots) {
            ch = tiles[tid].chunks[0];
            keys[tid] = ch.K;
        }
        __syncthreads();
        if (tid < n_slots) {
            int rank = 0;
            for (int j = 0; j < n_slots; ++j) rank += (keys[j] > ch.K || (keys[j] == ch.K && j < tid)) ? 1 : 0;
            EnqSlot s;
            s.xt = ch.a_buf - x_buf0; s.node = ch.a_off / ch.K; s.K = ch.K; s.sign_off = ch.sign_off; s.w16_row = ch.w16_row;
            s.n_kb = (ch.K + 63) / 64; s.tile = tid; s.pad = 0;
            ctl.slots[rank] = s;
        }
    }
    if (tid == 0) {
        for (int s = 0; s < ENQ_STAGES; ++s) {
            mbar_init(full0 + 8 * s, 1 + 8);                 // weight TMA + the eight converter warps
            mbar_init(empty0 + 8 * s, 1);
            mbar_init(landed0 + 16 * s, 1);
            mbar_init(landed0 + 16 * s + 8, 1);
        }
        for (int b = 0; b < 2; ++b) { mbar_init(acc_full0 + 8 * b, 1); mbar_init(acc_free0 + 8 * b, 256); }
        for (int q = 0; q < ENQ_ITEM_Q; ++q) { mbar_init(smem_u32(&ctl.item_full[q]), 1); mbar_init(smem_u32(&ctl.item_empty[q]), ENQ_ITEM_CONSUMERS); }
        mbar_init(smem_u32(&ctl.res_bar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(&ctl.tmem_base), ENQ_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = ctl.tmem_base;

    if (warp < ENQ_CONV_WARP0) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
        if (warp == 0) {
            if (lane == 0) {
                // ---------------- scheduler + weight tiles ----------------
                const uint32_t tx_bytes = split ? 2 * ENC_TILE_BYTES : ENC_TILE_BYTES;
                auto publish = [&](const int m, const uint32_t id) {
                    const int q = m % ENQ_ITEM_Q;
                    mbar_wait(smem_u32(&ctl.item_empty[q]), ((uint32_t)(m / ENQ_ITEM_Q) & 1u) ^ 1u);
                    *reinterpret_cast<volatile int*>(&ctl.items[q]) = (int)(id < (uint32_t)n_items ? id : (uint32_t)n_items);
                    mbar_arrive(smem_u32(&ctl.item_full[q]));
                };
                uint32_t id_cur = atomicAdd(counter, 1u), id_next = atomicAdd(counter, 1u);
                publish(0, id_cur);
                uint32_t kbi = 0;
                int pf_pos = 0;                              // next K block (relative to the current item's first) the L2 prefetch cursor will request
                for (int m = 0;; ++m) {
                    publish(m + 1, id_next);                 // the producers open the next item while this one is still in the pipeline
                    const uint32_t id_after = id_next < (uint32_t)n_items ? atomicAdd(counter, 1u) : (uint32_t)n_items;
                    if (id_cur >= (uint32_t)n_items) break;
                    const int si = (int)id_cur / n_pairs;
                    const EnqSlot& sl = ctl.slots[si];
                    const int row0 = ((int)id_cur - si * n_pairs) * item_rows;
                    const bool two = tpi == 2 && (int64_t)row0 + TILE_M < Bp;
                    const int wrow = sl.w16_row, n_kb = sl.n_kb, node = sl.node;
                    const CUtensorMap* xm = &maps.x[sl.xt];
                    // the item after this one, for the L2 prefetch cursor
                    const bool nx_ok = id_next < (uint32_t)n_items;
                    const int nsi = nx_ok ? (int)id_next / n_pairs : 0;
                    const EnqSlot& nsl = ctl.slots[nsi];
                    const int nrow0 = ((int)id_next - nsi * n_pairs) * item_rows;
                    const bool ntwo = tpi == 2 && (int64_t)nrow0 + TILE_M < Bp;
                    for (int i = 0; i < n_kb; ++i, ++kbi) {
                        // optional L2 prefetch of the feature boxes pf K blocks ahead of the loads (through this item into the next one).  Idea: the
                        // landing zones are the two operand stages, so a stage that is being converted or multiplied requests nothing - a prefetch
                        // would keep DRAM busy meanwhile.  Measured (same box): 2 K blocks ahead no change, 4: 0.21 -> 0.235 ms,
                        // 8: 0.266 ms - the extra requests compete with the demand loads instead of preceding them.  The host passes pf = 0.
                        while (pf > 0 && pf_pos <= i + pf) {
                            if (pf_pos < n_kb) {
                                tma_prefetch_3d(xm, pf_pos * 64, node, row0);
                                if (two) tma_prefetch_3d(xm, pf_pos * 64, node, row0 + TILE_M);
                            } else if (nx_ok && pf_pos - n_kb < nsl.n_kb) {
                                tma_prefetch_3d(&maps.x[nsl.xt], (pf_pos - n_kb) * 64, nsl.node, nrow0);
                                if (ntwo) tma_prefetch_3d(&maps.x[nsl.xt], (pf_pos - n_kb) * 64, nsl.node, nrow0 + TILE_M);
                            } else
                                break;
                            ++pf_pos;
                        }
                        const uint32_t s = kbi & 1u;
                        mbar_wait(empty0 + 8 * s, ((kbi >> 1) & 1u) ^ 1u);
                        const uint32_t st = smem_base + s * ENQ_STAGE_BYTES;
                        // raw feature rows of both row tiles (graphs >= B and columns >= K are zero-filled by the TMA unit)
                        const uint32_t lb = landed0 + 16 * s;
                        mbar_expect_tx(lb, 2 * ENC_TILE_BYTES);
                        tma_load_3d(st, xm, lb, i * 64, node, row0);
                        if (two) {
                            mbar_expect_tx(lb + 8, 2 * ENC_TILE_BYTES);
                            tma_load_3d(st + 2 * ENC_TILE_BYTES, xm, lb + 8, i * 64, node, row0 + TILE_M);
                        } else
                            mbar_arrive(lb + 8);             // nothing to copy, but every barrier keeps one phase per K block
                        const uint32_t fb = full0 + 8 * s;
                        if (dbg & 4) { mbar_arrive(fb); continue; }
                        mbar_expect_tx(fb, tx_bytes);
                        tma_load_2d(st + 4 * ENC_TILE_BYTES, &maps.w_hi, fb, i * 64, wrow);
                        if (split) tma_load_2d(st + 5 * ENC_TILE_BYTES, &maps.w_lo, fb, i * 64, wrow);
                    }
                    pf_pos = pf_pos > n_kb ? pf_pos - n_kb : 0;      // positions are relative to the first K block of the current item
                    id_cur = id_next;
                    id_next = id_after;
                }
            }
        } else if (warp == 1) {
            if (lane == 0) {
                // ---------------- MMA issuer ----------------
                uint32_t kbi = 0;
                for (int m = 0;; ++m) {
                    const int id = enq_take(ctl, m, false, 0);
                    if (id >= n_items) break;
                    const int si = id / n_pairs;
                    const int row0 = (id - si * n_pairs) * item_rows;
                    const int n_tiles = (tpi == 2 && (int64_t)row0 + TILE_M < Bp) ? 2 : 1;
                    const int n_kb = ctl.slots[si].n_kb;
                    const uint32_t b = (uint32_t)m & 1u;
                    mbar_wait(acc_free0 + 8 * b, (((uint32_t)m >> 1) & 1u) ^ 1u);       // the epilogue has drained this accumulator pair
                    tc_fence_after();
                    for (int i = 0; i < n_kb; ++i, ++kbi) {
                        const uint32_t s = kbi & 1u;
                        mbar_wait(full0 + 8 * s, (kbi >> 1) & 1u);
                        tc_fence_after();
                        const uint32_t st = smem_base + s * ENQ_STAGE_BYTES;
                        const uint64_t w_hi = smem_desc_sw128(st + 4 * ENC_TILE_BYTES), w_lo = smem_desc_sw128(st + 5 * ENC_TILE_BYTES);
                        for (int tl = 0; tl < n_tiles; ++tl) {
                            const uint64_t a_hi = smem_desc_sw128(st + (2 * tl) * ENC_TILE_BYTES), a_lo = smem_desc_sw128(st + (2 * tl + 1) * ENC_TILE_BYTES);
                            const uint32_t acc = tmem_base + b * 256u + (uint32_t)tl * 128u;
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                if (dbg & 2) continue;
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
                    umma_commit(acc_full0 + 8 * b);
                }
            }
        }
    } else if (warp < ENQ_EPI_WARP0) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 168;");
        // ---------------- converters: group g turns the raw rows of row tile g into the signed (hi, lo) operand images, in place ----------------
        const int g = (warp - ENQ_CONV_WARP0) >> 2;
        const int gt = tid - ENQ_CONV_WARP0 * 32 - g * 128;
        const int kq = gt & 15;                                   // which 4-column group of the 64-column block
        const int rsub = gt >> 4;                                 // 0..7: rows rsub + 8 u
        const float* signs = (const float*)bt.p[2];
        uint32_t kbi = 0;
        for (int m = 0;; ++m) {
            const int id = enq_take(ctl, m, true, lane);
            if (id >= n_items) break;
            const int si = id / n_pairs;
            const int64_t row0 = (int64_t)(id - si * n_pairs) * item_rows + g * TILE_M;
            const EnqSlot sl = ctl.slots[si];
            const bool live = g < tpi && row0 < Bp;
            for (int i = 0; i < sl.n_kb; ++i, ++kbi) {
                const uint32_t s = kbi & 1u;
                if (!live) {
                    // nothing lands for this row tile: the scheduler's bare arrival says the stage has been released (one phase per K block on every barrier)
                    mbar_wait(landed0 + 16 * s + 8 * g, (kbi >> 1) & 1u);
                    __syncwarp();
                    if (lane == 0) mbar_arrive(full0 + 8 * s);
                    continue;
                }
                const int k = i * 64 + kq * 4;
                float4 sg = make_float4(1.f, 1.f, 1.f, 1.f);
                if (sl.sign_off >= 0 && k < sl.K) sg = __ldg(reinterpret_cast<const float4*>(signs + sl.sign_off + k));     // K, sign_off: multiples of 4 (enq_rows_ok)
                const uint32_t st = smem_base + s * ENQ_STAGE_BYTES + (uint32_t)g * (2 * ENC_TILE_BYTES);
                mbar_wait(landed0 + 16 * s + 8 * g, (kbi >> 1) & 1u);
                float4 v[16];
#pragma unroll
                for (int u = 0; u < 16; ++u) {
                    const int r = u * 8 + rsub;
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[u].x), "=f"(v[u].y), "=f"(v[u].z), "=f"(v[u].w) : "r"(st + (uint32_t)(r * 256 + kq * 16)));
                }
                asm volatile("bar.sync %0, 128;" ::"r"(2 + g) : "memory");       // every raw row of the tile is in registers: the images may overwrite them
                if (!(dbg & 1)) {
#pragma unroll
                    for (int u = 0; u < 16; ++u) {
                        const int r = u * 8 + rsub;
                        const uint32_t off = (uint32_t)(r * 128 + ((((kq >> 1) ^ (r & 7))) << 4) + ((kq & 1) << 3));
                        split_to_smem(st + off, st + ENC_TILE_BYTES + off, v[u], sg);
                    }
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(full0 + 8 * s);
            }
        }
    } else {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 112;");
        // ---------------- epilogue: accumulator pair (m & 1) of item m, one row tile after the other ----------------
        const int et = tid - ENQ_EPI_WARP0 * 32;
        uint32_t res_count = 0;
        for (int m = 0;; ++m) {
            const int id = enq_take(ctl, m, true, lane);
            if (id >= n_items) break;
            const int si = id / n_pairs;
            const int row0 = (id - si * n_pairs) * item_rows;
            const int n_tiles = (tpi == 2 && (int64_t)row0 + TILE_M < Bp) ? 2 : 1;
            group_bar_sync(0);                                   // every warp is done with the previous item's tile
            {
                const int* src = reinterpret_cast<const int*>(tiles + ctl.slots[si].tile);
                int* dst = reinterpret_cast<int*>(&ctl.t);
                for (int i = et; i < (int)(sizeof(Tile) / 4); i += 128) dst[i] = __ldg(src + i);
            }
            group_bar_sync(0);
            const uint32_t b = (uint32_t)m & 1u;
            for (int tl = 0; tl < n_tiles; ++tl) {
                EpiSmem es;
                es.stg = smem_base + ENQ_STAGES * ENQ_STAGE_BYTES; es.bias = smem_u32(ctl.bias); es.res_bar = smem_u32(&ctl.res_bar);
                es.accum_bar = acc_full0 + 8 * b; es.free_bar = acc_free0 + 8 * b;
                es.acc_parity = ((uint32_t)m >> 1) & 1u; es.res_parity = 0; es.persistent = 1; es.n_groups = 1;
                tc_epilogue_alt(ctl.t, bt, br, &maps.o, tmem_base + b * 256u + (uint32_t)tl * 128u, row0 + tl * TILE_M, B, Bp, split, warp, lane, 0, es, res_count);
            }
            if (n_tiles == 1) {                                  // the barrier counts both row tiles of a pair
                tc_fence_before();
                mbar_arrive(acc_free0 + 8 * b);
            }
        }
        if (((warp - 2) & 3) == 0 && lane == 0) tma_store_wait_all();       // the thread tc_epilogue_alt issues the stores from
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, ENQ_TMEM_COLS);
    }
}

}  // namespace mshgnn
