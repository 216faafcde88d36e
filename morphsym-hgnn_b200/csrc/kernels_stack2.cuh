// CTA-pair variant of the cross-layer stack kernel (kernels_stack.cuh): a cluster of two CTAs on the two SMs of a TPC runs
// every item on TWO row tiles at once with tcgen05.mma.cta_group::2 (M = 256: 128 graph rows per CTA, N = 128).
//
//  Why: the one-CTA kernel is bound by SHARED-MEMORY bandwidth, not by the tensor pipe or L2.  An SS-mode 128 x 128 x 16 MMA
//  reads 4 KB of A and 4 KB of B from shared memory in its 64 cycles - 128 B / cycle, all an SM has - while the TMA ring
//  writes the next operands into the same memory (83 B per tensor cycle: every product of the fp32-class mode streams a
//  (hi, lo) activation tile and a (hi, lo) weight tile) and the epilogue stages residuals / results through it.  Per
//  three-product step that is ~1.2 MB of shared-memory traffic against 4608 tensor cycles = 590 KB of bandwidth: the tensor
//  pipe cannot be more than ~48 % busy (measured: 47-51 %, profiles/r2_stack_timing.txt "mma:issue" = back-pressured MMA issue).
//  With a CTA pair each SM holds only ITS half of every weight K block (64 of the 128 output channels): the weight fill and
//  the B-operand reads per SM halve (40 KB -> 30 KB per K = 16 step and SM), and one thread issues the MMAs of both SMs.
//
//  Structure (everything not listed is the one-CTA kernel, per CTA: epilogue groups, staging, residual fetch, chained
//  base_transform steps, completion signals of the CTA's own row tile):
//   * item = (phase, row-tile PAIR, node slot); CTA r of the cluster owns row tile 2 x pair + r (Bp is a multiple of 256);
//   * the leader's scheduler warp draws the item, waits for the dependencies of BOTH row tiles and publishes the decoded
//     entry into the queues of both CTAs (st.shared::cluster + release / acquire at cluster scope);
//   * each CTA's TMA warp loads its own A tiles and its half of the weight K block (.cta_group::2 loads signalling the
//     LEADER's full barrier: 96 KB per stage in total);
//   * the leader's MMA thread issues for the pair; tcgen05.commit multicasts the "stage free" / "accumulator complete"
//     arrivals to the barriers of both CTAs;
//   * the peer's (otherwise idle) warp 1 relays "my epilogue has drained accumulator a" / "my four groups have staged the
//     chained operand" to the leader with remote mbarrier arrivals.
#pragma once
#include "kernels_stack.cuh"

namespace mshgnn {

constexpr int S2_W_BYTES = SK_TILE_BYTES / 2;                              // 64 weight rows x 64 fp16 = 8 KB per CTA
constexpr int S2_STAGE_BYTES = 2 * SK_TILE_BYTES + 2 * S2_W_BYTES;         // A_hi, A_lo, W_hi half, W_lo half = 48 KB
constexpr int S2_STAGES = 3;
constexpr int S2_PIPE_BYTES = S2_STAGES * S2_STAGE_BYTES;                  // 144 KB
constexpr int S2_SMEM_BYTES = S2_PIPE_BYTES + SK_STG_BYTES + 1024 /*align*/ + 512 /*barriers*/;
// kind::f16, A = B = fp16, D = fp32, both K-major, M = 256 (two CTAs x 128), N = 128
constexpr uint32_t TC_IDESC_2CTA = (1u << 4) | ((128u >> 3) << 17) | ((256u >> 4) << 24);

__device__ __forceinline__ uint32_t cluster_cta_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// shared::cluster address of the same shared-memory location in CTA `rank` of this cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_f16_2cta(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives (once all MMAs issued so far have completed) on the barrier at this shared-memory offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_2cta(uint32_t bar) {
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask)
                 : "memory");
}
// TMA load of one CTA of the pair; the transaction bytes are counted on `bar` (a shared::cluster address: the leader's barrier)
__device__ __forceinline__ void tma_load_2d_2cta(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP_C:\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE_C;\n"
        "bra WAIT_LOOP_C;\n"
        "WAIT_DONE_C:\n"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void st_cluster_v4(uint32_t cluster_addr, const int4 v) {
    asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(cluster_addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void st_release_cluster(uint32_t cluster_addr, const int v) {
    asm volatile("st.release.cluster.shared::cluster.u32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_cluster(uint32_t saddr) {
    int v;
    asm volatile("ld.acquire.cluster.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(saddr) : "memory");
    return v;
}

template <bool PRIV>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(SK_THREADS, 1)
k_tc_stack2(const __grid_constant__ TcMaps maps, const __grid_constant__ CUtensorMap map_w, const Tile* __restrict__ tiles,
            const StackItem* __restrict__ items, const __grid_constant__ StackArgs args, const BufTable bt, const BufRows br) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(16) float bias_w[16][32];        // one copy per epilogue warp
    __shared__ __align__(16) int4 q_ent[SK_QUEUE][2];     // written by the LEADER's scheduler warp (into both CTAs)
    __shared__ __align__(16) int4 q_chunk[SK_QUEUE][SK_QCHUNKS];   // operand rows of the item's chunks (stack_chunk_desc), same for both CTAs
    __shared__ __align__(16) int4 q_hdr[SK_QUEUE][SK_QSTEPS][SK_HDR16];   // tile headers of the item's steps
    __shared__ int q_count;                               // entries published (release / acquire at cluster scope)
    __shared__ volatile int q_prod;                       // leader: entries its TMA producer has started

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_cta_rank();
    const bool is_leader = rank == 0;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S2_PIPE_BYTES + SK_STG_BYTES);
    // barrier table (8 bytes each); the dynamic shared-memory offsets are identical in the two CTAs
    const uint32_t full0 = smem_u32(bars), empty0 = full0 + 8 * S2_STAGES, acc_full0 = empty0 + 8 * S2_STAGES, acc_free0 = acc_full0 + 8 * SK_ACCS,
                   res_bar = acc_free0 + 8 * SK_ACCS, stage_bar = res_bar + 8 * 4, peer_free0 = stage_bar + 8, peer_stage = peer_free0 + 8 * SK_ACCS;
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t stg_base = smem_base + S2_PIPE_BYTES;
    const uint32_t q_count_a = smem_u32(&q_count);

    if (tid == 0) {
        for (int s = 0; s < S2_STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        for (int a = 0; a < SK_ACCS; ++a) { mbar_init(acc_full0 + 8 * a, 1); mbar_init(acc_free0 + 8 * a, 512); mbar_init(peer_free0 + 8 * a, 1); }
        for (int g = 0; g < 4; ++g) mbar_init(res_bar + 8 * g, 1);
        mbar_init(stage_bar, 4);
        mbar_init(peer_stage, 1);
        q_count = 0; q_prod = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    cluster_sync_all();                            // the peer's barriers and queue exist before anything remote touches them
    if (warp == 1) tmem_alloc_2cta(smem_u32(&tmem_base_s), SK_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    constexpr int SPC = H / SK_KB;
    const StackProg& pg = args.prog;
    const int NT = args.n_row_tiles, NP = NT >> 1, RC2 = args.delay, n_total = args.n_total, split = args.split;
    const int64_t Bp = args.Bp;
    uint32_t* const err = args.err;
    const bool dbg_no_a = args.debug & 1, dbg_no_w = args.debug & 2, dbg_no_mma = args.debug & 4, dbg_bare_epi = args.debug & 8;
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    auto next_item = [&](const int n, int4& a, int4& b) {
        if (lane == 0) { while (ld_acquire_cluster(q_count_a) <= n) { } }
        __syncwarp();
        a = q_ent[n % SK_QUEUE][0];
        b = q_ent[n % SK_QUEUE][1];
    };

    if (warp == 18) {
        if (is_leader) {
            int n_pub = 0;
            for (;;) {
                int cur = 0;
                if (lane == 0) {
                    while (n_pub - q_prod >= args.lookahead) { }
                    cur = (int)atomicAdd(args.next, 1u);
                }
                cur = __shfl_sync(0xffffffffu, cur, 0);
                int4 a = make_int4(0, 0, 0, 0), b = make_int4(0, 0, 0, 0);
                const int slot = n_pub % SK_QUEUE;
                if (cur < n_total) {
                    const ItemRef ir = args.chunked ? stack_decode_chunked(pg, NP, RC2, cur) : stack_decode(pg, NP, RC2, cur);
                    const StackItem it = items[ir.item];
                    const int mdl = stack_model(args, 2 * ir.row_tile);      // Bm is a multiple of 256: both row tiles are the model's
                    // descriptors first (they do not depend on the dependency; the slot is invisible until q_count moves),
                    // dependency wait second: the global round trips and the remote stores overlap
                    if (lane < SK_QCHUNKS) {
                        const int4 d = stack_chunk_desc(tiles, it.tile, it.n_steps, it.meta, lane, br, Bp, mdl * args.w16_rows);
                        const uint32_t qc = smem_u32(&q_chunk[slot][lane]);
                        st_cluster_v4(map_to_cta(qc, 0), d);
                        st_cluster_v4(map_to_cta(qc, 1), d);
                    }
                    if (lane < it.n_steps * SK_HDR16) {
                        const int4 h = stack_model_hdr(__ldg(reinterpret_cast<const int4*>(tiles + it.tile + lane / SK_HDR16) + lane % SK_HDR16), lane % SK_HDR16,
                                                       tiles + it.tile + lane / SK_HDR16, mdl, args);
                        const uint32_t qh = smem_u32(&q_hdr[slot][lane / SK_HDR16][lane % SK_HDR16]);
                        st_cluster_v4(map_to_cta(qh, 0), h);
                        st_cluster_v4(map_to_cta(qh, 1), h);
                    }
                    if (ir.phase > 0 && it.dep_mask) {
                        const uint32_t* ctr = args.sync + ((size_t)(ir.phase - 1) * NT + 2 * ir.row_tile) * args.n_slots;
                        stack_wait2(ctr, ctr + args.n_slots, it.dep_mask, lane, err);
                    }
                    a = make_int4(2 * ir.row_tile, ir.phase, it.tile, it.n_steps);
                    b = make_int4(it.meta, it.out_slot, 0, 0);
                }
                asm volatile("fence.acq_rel.cluster;" ::: "memory");
                __syncwarp();
                if (lane < 2) {                                  // lane r publishes to CTA r
                    int4 ar = a;
                    ar.x += lane;
                    const uint32_t e = map_to_cta(smem_u32(&q_ent[slot][0]), (uint32_t)lane);
                    st_cluster_v4(e, ar);
                    st_cluster_v4(e + 16, b);
                    st_release_cluster(map_to_cta(q_count_a, (uint32_t)lane), n_pub + 1);
                }
                __syncwarp();
                // L1 prefetch of the epilogue's global reads of this CTA's row tile (the entry was written through the cluster
                // window: read it back only after the release above)
                if (a.w && !(args.debug & 64)) { ld_acquire_cluster(q_count_a); for (int s = 0; s < a.w; ++s) stack_prefetch_step(*reinterpret_cast<const TileHdr*>(q_hdr[slot][s]), bt, a.x * TILE_M, Bp, lane); }
                ++n_pub;
                if (cur >= n_total) break;
            }
        } else {
            // the peer's scheduler warp has nothing to schedule: it prefetches for its own row tile
            for (int n = 0;; ++n) {
                int4 qa, qb;
                next_item(n, qa, qb);
                if (qa.w == 0) break;
                if (!(args.debug & 64)) for (int s = 0; s < qa.w; ++s) stack_prefetch_step(*reinterpret_cast<const TileHdr*>(q_hdr[n % SK_QUEUE][s]), bt, qa.x * TILE_M, Bp, lane);
            }
        }
    } else if (warp == 0) {
        const uint32_t full_leader0 = map_to_cta(full0, 0);
        uint32_t g = 0;
        for (int n = 0;; ++n) {
            int4 qa, qb;
            next_item(n, qa, qb);
            if (qa.w == 0) break;
            if (lane == 0) {
                if (is_leader) q_prod = n + 1;
                asm volatile("fence.proxy.async.global;" ::: "memory");
                const int row0 = qa.x * TILE_M;
                const int4* qc = q_chunk[n % SK_QUEUE];
                for (int s = 0; s < qa.w; ++s) {
                    const int n_chunks = (qb.x >> (8 * s)) & 0xf, a_stage = (qb.x >> (8 * s + 4)) & 1;
                    for (int c = 0; c < n_chunks; ++c) {
                        const bool from_stage = a_stage && c == 0;
                        const int4 d = *qc++;
                        const int arow_hi = d.x + row0, arow_lo = d.y + row0, w16_row = d.z + 64 * (int)rank;
                        // bytes of BOTH CTAs land on the leader's barrier
                        const uint32_t tx_bytes = 2u * (uint32_t)((split ? 2 : 1) * ((from_stage || dbg_no_a ? 0 : SK_TILE_BYTES) + (dbg_no_w ? 0 : S2_W_BYTES)));
                        for (int kb = 0; kb < SPC; ++kb, ++g) {
                            const uint32_t s3 = g % S2_STAGES;
                            if (!is_leader && dbg_no_a && dbg_no_w) continue;     // ablation: nothing would couple this thread to the leader's ring
                            mbar_wait(empty0 + 8 * s3, ((g / S2_STAGES) & 1) ^ 1);
                            const int kcol = kb * SK_KB;
                            const uint32_t st = smem_base + s3 * S2_STAGE_BYTES;
                            const uint32_t fb = full_leader0 + 8 * s3;
                            if (is_leader) mbar_expect_tx(full0 + 8 * s3, tx_bytes);
                            if (!from_stage && !dbg_no_a) tma_load_2d_2cta(st, &maps.o, fb, kcol, arow_hi);
                            if (!dbg_no_w) tma_load_2d_2cta(st + 2 * SK_TILE_BYTES, &map_w, fb, kcol, br.w_hi + w16_row);
                            if (split) {
                                if (!from_stage && !dbg_no_a) tma_load_2d_2cta(st + SK_TILE_BYTES, &maps.o, fb, kcol, arow_lo);
                                if (!dbg_no_w) tma_load_2d_2cta(st + 2 * SK_TILE_BYTES + S2_W_BYTES, &map_w, fb, kcol, br.w_lo + w16_row);
                            }
                        }
                    }
                }
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        uint32_t g = 0, k = 0, n_staged = 0;
        const uint32_t peer_free_leader0 = map_to_cta(peer_free0, 0), peer_stage_leader = map_to_cta(peer_stage, 0);
        for (int n = 0;; ++n) {
            int4 qa, qb;
            next_item(n, qa, qb);
            if (qa.w == 0) break;
            if (lane == 0) {
                for (int s = 0; s < qa.w; ++s, ++k) {
                    const int n_chunks = (qb.x >> (8 * s)) & 0xf, a_stage = (qb.x >> (8 * s + 4)) & 1;
                    const uint32_t a = k % SK_ACCS;
                    mbar_wait(acc_free0 + 8 * a, ((k / SK_ACCS) & 1) ^ 1);         // this CTA's epilogue has drained the accumulator
                    if (!is_leader) {
                        // relay: the leader's MMA thread waits for both CTAs
                        tc_fence_after();
                        mbar_arrive_remote(peer_free_leader0 + 8 * a);
                        if (a_stage && n_chunks > 0) {
                            mbar_wait(stage_bar, n_staged & 1);
                            ++n_staged;
                            mbar_arrive_remote(peer_stage_leader);
                        }
                        continue;
                    }
                    mbar_wait_cluster(peer_free0 + 8 * a, (k / SK_ACCS) & 1);
                    tc_fence_after();
                    const uint32_t d0 = tmem_base + a * 128;
                    for (int c = 0; c < n_chunks; ++c) {
                        const bool from_stage = a_stage && c == 0;
                        if (from_stage) {
                            mbar_wait(stage_bar, n_staged & 1);
                            mbar_wait_cluster(peer_stage, n_staged & 1);
                            ++n_staged;
                            tc_fence_after();
                        }
                        for (int kb = 0; kb < SPC; ++kb, ++g) {
                            const uint32_t s3 = g % S2_STAGES;
                            mbar_wait_cluster(full0 + 8 * s3, (g / S2_STAGES) & 1);
                            tc_fence_after();
                            const uint32_t st = smem_base + s3 * S2_STAGE_BYTES;
                            const uint64_t w_hi = smem_desc_sw128(st + 2 * SK_TILE_BYTES), w_lo = smem_desc_sw128(st + 2 * SK_TILE_BYTES + S2_W_BYTES);
#pragma unroll
                            for (int ks = 0; ks < SK_KB / 16; ++ks) {
                                uint64_t a_hi, a_lo;
                                if (from_stage) {
                                    const uint32_t blk = stg_base + (uint32_t)(kb * (SK_KB / 32) + (ks >> 1)) * 16384u;
                                    a_hi = smem_desc_sw64(blk) + (uint64_t)((ks & 1) * 2);
                                    a_lo = smem_desc_sw64(blk + 8192u) + (uint64_t)((ks & 1) * 2);
                                } else {
                                    a_hi = smem_desc_sw128(st) + (uint64_t)(ks * 2);
                                    a_lo = smem_desc_sw128(st + SK_TILE_BYTES) + (uint64_t)(ks * 2);
                                }
                                const uint64_t adv = (uint64_t)(ks * 2);
                                if (dbg_no_mma) continue;
                                umma_f16_2cta(d0, a_hi, w_hi + adv, TC_IDESC_2CTA, (c | kb | ks) ? 1u : 0u);
                                if (split) {
                                    umma_f16_2cta(d0, a_lo, w_hi + adv, TC_IDESC_2CTA, 1u);
                                    umma_f16_2cta(d0, a_hi, w_lo + adv, TC_IDESC_2CTA, 1u);
                                }
                            }
                            umma_commit_2cta(empty0 + 8 * s3);
                        }
                    }
                    umma_commit_2cta(acc_full0 + 8 * a);
                }
            }
            __syncwarp();
        }
    } else {
        const int grp = (warp - 2) >> 2;
        const bool sig_leader = (warp & 3) == 2 && lane == 0;
        StackEpi es;
        es.stg = stg_base + grp * 16384; es.bias = smem_u32(bias_w[warp - 2]); es.res_bar = res_bar + 8 * grp; es.stage_bar = stage_bar;
        uint32_t k = 0, n_res = 0;
        uint32_t* pending = nullptr;               // group leader: completion counter of the last item, not yet published
        for (int n = 0;; ++n) {
            int4 qa, qb;
            if (lane == 0) { while (ld_acquire_cluster(q_count_a) <= n) { if (sig_leader) stack_flush_signal(pending); } }
            __syncwarp();
            qa = q_ent[n % SK_QUEUE][0];
            qb = q_ent[n % SK_QUEUE][1];
            if (qa.w == 0) break;
            uint32_t* const ctr = args.sync + ((size_t)qa.y * NT + qa.x) * args.n_slots + qb.y;
            for (int s = 0; s < qa.w; ++s, ++k) {
                TileHdr t;
#pragma unroll
                for (int i = 0; i < SK_HDR16; ++i) reinterpret_cast<int4*>(&t)[i] = q_hdr[n % SK_QUEUE][s][i];
                const uint32_t a = k % SK_ACCS;
                es.accum_bar = acc_full0 + 8 * a; es.free_bar = acc_free0 + 8 * a;
                es.acc_parity = (k / SK_ACCS) & 1;
                    const int live_end = stack_live_end(args, stack_model(args, qa.x));
                    stack_epilogue<PRIV>(t, bt, br, &maps.k, tmem_base + a * 128, qa.x * TILE_M, live_end, Bp, warp, lane, grp, es, n_res, s == qa.w - 1 ? ctr : nullptr,
                                   pending, args.ws, dbg_bare_epi, args.debug);
            }
        }
        if (sig_leader) { stack_flush_signal(pending); tma_store_wait_all(); }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                            // no CTA of the pair leaves while the other may still signal its barriers
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_2cta(tmem_base, SK_TMEM_COLS);
    }
}

}  // namespace mshgnn
