// Cross-layer "stack" kernel of the MS-HGNN layer loop (hgnn_k4.py:L170-186 and its autograd mirror), sm_100a only.
//
//  The per-layer launch sequence (kernels_tc.cuh) streams every activation slab through HBM once per layer: 8 x (conv,
//  Linear, Linear) launches forward and 8 x (2 Linear, dX) backward, each writing a [slots x graphs x 128] (hi, lo) slab
//  that the next launch reads back - 6.2 GB of the 11.3 GB a train step moved (profiles/r1_tc_v7_step_traffic.json),
//  where SURVEY 8d counts ZERO mandatory bytes for the layer stack.  A tile of 128 graphs x 20 node slots x (hi, lo)
//  images is 1.3 MB - it cannot be resident in one SM's 227 KB of shared memory (and five 128-row role tiles, the
//  smallest closed set under the morphology's edges, are 320 KB) - so this kernel keeps it resident one level up:
//
//   * ONE persistent launch walks all layers.  Work items are ordered as a diagonal wavefront (stack_decode): a row tile
//     of 128 graphs advances one layer every D time slots, so only ~L x D row tiles (a few thousand graphs) are between
//     their first and last layer at any time and the slabs a layer reads were written a few hundred items earlier - they
//     are still in the 126 MB L2.  In inference the ping-pong slabs never reach HBM at all; in training every h_l is
//     written once (the backward pass needs it) and never read back from DRAM by the forward.
//   * No grid-wide barrier: layer l + 1 of row tile r starts as soon as every item of layer l of row tile r has
//     signalled a global counter (release / acquire at gpu scope, bounded spin).  Items are drawn from one atomic work
//     counter in wavefront order, so no CTA falls behind and the dependency distance (D x items per slot) stays above
//     the number of items in flight: the waits are normally already satisfied.
//   * base_transform (Linear -> ReLU -> Linear, + residual) is CHAINED behind the conv tile of its node inside one item:
//     the epilogue leaves the (hi, lo) result in its staging tiles, which have exactly the operand K-block layout
//     (128 rows x 32 fp16, SWIZZLE_64B), and the MMA warp issues the next GEMM straight from them.  The same chain runs
//     backward (dX of a base node -> dpre -> dc).  That removes 32 short launches per step and, in inference, every
//     byte of the intermediates.
//
//  Roles as in k_tc_rowgemm_persistent: warp 0 = TMA producer (4-stage ring: A_hi, A_lo, W_hi, W_lo K blocks), warp 1 =
//  tcgen05.mma issuer (two 128-column accumulators in TMEM), warps 2..17 = four epilogue groups (one 32-column quarter
//  each, private 16 KB staging pair).
#pragma once
#include "kernels_tc.cuh"

namespace mshgnn {

// Operand K blocks are 64 fp16 wide (128-byte rows, SWIZZLE_128B): with the 32-column blocks of the per-layer kernels the
// MMA warp spent 40-50 % of the kernel waiting for operands while the producer rarely waited for a ring slot - the
// L2 -> SM stream of 64-byte row segments was the bottleneck (profiles/r2_stack_timing.txt), not the bytes in flight.
constexpr int SK_KB = 64;
constexpr int SK_TILE_BYTES = 128 * SK_KB * 2;                            // 16 KB
constexpr int SK_STAGE_BYTES = 4 * SK_TILE_BYTES;                         // A_hi, A_lo, W_hi, W_lo = 64 KB
constexpr int SK_STAGES = 2;
constexpr int SK_QUEUE = 16;                                              // in-CTA item queue (the scheduler runs <= 2 items ahead of the producer)
constexpr int SK_QSTEPS = 3;                                              // steps per item (StackItem::n_steps)
constexpr int SK_HDR16 = 5;                                               // sizeof(TileHdr) / 16
constexpr int SK_QCHUNKS = 16;                                            // chunk descriptors per queued item (all steps of the item together)
constexpr int SK_THREADS = 608;                                           // TMA warp, MMA warp, 16 epilogue warps, scheduler warp
constexpr int SK_PIPE_BYTES = SK_STAGES * SK_STAGE_BYTES;                  // 128 KB operand ring
constexpr int SK_STG_BYTES = 65536;                                       // 4 groups x (hi | lo) x 8 KB
constexpr int SK_SMEM_BYTES = SK_PIPE_BYTES + SK_STG_BYTES + 1024 /*align*/ + 256 /*barriers*/;
constexpr uint32_t SK_TMEM_COLS = 512;                                    // four 128-column accumulators: the MMA warp runs up to three steps ahead of the epilogue
constexpr int SK_ACCS = 4;
constexpr unsigned SK_SPIN_LIMIT = 1u << 22;                              // ~ seconds: a broken dependency must not hang the GPU

struct StackArgs {
    StackProg prog;
    int n_row_tiles;             // Bp / 128
    int delay;                   // D: time slots between consecutive phases of a row tile (see stack_decode); chunked order: row tiles per chunk
    int chunked;                 // 1: chunked order (stack_decode_chunked)
    int lookahead;               // items the scheduler warp may draw ahead of the TMA producer
    int n_slots;                 // node slots per graph: the completion counters are [phase][row tile][slot]
    int n_total;                 // n_row_tiles * prog.items_per_row
    int split;                   // 1: (hi, lo) operands, 3 MMAs per product; 0: hi only
    int64_t B, Bp;
    // model batch: row tile r belongs to model r / tiles_m, which reads its own weight-image rows (w16_rows per model) and biases
    // (n_params / n_derived per model); the scheduler warp resolves both, and the model's bound on live rows, once per item
    int tiles_m, w16_rows, n_params, n_derived;
    uint32_t* sync;              // [n_phases][n_row_tiles][n_slots] completion counters (4 = the four epilogue groups of the producing item)
    uint32_t* err;               // error word (a dependency wait timed out)
    uint32_t* next;              // work counter: the next item index to hand out (zeroed with the completion counters)
    char* ws;                    // workspace base (thread-private fp32 tensors live in the image area of their buffer)
    int debug;                   // ablation switches for timing experiments (the host passes 0; results are garbage otherwise): 1 no A loads,
                                 // 2 no W loads, 4 no MMAs, 8 epilogue reduced to its handshakes, 16 completion signal at once, 32 barrier before every staging write,
                                 // 64 no L1 prefetch, 256 no second output of two-output tiles, 512 no residuals (CTA-pair kernel only)
};

struct ItemRef { int phase, row_tile, item; };

// Item order: a DIAGONAL wavefront.  Time slot t holds, for every phase p, the items of row tile r = t - p * D (when
// 0 <= r < NT): row tiles enter phase 0 one per slot and advance one phase every D slots.  The items of (p, r) are therefore
// handed out D slots - D x (items per slot) items - after those of (p - 1, r), for EVERY phase (with row chunks walked phase
// by phase the pruned last layers, which have few items per row tile, followed their producers too closely and a quarter
// of the kernel was spent in dependency waits), while only P x D row tiles are between their first and last phase at any
// time - the L2-resident working set.
__device__ __forceinline__ int stack_count(const StackProg& pg, const int NT, const int D, const int t) {   // items in slots [0, t)
    int c = 0;
    for (int p = 0; p < pg.n_phases; ++p) c += pg.n_items[p] * min(max(t - p * D, 0), NT);
    return c;
}
// chunked order: chunks of RC row tiles, phase-major inside a chunk (the order the host selects: StackArgs::chunked = 1)
__device__ __forceinline__ ItemRef stack_decode_chunked(const StackProg& pg, const int NT, const int RC, const int i) {
    const int chunk_items = RC * pg.items_per_row;
    const int c = i / chunk_items;
    int j = i - c * chunk_items;
    const int rows_c = min(RC, NT - c * RC);
    int p = 0;
    for (; p < pg.n_phases - 1; ++p) {
        const int blk = rows_c * pg.n_items[p];
        if (j < blk) break;
        j -= blk;
    }
    const int n = pg.n_items[p];
    ItemRef r;
    r.phase = p; r.row_tile = c * RC + j / n; r.item = pg.first_item[p] + j % n;
    return r;
}
__device__ __forceinline__ ItemRef stack_decode(const StackProg& pg, const int NT, const int D, const int i) {
    int lo = 0, hi = NT + (pg.n_phases - 1) * D;          // count(lo) <= i < count(hi)
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (stack_count(pg, NT, D, mid) <= i) lo = mid; else hi = mid;
    }
    int j = i - stack_count(pg, NT, D, lo);
    ItemRef r;
    r.phase = 0; r.row_tile = 0; r.item = 0;
    for (int p = 0; p < pg.n_phases; ++p) {
        const int row = lo - p * D;
        if (row < 0 || row >= NT) continue;
        const int n = pg.n_items[p];
        if (j < n) { r.phase = p; r.row_tile = row; r.item = pg.first_item[p] + j; break; }
        j -= n;
    }
    return r;
}

// Bounded acquire-spin of a whole warp on the completion counters of the node slots in `mask` (lane l polls slots l and
// l + 32).  On timeout (or when another CTA already timed out) the error word is set and the wait gives up: the results
// are then garbage, but the kernel terminates and the host reports the error (mshgnn_stack_status).
__device__ __forceinline__ void stack_wait(const uint32_t* ctr, const unsigned long long mask, const int lane, uint32_t* err) {
    unsigned spins = 0;
    for (;;) {
        bool ok = true;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int sl = lane + 32 * h;
            if ((mask >> sl) & 1ull) {
                uint32_t v;
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr + sl) : "memory");
                ok = ok && v >= 4u;
            }
        }
        if (__all_sync(0xffffffffu, ok)) break;
        ++spins;
        if ((spins & 1023u) == 0) {
            uint32_t e;
            asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(e) : "l"(err) : "memory");
            if (e || spins >= SK_SPIN_LIMIT) { asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(err), "r"(1u) : "memory"); break; }
        }
        __nanosleep(40);
    }
}

// The same wait on the counters of TWO row tiles (CTA-pair kernel) in one polling loop: one load round trip per poll instead of two
// waits in series - the dependency wait sits on the scheduler warp's per-item chain (draw -> decode -> wait -> publish).
__device__ __forceinline__ void stack_wait2(const uint32_t* ctr0, const uint32_t* ctr1, const unsigned long long mask, const int lane, uint32_t* err) {
    unsigned spins = 0;
    for (;;) {
        bool ok = true;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int sl = lane + 32 * h;
            if ((mask >> sl) & 1ull) {
                uint32_t v0, v1;
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v0) : "l"(ctr0 + sl) : "memory");
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v1) : "l"(ctr1 + sl) : "memory");
                ok = ok && v0 >= 4u && v1 >= 4u;
            }
        }
        if (__all_sync(0xffffffffu, ok)) break;
        ++spins;
        if ((spins & 1023u) == 0) {
            uint32_t e;
            asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(e) : "l"(err) : "memory");
            if (e || spins >= SK_SPIN_LIMIT) { asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(err), "r"(1u) : "memory"); break; }
        }
        __nanosleep(40);
    }
}

__device__ __forceinline__ void stack_signal(uint32_t* ctr) {
    // one gpu-scope release: it is cumulative over everything that happens-before it (this thread's completed TMA stores, the other
    // epilogue threads' global stores ordered by the group barrier).  A separate fence.acq_rel.gpu in front of it doubled the cost of
    // what the stall profile shows as the single most expensive instruction of the backward launch (21 % + 5 % of the warp samples;
    // train step 3.09 -> 3.03 ms).  Moving the release to a dedicated signal warp (mailboxes in shared memory, the group leader only
    // posting the counter address) was measured afterwards: no further gain (3.05 ms against 3.03), dropped.
    asm volatile("fence.proxy.async.global;" ::: "memory");
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(ctr), "r"(1u) : "memory");
}

__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}

template <int N>
__device__ __forceinline__ void tma_store_wait_pending() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }

// Operand rows of one chunk of an item, resolved by the scheduler warp (lane l = l-th chunk of the item, steps in order) so
// that the single-thread TMA producer never waits for a descriptor load: {first row of the A hi image of the node slot,
// same for the lo image, first row of the weight image, -}.  `meta` holds one byte per step: chunks | a_stage << 4.
__device__ __forceinline__ int4 stack_chunk_desc(const Tile* tiles, const int first_tile, const int n_steps, const int meta, const int lane,
                                                 const BufRows& br, const int64_t Bp, const int w16_add) {
    int cum = 0;
    int4 d = make_int4(0, 0, 0, 0);
    for (int s = 0; s < n_steps && s < 4; ++s) {
        const int nc = (meta >> (8 * s)) & 0xf;
        if (lane >= cum && lane < cum + nc) {
            const Chunk* c = &tiles[first_tile + s].chunks[lane - cum];
            const int a_buf = __ldg(&c->a_buf), a_slot = __ldg(&c->a_slot);
            d = make_int4(br.hi[a_buf] + (int)((int64_t)a_slot * Bp), br.lo[a_buf] + (int)((int64_t)a_slot * Bp), __ldg(&c->w16_row) + w16_add, 0);
        }
        cum += nc;
    }
    return d;
}

// header of a Tile (everything but the chunk list), fetched once per step into registers
struct TileHdr {
    int n_chunks, out_buf, out_slot, bias_buf, bias_off, relu, posmask_buf, posmask_slot, res_buf, res_slot, mask_out_buf,
        out2_buf, out2_slot, out2_mask_kind, out2_mask_buf, out2_mask_slot, mask_out_slot, a_stage, stage_out, priv;
};
static_assert(sizeof(TileHdr) == offsetof(Tile, chunks), "TileHdr must mirror the head of Tile");
__device__ __forceinline__ TileHdr load_hdr(const Tile* t) {
    TileHdr h;
    const int4* src = reinterpret_cast<const int4*>(t);
    int4* dst = reinterpret_cast<int4*>(&h);
#pragma unroll
    for (int i = 0; i < (int)(sizeof(TileHdr) / 16); ++i) dst[i] = __ldg(src + i);
    return h;
}
static_assert(sizeof(TileHdr) == 16 * SK_HDR16, "queue header slots must hold a TileHdr");
static_assert(offsetof(TileHdr, bias_off) == 16, "stack_model_hdr patches bias_off as word x of header vector 1");

// Model of a model batch that row tile `row_tile` (of 128 rows) belongs to
__device__ __forceinline__ int stack_model(const StackArgs& a, const int row_tile) { return row_tile / a.tiles_m; }
// Rows of the workspace below this bound are live for an item of model `mdl` (its graphs end there; the rest of its block is padding)
__device__ __forceinline__ int stack_live_end(const StackArgs& a, const int mdl) { return mdl * a.tiles_m * TILE_M + (int)a.B; }
// Header vector `v` of a step of model `mdl`: its bias offset moved to that model's parameters / derived bias sums
__device__ __forceinline__ int4 stack_model_hdr(int4 h, const int v, const Tile* tile, const int mdl, const StackArgs& a) {
    if (mdl && v == 1) {
        const int bb = __ldg(&tile->bias_buf);
        h.x += bb == BUF_PARAMS_ID ? mdl * a.n_params : (bb == BUF_DERIVED_ID ? mdl * a.n_derived : 0);
    }
    return h;
}
static_assert(sizeof(TileHdr) % 16 == 0 && sizeof(Tile) % 16 == 0, "Tile entries are read with 128-bit loads");

struct StackEpi {
    uint32_t stg;            // this group's staging pair: hi tile (8 KB) | lo tile (8 KB)
    uint32_t bias;           // 128 B of shared memory private to this WARP: bias of the group's column quarter
    uint32_t res_bar, accum_bar, free_bar, stage_bar;
    uint32_t acc_parity;
};

// Accumulator -> value arithmetic of one thread's 32 columns, specialised on the (CTA-uniform) tile flags: with the flags as run-time
// values the compiler predicates the per-element mask / ReLU code instead of branching around it - ~190 of the ~720 instructions of
// a backward step were compare / select / min-max instructions of features the backward tiles do not have.
template <bool BIAS, bool MASK, bool RELU>
__device__ __forceinline__ unsigned epi_affine(const uint32_t (&raw)[32], float (&v)[32], const uint32_t bias_smem) {
    unsigned mask = 0;
#pragma unroll
    for (int j4 = 0; j4 < 8; ++j4) {
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (BIAS) asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b4.x), "=f"(b4.y), "=f"(b4.z), "=f"(b4.w) : "r"(bias_smem + 16u * j4));
        const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int j = j4 * 4 + e;
            float x = BIAS ? fmaf(__uint_as_float(raw[j]), TC_W_UNSCALE, bb[e]) : __uint_as_float(raw[j]) * TC_W_UNSCALE;
            if (MASK && x > 0.f) mask |= 1u << j;
            if (RELU) x = fmaxf(x, 0.f);
            v[j] = x;
        }
    }
    return mask;
}
__device__ __forceinline__ unsigned epi_affine_any(const bool has_bias, const bool want_mask, const bool relu, const uint32_t (&raw)[32], float (&v)[32],
                                                   const uint32_t bias_smem) {
    if (!has_bias && !want_mask && !relu) return epi_affine<false, false, false>(raw, v, bias_smem);      // backward tiles
    if (has_bias && want_mask && relu) return epi_affine<true, true, true>(raw, v, bias_smem);            // training: conv, Linear + ReLU
    if (has_bias && !want_mask && relu) return epi_affine<true, false, true>(raw, v, bias_smem);          // inference: the same
    if (has_bias && !want_mask && !relu) return epi_affine<true, false, false>(raw, v, bias_smem);        // base-node conv, second Linear
    // anything else (a stored mask without ReLU ...): flags as run-time values
    unsigned mask = 0;
#pragma unroll
    for (int j4 = 0; j4 < 8; ++j4) {
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (has_bias) asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b4.x), "=f"(b4.y), "=f"(b4.z), "=f"(b4.w) : "r"(bias_smem + 16u * j4));
        const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int j = j4 * 4 + e;
            float x = fmaf(__uint_as_float(raw[j]), TC_W_UNSCALE, bb[e]);
            if (want_mask && x > 0.f) mask |= 1u << j;
            if (relu) x = fmaxf(x, 0.f);
            v[j] = x;
        }
    }
    return mask;
}

// L1 prefetches of what the epilogue of one step reads from global memory (bias quarter lines, stored ReLU bit masks of the
// 128 rows): issued by the scheduler warp when the item is published, one or two items before the epilogue gets there.
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ void stack_prefetch_step(const TileHdr& t, const BufTable& bt, const int row0, const int64_t Bp, const int lane) {
    if (t.bias_buf >= 0 && lane < 4) prefetch_l1((const float*)bt.p[t.bias_buf] + t.bias_off + 32 * lane);
    if (t.posmask_buf >= 0 && lane < 16)
        prefetch_l1(reinterpret_cast<const uint32_t*>(bt.p[t.posmask_buf]) + ((int64_t)t.posmask_slot * Bp + row0) * 4 + 32 * lane);
    if (t.out2_buf >= 0 && t.out2_mask_kind == MK_BITS && lane >= 16)
        prefetch_l1(reinterpret_cast<const uint32_t*>(bt.p[t.out2_mask_buf]) + ((int64_t)t.out2_mask_slot * Bp + row0) * 4 + 32 * (lane - 16));
}

// Completion signal of an item, deferred by its group leader: waiting for the item's last TMA stores to land costs a store
// round trip (~1.5 k cycles) that nothing in the group overlaps.  The leader therefore keeps the counter address and publishes
// it (a) at once when it would idle anyway - the next step's accumulator is not complete yet, or the item queue is empty -
// and (b) otherwise right after the next step's accumulator read-back, when the stores have long landed.  (Deferring to
// the END of the next step was measured before: it added an item time to every dependency chain.)
__device__ __forceinline__ void stack_flush_signal(uint32_t*& pending) {
    if (pending) {
        tma_store_wait_all();
        stack_signal(pending);
        pending = nullptr;
    }
}

// One step of an item through one epilogue group (cf. tc_epilogue_q).  `sig`: completion counter of the item (last step only).
// PRIV: the program has thread-private fp32 tensors (backward launches of the MS-HGNN models); the forward instantiation carries
// none of that code - at the 96-register cap of a 608-thread CTA a few more live values cost every path 10 % and more.
template <bool PRIV>
__device__ __forceinline__ void stack_epilogue(const TileHdr& t, const BufTable& bt, const BufRows& br, const CUtensorMap* map_k,
                                               const uint32_t tmem_acc, const int row0, const int64_t B, const int64_t Bp,
                                               const int warp, const int lane, const int grp, const StackEpi es, uint32_t& res_count,
                                               uint32_t* sig, uint32_t*& pending, char* const ws, const bool dbg_bare = false, const int dbg = 0) {
    const int q = warp & 3;                        // TMEM lane quarter this warp may access (hardware rule: warp index mod 4)
    const bool leader = q == 2 && lane == 0;       // first warp of the group (warps 2 + 4g .. 5 + 4g): warp index = 2 mod 4
    const int rl = q * 32 + lane;                  // row inside the tile
    const int64_t row = (int64_t)row0 + rl;
    const bool live = row < B;
    const bool all_live = (int64_t)row0 + TILE_M <= B;
    const uint32_t rsw = (uint32_t)((rl >> 1) & 3);     // SWIZZLE_64B: 16-byte chunk index ^= address bits [7, 9)
    const uint32_t tile = es.stg + (uint32_t)rl * 64u;
    // Thread-private fp32 tensors (Tile::priv): a [128 rows x 32 columns] quarter is stored as eight 2 KB chunks, chunk j = the
    // 16 bytes (columns 4j .. 4j + 3) of every row - each thread owns 16 bytes of every chunk, a warp reads / writes 512
    // contiguous bytes, and the quarter (16 KB, contiguous) comes back with ONE bulk copy.  The 64 KB of a (node slot, row tile)
    // occupy the rows of the slot's hi image (quarters 0, 1) and lo image (quarters 2, 3).
    const bool res_priv = PRIV && (t.priv & TILE_RES_PRIV) != 0, out_priv = PRIV && (t.priv & TILE_OUT_PRIV) != 0;
    // (Reading a private residual straight into registers - eight coalesced 128-bit loads per thread instead of the bulk copy through
    // the staging tiles - was measured: +10 % on the backward launch, and the 32 extra live registers at the 96-register cap cost the
    // forward launch 12 % as well.)
    auto priv_quarter = [&](const int buf, const int slot) -> char* {
        return ws + ((size_t)((grp < 2 ? br.hi[buf] : br.lo[buf]) + (int)((int64_t)slot * Bp) + row0) << 8) + (size_t)(grp & 1) * 16384u;
    };
    const bool has_out = t.out_buf >= 0 && !out_priv, has_out2 = t.out2_buf >= 0 && !((dbg & 256) && t.out_buf >= 0), has_res = t.res_buf >= 0 && !dbg_bare && !(dbg & 512);
    const bool res_staged = has_res;
    const bool want_mask = t.relu || t.mask_out_buf >= 0;
    const bool writes_stage = has_out || has_out2 || t.stage_out;
    const int col0 = grp * 32;
    if (dbg_bare) {                                // ablation: accumulator handshake, staged-operand handshake and completion signal only
        mbar_wait(es.accum_bar, es.acc_parity);
        tc_fence_after();
        tc_fence_before();
        mbar_arrive(es.free_bar);
        group_bar_sync(grp);
        if (leader && t.stage_out) mbar_arrive(es.stage_bar);
        if (leader && sig) stack_signal(sig);
        return;
    }

    auto fetch_residual = [&]() {
        mbar_expect_tx(es.res_bar, 2u * 8192u);
        if (PRIV && res_priv) {
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(es.stg),
                         "l"(priv_quarter(t.res_buf, t.res_slot)), "r"(16384u), "r"(es.res_bar)
                         : "memory");
            return;
        }
        const int r_hi = br.hi[t.res_buf] + (int)((int64_t)t.res_slot * Bp) + row0, r_lo = br.lo[t.res_buf] + (int)((int64_t)t.res_slot * Bp) + row0;
        tma_load_2d(es.stg, map_k, es.res_bar, col0, r_hi);
        tma_load_2d(es.stg + 8192, map_k, es.res_bar, col0, r_lo);
    };
    if (leader) {
        tma_store_wait_read();                     // the staging tiles may still feed this group's previous TMA stores
        // early fetch (hidden behind the MMAs of this step); the item is only published to this warp once its input
        // dependency - the residual is an output of the previous phase - has been seen satisfied by the producer warp
        if (res_staged && !t.a_stage) {
            asm volatile("fence.proxy.async.global;" ::: "memory");
            fetch_residual();
        }
    }
    // global reads of this step (L1-prefetched by the scheduler warp), issued before the accumulator wait.  Bias: lane j of
    // EVERY warp fetches column col0 + j and the warp keeps its own 128-byte copy in shared memory (read back as broadcasts):
    // no barrier between warps, no dependent global round trip in front of the arithmetic.  Measured alternatives: per-lane
    // values + 32 shuffles per warp and step (slower: SHFL shares the crossbar the MMA operand reads saturate), eight
    // warp-uniform 128-bit global loads inside the loop (slower in the forward pass, which has the biases).
    const bool has_bias = t.bias_buf >= 0;
    const float bias_l = has_bias ? __ldg((const float*)bt.p[t.bias_buf] + t.bias_off + col0 + lane) : 0.f;
    uint32_t pm = ~0u, m2 = ~0u;
    if (live && t.posmask_buf >= 0) pm = __ldg(reinterpret_cast<const uint32_t*>(bt.p[t.posmask_buf]) + ((int64_t)t.posmask_slot * Bp + row) * 4 + grp);
    if (live && has_out2 && t.out2_mask_kind == MK_BITS)
        m2 = __ldg(reinterpret_cast<const uint32_t*>(bt.p[t.out2_mask_buf]) + ((int64_t)t.out2_mask_slot * Bp + row) * 4 + grp);
    if (leader && pending && !mbar_test(es.accum_bar, es.acc_parity)) stack_flush_signal(pending);     // idle anyway

    mbar_wait(es.accum_bar, es.acc_parity);
    tc_fence_after();
    uint32_t raw[32];
    tmem_ld32(tmem_acc + ((uint32_t)(q * 32) << 16) + col0, raw);
    tmem_ld_wait();
    tc_fence_before();
    mbar_arrive(es.free_bar);                      // this thread's part of the accumulator is in registers
    if (leader) stack_flush_signal(pending);       // the previous item's stores landed long ago
    if (res_staged) {
        // chained step: the staging tiles were the A operand of THIS step's MMAs, which have completed by now
        if (t.a_stage && leader) fetch_residual();
        mbar_wait(es.res_bar, res_count & 1u);
        ++res_count;
    }
    float v[32];
    if (has_bias) {
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(es.bias + 4u * lane), "f"(bias_l) : "memory");
        __syncwarp();
    }
    const unsigned mask = epi_affine_any(has_bias, want_mask, t.relu != 0, raw, v, es.bias);
    if (t.posmask_buf >= 0) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = ((pm >> j) & 1u) ? v[j] : 0.f;
    }
    // (discard.global.L2 of the consumed quarter - a residual-only dh is dead once read - was tried: ncu counted 2.11 GB of DRAM writes
    // against 2.21 GB without it, and the CCTL + error-barrier sequence it compiles to held 9 % of the warp samples.  Dropped.)
    if (PRIV && has_res && res_priv) {
        // fp32 residual: this thread's 16 bytes of each of the eight chunks; the chunks overlap OTHER threads' output bytes, so
        // every thread of the group has to be done reading before the first staging write (barrier below)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint4 r = lds128(es.stg + (uint32_t)j * 2048u + (uint32_t)rl * 16u);
            v[4 * j] += __uint_as_float(r.x); v[4 * j + 1] += __uint_as_float(r.y); v[4 * j + 2] += __uint_as_float(r.z); v[4 * j + 3] += __uint_as_float(r.w);
        }
    }
    if (has_res && !res_priv) {
        // image residual: read in place (the bytes this thread overwrites with its own result below)
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            const uint32_t a = tile + ((((uint32_t)g) ^ rsw) << 4);
            join8_add(v + g * 8, lds128(a), lds128(a + 8192));
        }
    }
    if (PRIV && out_priv) {
        float4* const o = reinterpret_cast<float4*>(priv_quarter(t.out_buf, t.out_slot) + (size_t)rl * 16u);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j * 128] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    }
    // the leader has seen the previous stores of this group read the staging tiles (has_res: the residual has landed in them)
    if (!has_res || res_priv || (dbg & 32)) group_bar_sync(grp);
    if (writes_stage) {
        const bool dead = !all_live && !live;       // rows [B, Bp) of every image stay zero
        if (!has_out && has_out2) {
            // the only staged output is the masked one: clear the masked-off columns as fp32 values (one select per element;
            // clearing the packed fp16 lanes of the hi and the lo image afterwards cost ~ 3.5 instructions per element)
            const uint32_t keep = dead ? 0u : m2;
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = ((keep >> j) & 1u) ? v[j] : 0.f;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const uint32_t a = tile + ((((uint32_t)g) ^ rsw) << 4);
                uint4 hi, lo;
                split8(v + g * 8, hi, lo);
                sts128(a, hi);
                sts128(a + 8192, lo);
            }
        } else {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const uint32_t a = tile + ((((uint32_t)g) ^ rsw) << 4);
                uint4 hi, lo;
                split8(v + g * 8, hi, lo);
                if (dead) { hi = make_uint4(0u, 0u, 0u, 0u); lo = hi; }
                sts128(a, hi);
                sts128(a + 8192, lo);
            }
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
        if (t.stage_out) mbar_arrive(es.stage_bar);        // this quarter of the next step's A operand is in place
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
    if (leader && sig) pending = sig;              // published by stack_flush_signal (see there)
    if (leader && (dbg & 16)) stack_flush_signal(pending);
}

template <bool PRIV>
__global__ void __launch_bounds__(SK_THREADS, 1)
k_tc_stack(const __grid_constant__ TcMaps maps, const Tile* __restrict__ tiles, const StackItem* __restrict__ items,
           const __grid_constant__ StackArgs args, const BufTable bt, const BufRows br) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(16) float bias_w[16][32];        // one copy per epilogue warp
    // Items are handed out dynamically: the scheduler warp (warp 18) draws the next global item index from an atomic counter
    // (so no CTA falls behind: the dependency of an item always points at items that are finished or running), decodes it,
    // waits for its input dependency and then publishes the decoded item to the other roles through this queue.  Decode,
    // dependency round trips and descriptor loads are thereby off the critical path of the single-thread TMA / MMA roles.
    __shared__ int4 q_ent[SK_QUEUE][2];                   // {row tile, phase, first tile, steps}, {per step one byte: chunks | a_stage << 4, -, -, -}
    __shared__ int4 q_chunk[SK_QUEUE][SK_QCHUNKS];        // operand rows of the item's chunks (stack_chunk_desc)
    __shared__ int4 q_hdr[SK_QUEUE][SK_QSTEPS][SK_HDR16]; // tile headers of the item's steps: the epilogue never waits for a descriptor load
    __shared__ volatile int q_count;                      // entries published
    __shared__ volatile int q_prod;                       // entries the TMA producer has started

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SK_PIPE_BYTES + SK_STG_BYTES);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + SK_STAGES), acc_full0 = smem_u32(bars + 2 * SK_STAGES),
                   acc_free0 = smem_u32(bars + 2 * SK_STAGES + SK_ACCS), res_bar = smem_u32(bars + 2 * SK_STAGES + 2 * SK_ACCS),   // 4 residual barriers
                   stage_bar = smem_u32(bars + 2 * SK_STAGES + 2 * SK_ACCS + 4);
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t stg_base = smem_base + SK_PIPE_BYTES;

    if (tid == 0) {
        for (int s = 0; s < SK_STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        for (int a = 0; a < SK_ACCS; ++a) { mbar_init(acc_full0 + 8 * a, 1); mbar_init(acc_free0 + 8 * a, 512); }
        for (int g = 0; g < 4; ++g) mbar_init(res_bar + 8 * g, 1);
        mbar_init(stage_bar, 4);
        q_count = 0; q_prod = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(&tmem_base_s), SK_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    constexpr int SPC = H / SK_KB;                 // pipeline steps (K blocks) per chunk
    const StackProg& pg = args.prog;
    const int NT = args.n_row_tiles, RC = args.delay, n_total = args.n_total, split = args.split;
    const int64_t Bp = args.Bp;
    uint32_t* const err = args.err;
    // Programmatic dependent launch: everything above ran while the previous kernel of the stream was still draining
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    // consumer side of the queue: the n-th item of this CTA (a.w = 0 steps: no more work)
    auto next_item = [&](const int n, int4& a, int4& b) {
        if (lane == 0) { while (q_count <= n) { } }
        __syncwarp();
        a = q_ent[n % SK_QUEUE][0];
        b = q_ent[n % SK_QUEUE][1];
    };

    if (warp == 18) {
        int n_pub = 0;
        for (;;) {
            int cur = 0;
            if (lane == 0) {
                while (n_pub - q_prod >= args.lookahead) { }       // stay close to the producer: a drawn item blocks its dependents
                cur = (int)atomicAdd(args.next, 1u);
            }
            cur = __shfl_sync(0xffffffffu, cur, 0);
            int4 a = make_int4(0, 0, 0, 0), b = make_int4(0, 0, 0, 0), cd = make_int4(0, 0, 0, 0), hd = make_int4(0, 0, 0, 0);
            if (cur < n_total) {
                const ItemRef ir = args.chunked ? stack_decode_chunked(pg, NT, RC, cur) : stack_decode(pg, NT, RC, cur);
                const StackItem it = items[ir.item];
                const int mdl = stack_model(args, ir.row_tile);
                // descriptor loads first, dependency wait second: the two global round trips overlap
                if (lane < SK_QCHUNKS) cd = stack_chunk_desc(tiles, it.tile, it.n_steps, it.meta, lane, br, Bp, mdl * args.w16_rows);
                if (lane < it.n_steps * SK_HDR16)
                    hd = stack_model_hdr(__ldg(reinterpret_cast<const int4*>(tiles + it.tile + lane / SK_HDR16) + lane % SK_HDR16), lane % SK_HDR16,
                                         tiles + it.tile + lane / SK_HDR16, mdl, args);
                if (ir.phase > 0 && it.dep_mask)
                    stack_wait(args.sync + ((size_t)(ir.phase - 1) * NT + ir.row_tile) * args.n_slots, it.dep_mask, lane, err);
                a = make_int4(ir.row_tile, ir.phase, it.tile, it.n_steps);
                b = make_int4(it.meta, it.out_slot, 0, 0);
            }
            if (lane < SK_QCHUNKS && a.w) q_chunk[n_pub % SK_QUEUE][lane] = cd;
            if (lane < a.w * SK_HDR16) q_hdr[n_pub % SK_QUEUE][lane / SK_HDR16][lane % SK_HDR16] = hd;
            __syncwarp();
            for (int s = 0; s < a.w; ++s) stack_prefetch_step(*reinterpret_cast<const TileHdr*>(q_hdr[n_pub % SK_QUEUE][s]), bt, a.x * TILE_M, Bp, lane);
            if (lane == 0) {
                q_ent[n_pub % SK_QUEUE][0] = a;
                q_ent[n_pub % SK_QUEUE][1] = b;
                __threadfence_block();
                q_count = n_pub + 1;
            }
            ++n_pub;
            if (cur >= n_total) break;
        }
    } else if (warp == 0) {
        uint32_t g = 0;                        // pipeline step counter, runs across items
        for (int n = 0;; ++n) {
            int4 qa, qb;
            next_item(n, qa, qb);
            if (qa.w == 0) break;
            if (lane == 0) {
                q_prod = n + 1;
                // the scheduler warp has acquired the completion of this item's inputs; they were written with TMA stores
                // (async proxy) and are read below with TMA loads (async proxy)
                asm volatile("fence.proxy.async.global;" ::: "memory");
                const int row0 = qa.x * TILE_M;
                const int4* qc = q_chunk[n % SK_QUEUE];
                for (int s = 0; s < qa.w; ++s) {
                    const int n_chunks = (qb.x >> (8 * s)) & 0xf, a_stage = (qb.x >> (8 * s + 4)) & 1;
                    for (int c = 0; c < n_chunks; ++c) {
                        const bool from_stage = a_stage && c == 0;
                        const int4 d = *qc++;
                        const int arow_hi = d.x + row0, arow_lo = d.y + row0, w16_row = d.z;
                        const uint32_t tx_bytes = (uint32_t)((from_stage ? 1 : 2) * (split ? 2 : 1) * SK_TILE_BYTES);
                        for (int kb = 0; kb < SPC; ++kb, ++g) {
                            const uint32_t s4 = g % SK_STAGES;
                            mbar_wait(empty0 + 8 * s4, ((g / SK_STAGES) & 1) ^ 1);
                            const int kcol = kb * SK_KB;
                            const uint32_t st = smem_base + s4 * SK_STAGE_BYTES;
                            const uint32_t fb = full0 + 8 * s4;
                            mbar_expect_tx(fb, tx_bytes);
                            if (!from_stage) tma_load_2d(st, &maps.o, fb, kcol, arow_hi);
                            tma_load_2d(st + 2 * SK_TILE_BYTES, &maps.o, fb, kcol, br.w_hi + w16_row);
                            if (split) {
                                if (!from_stage) tma_load_2d(st + SK_TILE_BYTES, &maps.o, fb, kcol, arow_lo);
                                tma_load_2d(st + 3 * SK_TILE_BYTES, &maps.o, fb, kcol, br.w_lo + w16_row);
                            }
                        }
                    }
                }
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        uint32_t g = 0, k = 0, n_staged = 0;
        for (int n = 0;; ++n) {
            int4 qa, qb;
            next_item(n, qa, qb);
            if (qa.w == 0) break;
            if (lane == 0) {
                for (int s = 0; s < qa.w; ++s, ++k) {
                    const int n_chunks = (qb.x >> (8 * s)) & 0xf, a_stage = (qb.x >> (8 * s + 4)) & 1;
                    const uint32_t a = k % SK_ACCS;
                    mbar_wait(acc_free0 + 8 * a, ((k / SK_ACCS) & 1) ^ 1);      // the epilogue has drained this accumulator
                    tc_fence_after();
                    const uint32_t d0 = tmem_base + a * 128;
                    for (int c = 0; c < n_chunks; ++c) {
                        const bool from_stage = a_stage && c == 0;
                        if (from_stage) {
                            mbar_wait(stage_bar, n_staged & 1);   // the four quarters of the previous step's result are staged
                            ++n_staged;
                            tc_fence_after();
                        }
                        for (int kb = 0; kb < SPC; ++kb, ++g) {
                            const uint32_t s4 = g % SK_STAGES;
                            mbar_wait(full0 + 8 * s4, (g / SK_STAGES) & 1);
                            tc_fence_after();
                            const uint32_t st = smem_base + s4 * SK_STAGE_BYTES;
                            const uint64_t w_hi = smem_desc_sw128(st + 2 * SK_TILE_BYTES), w_lo = smem_desc_sw128(st + 3 * SK_TILE_BYTES);
#pragma unroll
                            for (int ks = 0; ks < SK_KB / 16; ++ks) {
                                uint64_t a_hi, a_lo;
                                if (from_stage) {
                                    // the staged operand keeps the epilogue's layout: four 32-column SWIZZLE_64B blocks (one per group)
                                    const uint32_t blk = stg_base + (uint32_t)(kb * (SK_KB / 32) + (ks >> 1)) * 16384u;
                                    a_hi = smem_desc_sw64(blk) + (uint64_t)((ks & 1) * 2);
                                    a_lo = smem_desc_sw64(blk + 8192u) + (uint64_t)((ks & 1) * 2);
                                } else {
                                    a_hi = smem_desc_sw128(st) + (uint64_t)(ks * 2);
                                    a_lo = smem_desc_sw128(st + SK_TILE_BYTES) + (uint64_t)(ks * 2);
                                }
                                const uint64_t adv = (uint64_t)(ks * 2);      // +32 bytes (16 fp16) along K inside the swizzle atom
                                umma_f16(d0, a_hi, w_hi + adv, TC_IDESC, (c | kb | ks) ? 1u : 0u);
                                if (split) {
                                    umma_f16(d0, a_lo, w_hi + adv, TC_IDESC, 1u);
                                    umma_f16(d0, a_hi, w_lo + adv, TC_IDESC, 1u);
                                }
                            }
                            umma_commit(empty0 + 8 * s4);
                        }
                    }
                    umma_commit(acc_full0 + 8 * a);
                }
            }
            __syncwarp();
        }
    } else {
        // group g (warps 2 + 4g .. 5 + 4g) drains column quarter g of every step
        const int grp = (warp - 2) >> 2;
        const bool sig_leader = (warp & 3) == 2 && lane == 0;
        StackEpi es;
        es.stg = stg_base + grp * 16384; es.bias = smem_u32(bias_w[warp - 2]); es.res_bar = res_bar + 8 * grp; es.stage_bar = stage_bar;
        uint32_t k = 0, n_res = 0;
        uint32_t* pending = nullptr;               // group leader: completion counter of the last item, not yet published
        for (int n = 0;; ++n) {
            int4 qa, qb;
            if (lane == 0) { while (q_count <= n) { if (sig_leader) stack_flush_signal(pending); } }
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
                stack_epilogue<PRIV>(t, bt, br, &maps.k, tmem_base + a * 128, qa.x * TILE_M, live_end, Bp, warp, lane, grp, es, n_res,
                                     s == qa.w - 1 ? ctr : nullptr, pending, args.ws);
            }
        }
        if (sig_leader) { stack_flush_signal(pending); tma_store_wait_all(); }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, SK_TMEM_COLS);
    }
}

}  // namespace mshgnn
