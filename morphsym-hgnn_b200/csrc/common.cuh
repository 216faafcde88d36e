// Internal structures shared by the plan builder (host) and the kernels (device).
//
// Data layout in HBM ("node-slot-major slabs"): every activation buffer is
//   slab[slot][row = graph][H]   (fp32, H = 128, rows padded to Bp = multiple of 128)
// where a slot is one node of the per-graph morphology template (K4 Mini Cheetah: 4 base +
// 12 joint + 4 foot = 20 slots).  All rows of a 128-row tile therefore belong to the same
// template node, so the reference's gather / scatter-add over edge_index
// (torch_geometric GraphConv, SURVEY 3.3) becomes "pick which slot tile feeds which weight":
// a compile-time table, no index tensors, no atomics.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace mshgnn {

constexpr int H = 128;
constexpr int MAX_CHUNKS = 8;
constexpr int MAX_BUFS = 128;
constexpr int TILE_M = 128;
constexpr int DEC_MAXC = 8;     // max decoder width
constexpr float LO_SCALE = 1.f; // scale of the low half of a (hi, lo) fp16 pair: lo = fp16((v - hi) * LO_SCALE)

enum AKind : int { A_SLAB = 0, A_EXT = 1 };
enum MaskKind : int { MK_NONE = 0, MK_BITS = 1 };

// base pointers resolved per call (buffer id -> device pointer)
struct BufTable {
    void* p[MAX_BUFS];
};

// One K-chunk of a row-GEMM: D[rows,128] += A[rows,K] * Wt[K,128]
struct Chunk {
    int a_kind;      // A_SLAB: fp32 slab tile; A_EXT: caller's x tensor (strided rows, f32/f64)
    int a_buf;       // buffer id
    int a_slot;      // slab slot (A_SLAB)
    int K;           // reduction length
    int lda;         // row stride in elements (A_EXT)
    int a_off;       // element offset of row 0 (A_EXT: local_node * in_width)
    int w_buf;       // buffer id of the weight in [K][128] ("k-major") form
    int w_off;       // float offset inside that buffer
    int sign_off;    // float offset into BUF_SIGNS of a [K] +-1 vector, or -1
    int w16_row;     // tensor-core path: first row of this weight's 128x128 fp16 image (W for forward, W^T for dX)
};

constexpr int TILE_RES_PRIV = 1, TILE_OUT_PRIV = 2;
// One 128-row x 128-col output tile of a row-GEMM launch.
struct Tile {
    int n_chunks;
    int out_buf, out_slot;            // primary fp32 slab output (-1: none)
    int bias_buf, bias_off;           // bias [128] (-1: none)
    int relu;                         // relu after bias
    int posmask_buf, posmask_slot;    // multiply by a stored ReLU bitmask after relu (-1: none)
    int res_buf, res_slot;            // residual add (-1: none)
    int mask_out_buf;                 // store bitmask of (pre-activation > 0) at mask_out_slot (-1: none)
    int out2_buf, out2_slot;          // secondary output = result (*) mask (-1: none)
    int out2_mask_kind, out2_mask_buf, out2_mask_slot;
    int mask_out_slot;
    // chained steps of the cross-layer stack kernel (kernels_stack.cuh); zero in every per-layer launch table
    int a_stage;                      // chunk 0 reads its A operand from the staging tiles the previous step of the item left on chip
    int stage_out;                    // the epilogue leaves the (hi, lo) result in the staging tiles for the next step of the item
    int priv;                         // stack programs only: TILE_RES_PRIV / TILE_OUT_PRIV (thread-private fp32 layout of residual-only tensors, kernels_stack.cuh)
    Chunk chunks[MAX_CHUNKS];
};

// ---- cross-layer stack program (kernels_stack.cuh) ----
// A program is a sequence of phases (one per layer).  An item of phase p on row tile r may start once the items of phase
// p - 1 of the same row tile that produce the node slots in its dep_mask have signalled (the dependency structure IS the
// morphology graph: a thigh tile waits for hip, thigh and calf, not for the slow base_transform chains).  An item is 1..3 chained steps (Tile entries, contiguous in the tile table) on one
// 128-row tile; the steps after the first take their A operand from on-chip staging.
constexpr int STACK_MAX_PHASES = 20;
struct StackItem {
    int tile;                         // first step (index relative to the program's first tile)
    int n_steps;                      // 1..3
    int out_slot;                     // node slot whose outputs (h / dh / dc) this item completes in its phase
    int meta;                         // one byte per step: chunks | a_stage << 4 (so the scheduler warp needs no dependent load for them)
    unsigned long long dep_mask;      // node slots of the PREVIOUS phase (same row tile) that must be complete before it starts:
                                      // the slots it reads (operands, residual) and, where buffers ping-pong, the readers of the slot it overwrites
};
struct StackProg {
    int n_phases;
    int items_per_row;                // sum of n_items over the phases
    int first_item[STACK_MAX_PHASES]; // index into the item table
    int n_items[STACK_MAX_PHASES];
};

// One (dC, A) pair of a reduce-over-rows GEMM: dW[128, K] += dC[rows,128]^T * A[rows,K]
struct RPair {
    int d_buf, d_slot;                // dC slab tile
    int a_kind, a_buf, a_slot;        // A operand
    int lda, a_off;                   // A_EXT addressing
    int sign_off;                     // A_EXT sign vector (-1: none)
};

struct RTask {
    int pair_begin, n_pairs;
    int K;                            // full in-width of the weight
    int k0;                           // first in-column handled by this task (tile of 128)
    int want_colsum;                  // also produce column sums of dC (bias gradient)
    int pad[3];
};

// Partial-slot layout of the weight-gradient tasks.  Launches of different sizes use different row-split counts (ws_layout
// fits them to whole waves), so the fp32 partials are packed segment by segment: the tasks [begin[s], begin[s+1]) of one
// launch wrote ns[s] partials each, task t's first slot is base[s] + (t - begin[s]) * ns[s].
constexpr int MAX_PART_SEGS = 20;
struct PartSegs {
    int n;
    int begin[MAX_PART_SEGS + 1];
    int ns[MAX_PART_SEGS];
    int base[MAX_PART_SEGS];
};
#ifdef __CUDACC__
__device__ __forceinline__ void part_lookup(const PartSegs& ps, const int task, int64_t& slot0, int& ns) {
    int s = 0;
    while (s + 1 < ps.n && task >= ps.begin[s + 1]) ++s;
    ns = ps.ns[s];
    slot0 = (int64_t)ps.base[s] + (int64_t)(task - ps.begin[s]) * ns;
}
#endif

// Final reduction of split partials into the flat gradient buffer.
struct OutGroup {
    int kind;                         // 0: weight tile, 1: bias (colsum)
    int n_tasks; int tasks[16];       // tasks whose partials are summed
    int n_outs;  int outs[4];         // float offsets in the gradient buffer that receive the sum
    int K, k0;                        // weight: row stride K and first column
    float scale;
    int pad;
};

// prep: derived weights (transposes, root sums, bias sums)
struct DeriveOp {
    int dst_off;                      // float offset in BUF_DERIVED
    int rows, cols;                   // shape of each source [rows][cols]
    int transpose;                    // dst[c][r] (1) or dst[r][c] (0)
    int n_src; int src_off[8];        // float offsets in params; summed
    int pad[3];
};

// fp16 (hi, lo) image of one 128x128 weight for the tensor-core kernels
struct Derive16Op {
    int dst_row;          // first row of the 128x128 matrix inside the fp16 weight tensor
    int transpose;        // dst[n][k] = src[k][n]
    int n_src;
    int src_off[4];       // float offsets in params, summed
    int pad;
};

// One unit of the tensor-core encoder weight gradient: dW_enc[t][:, k0 : k0 + 64*nkb] += sum over <= 4 slots of type t
// and one row split of dpre[slot]^T (x[slot] * sign[slot]).
struct EncDwUnit {
    int x_buf, lda, K;             // caller's x tensor of the node type, graph-row stride (elements), in-width
    int k0, nkb;                   // first in-column (multiple of 64), number of 64-column blocks (1..3)
    int n_slots;                   // 1..4
    int d_slot[4];                 // slab slot of dpre (BUF_DC1 images)
    int a_off[4];                  // element offset of the slot inside a graph's row block (local node * in_width)
    int sign_off[4];               // BUF_SIGNS offset of the [K] +-1 vector or -1
    int want_colsum;               // also reduce the bias gradient (only the k0 == 0 units)
    int pad;
};

// Units [first, first + count) share (type, k0): the reduce sums their partials into the flat gradient buffer.
struct EncDwGroup {
    int first, count;
    int K, k0, width;              // in-width of the type, first column, valid columns (<= 192)
    int w_off, b_off;              // flat gradient offsets of encoder weight / bias (b_off = -1: no bias in this group)
    int pad;
};

// One node slot of the input gradient dx[t][g * nodes + node, :] = sign[slot] * (dpre0[slot][g] W_enc[t]) (k_tc_encoder_dx,
// k_encoder_dx): every slot of every type has one, in slot order.  A dead slot (need[0][slot] == 0) has no dpre0: its rows are zeros.
struct DxUnit {
    int type, slot, node;          // node type, slab slot, local node inside a graph
    int K, n_kb;                   // in-width of the type, 64-column blocks
    int sign_off;                  // BUF_SIGNS offset of the [K] +-1 vector or -1
    int live;                      // need[0][slot]
    int pad;
};
// the caller's input-gradient tensors dx[t] (NULL: type not requested), graph-major like x[t]
struct DxOut {
    float* p[4];
    int nodes[4];
    int64_t w_off[4];              // flat parameter offset of W_enc[t] (the fp32 kernel)
    int tma;                       // bit t: dx[t] is stored through a tensor map (16-byte rows, tensor-core kernel)
};

// One parameter tensor of a padded plan (kernels_pad.cuh): [rows, cols] row-major at ext_off of the caller's flat buffer
// (the model's own width) is the top-left block of [rows_i, cols_i] at int_off of the 128-wide internal buffer; the rest
// of the internal tensor is zero.
struct PadSeg {
    int64_t ext_off, int_off;
    int rows, cols, rows_i, cols_i;
};

struct DecoderDesc {
    int n_dec;                        // decoded nodes per graph
    int C;                            // output channels
    int slots[16];                    // slab slot per decoded node
    int w_off, b_off;                 // params offsets
    int sign_off;                     // BUF_SIGNS offset of [n_dec*C] or -1
};

static inline __host__ __device__ int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }

}  // namespace mshgnn
