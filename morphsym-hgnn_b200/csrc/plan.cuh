// Host-side plan: compiles the morphology template + model description into constant
// gather tables (tiles / chunks / reduce tasks) and a workspace layout.
#pragma once
#include <mutex>
#include <string>
#include <vector>

#include "../../include/mshgnn_b200.h"
#include "common.cuh"

namespace mshgnn {

// buffer ids (BufTable / BufRows slots; ws_layout places each one in WsLayout::buf / buf16)
enum : int {
    BUF_PARAMS = 0, BUF_DERIVED = 1, BUF_SIGNS = 2, BUF_GRADS = 3,
    BUF_X0 = 4,                       // +type
    BUF_MASKE = 13,                   // ReLU bitmask of the encoder output

    BUF_H0 = 16,                      // +layer (0..L)
    BUF_CT0 = 32,                     // +layer
    BUF_MASK0 = 48,                   // +layer: ReLU bitmasks, slots [0,S) conv outputs, [S,S+nm) base-MLP hidden
    // backward quantities, one id per layer.  Under the per-layer launch sequence ws_layout aliases them onto two ping-pong
    // buffers (dh_l -> dh[l & 1], dc_l -> dc[(l + 2) & 1], du_l -> du); the cross-layer stack kernel runs the whole dX chain
    // in one launch, before the weight-gradient kernels, so there every layer keeps its own buffer.
    BUF_DHL0 = 64,                    // +l (0..L):  dL/dh_l
    BUF_DCL0 = 81,                    // +l (-1..L-1, i.e. BUF_DCL0 - 1 = dpre of the encoder): dL/dc_l (pre-activation gradients)
    BUF_DUL0 = 96                     // +l (0..L-1): gradient at the hidden ReLU of base_transform
};
constexpr int MAX_LAYERS = 15;
static_assert(BUF_DCL0 - 1 == 80, "kernels_tc.cuh BUF_DC1_ID names the encoder dpre buffer by number");
static_assert(BUF_PARAMS == 0 && BUF_DERIVED == 1, "kernels_tc.cuh BUF_PARAMS_ID / BUF_DERIVED_ID name these buffers by number");

struct Launch { int begin = 0, count = 0; };

// flat parameter layout at one hidden width, reference named_parameters() order
struct ParamLayout {
    int64_t n = 0;
    int64_t enc_w[MSHGNN_MAX_NODE_TYPES] = {0}, enc_b[MSHGNN_MAX_NODE_TYPES] = {0};
    std::vector<int64_t> rel_w, rel_b, root_w;   // [l * n_etypes + e]
    int64_t mlp_w[2] = {-1, -1}, mlp_b[2] = {-1, -1};
    int64_t dec_w = 0, dec_b = 0;
};

struct Plan {
    // ---- description (deep copy) ----
    int n_types = 0, n_etypes = 0, L = 0, morph_sym = 0, mlp_type = -1, dec_type = 0, C = 0;
    // Hidden widths.  The kernels are H = 128 wide: a padded plan (a width < H: MSHGNN_PLAN_PAD_HIDDEN or
    // mshgnn_plan_create_models) runs each model as the 128-wide one whose weights are its zero-padded copy.  Every table
    // below except `ext` refers to that 128-wide internal layout; the caller's params / grads are in `ext`, copied by
    // k_pad_params / k_compact_grads.
    // A plan of mshgnn_plan_create_models with M > 1 describes n_models = M models that differ only in width (a "mixed" plan):
    // model m's layout ext[m] starts at ext_base[m] of the caller's buffer (the layouts laid end to end), its 128-wide
    // internal copy at m * n_params, and the PadSeg table holds absolute offsets for all of them.  Other plans have
    // n_models = 1 and serve a model batch of any M through per-model strides (blockIdx.z of the pad kernels).
    int n_models = 1;
    std::vector<int> hidden;           // [n_models]
    bool padded = false;
    std::vector<ParamLayout> ext;      // [n_models], offsets from the model's own start
    std::vector<int64_t> ext_base;     // [n_models + 1]; ext_base[n_models] = mshgnn_param_count
    std::vector<PadSeg> pad_segs;      // one per parameter tensor and model: every model's encoder block, then every model's rest
    int n_pad_enc = 0;                 // segments [0, n_pad_enc) are the encoder blocks
    int nodes[MSHGNN_MAX_NODE_TYPES] = {0}, in_w[MSHGNN_MAX_NODE_TYPES] = {0};
    int e_src_t[MSHGNN_MAX_EDGE_TYPES] = {0}, e_dst_t[MSHGNN_MAX_EDGE_TYPES] = {0}, e_mean[MSHGNN_MAX_EDGE_TYPES] = {0};
    std::vector<int> e_src[MSHGNN_MAX_EDGE_TYPES], e_dst[MSHGNN_MAX_EDGE_TYPES];

    // ---- slots ----
    int S = 0;                         // slots per graph
    int type_base[MSHGNN_MAX_NODE_TYPES] = {0};
    std::vector<int> slot_type, slot_local;
    int nm = 0;                        // nodes of the MLP type

    // ---- flat parameter layout of the kernels (reference named_parameters order, 128 wide) ----
    int64_t n_params = 0;
    int64_t off_enc_w[MSHGNN_MAX_NODE_TYPES], off_enc_b[MSHGNN_MAX_NODE_TYPES];
    std::vector<int64_t> off_rel_w, off_rel_b, off_root_w;   // [l * n_etypes + e]
    int64_t off_mlp_w[2] = {-1, -1}, off_mlp_b[2] = {-1, -1};
    int64_t off_dec_w = 0, off_dec_b = 0;

    // ---- derived weights layout ----
    int64_t n_derived = 0;
    int64_t der_encT[MSHGNN_MAX_NODE_TYPES];
    std::vector<int64_t> der_relT;                            // [l*n_etypes+e]
    std::vector<int64_t> der_rootT, der_root, der_bias;       // [l*n_types+t]  (-1 when type has no in-edges)
    int64_t der_mlpT[2] = {-1, -1};
    std::vector<DeriveOp> derive_ops;                            // bias sums first (n_derive_bias of them): all the tensor-core modes need
    int n_derive_bias = 0;
    std::vector<Derive16Op> derive16_ops;   // fp16 (hi, lo) weight images for the tensor-core kernels
    int n_mats16 = 0;

    // ---- signs ----
    std::vector<float> signs;          // host copy of BUF_SIGNS
    std::vector<int> sign_off_slot;    // per slot (-1 none)
    int sign_off_out = -1;

    // ---- liveness ----
    std::vector<std::vector<char>> need;   // need[l][slot], l = 0..L

    // ---- compiled tables ----
    std::vector<Tile> tiles;
    Launch enc_launch, enc_train;
    std::vector<Launch> conv_train, conv_infer, mlp1, mlp1_train, mlp2;      // per layer
    std::vector<Launch> bwd_m1, bwd_m2, bwd_dx;                  // per layer
    // cross-layer stack programs (kernels_stack.cuh): tiles [tiles.begin, +count) of `tiles`, items in stack_items
    struct Stack { Launch tiles; int item0 = 0; StackProg prog{}; };
    Stack stack_infer, stack_train, stack_bwd;
    std::vector<StackItem> stack_items;
    std::vector<RTask> rtasks;
    std::vector<RPair> rpairs;
    std::vector<Launch> dw_layer;                                // per layer (task ranges)
    Launch dw_enc;
    std::vector<OutGroup> groups;
    // tensor-core encoder: fp16 weight image [n_types*128][enc_kmax] and weight-gradient units
    int enc_kmax = 64;
    std::vector<EncDwUnit> enc_units;
    std::vector<EncDwGroup> enc_groups;
    int n_groups_layers = 0;           // groups [0, n_groups_layers) belong to the layer stack, the rest to the encoder
    std::vector<DxUnit> dx_units;      // input gradient: one per node slot (mshgnn_input_grad)
    DecoderDesc dec;

    // ---- device copies (lazy) ----
    mutable std::mutex mu;
    mutable bool uploaded = false;
    mutable int device = -1;
    mutable Tile* d_tiles = nullptr;
    mutable StackItem* d_stack_items = nullptr;
    mutable int* d_edge_tpl = nullptr;   // per edge type [src E | dst E] local node indices (k_check_edges)
    mutable RTask* d_rtasks = nullptr;
    mutable RPair* d_rpairs = nullptr;
    mutable OutGroup* d_groups = nullptr;
    mutable DeriveOp* d_derive = nullptr;
    mutable Derive16Op* d_derive16 = nullptr;
    mutable float* d_signs = nullptr;
    mutable EncDwUnit* d_enc_units = nullptr;
    mutable EncDwGroup* d_enc_groups = nullptr;
    mutable DxUnit* d_dx_units = nullptr;
    mutable PadSeg* d_pad_segs = nullptr;
    mutable std::vector<void*> d_allocs;   // every device table above, freed by mshgnn_plan_destroy

    int slot_of(int type, int local) const { return type_base[type] + local; }
};

struct WsLayout {
    // A model batch of M models keeps model m's graphs in rows [m Bm, m Bm + B) of every slab, Bm = B padded to the row-tile
    // granularity of the stack kernel (128, 256 for the CTA-pair kernel), so no row tile belongs to two models.  Bp = M Bm.
    int M = 1;
    int64_t Bm = 0;
    int64_t Bp = 0;
    int n_splits = 1;                  // row splits of the SIMT reduce-GEMM (<= 512 rows each)
    int n_splits_tc = 1, rows_per_tc = 64;   // default row splits of the tcgen05 reduce-GEMM (multiples of 64 rows)
    int dw_ns[MAX_LAYERS], dw_rows[MAX_LAYERS];   // per layer launch: row splits actually used (wave-fitted, see ws_layout)
    PartSegs segs;                     // packed partial slots of the weight-gradient tasks (common.cuh)
    int dw_slot0[MAX_LAYERS];          // first partial slot of each layer launch
    int64_t part_slots = 0;            // slots of one model ([128][128] fp32 weight partial + [128] bias partial each); model m's follow model m-1's
    // Where every buffer id lives (byte offsets into the workspace, -1 when the call has no such buffer).  ws_layout makes
    // every aliasing decision here: several ids may name one buffer (the ping-pong slabs and images).
    int64_t buf[MAX_BUFS];             // fp32: derived weights, slabs (MODE_FP32) and ReLU bitmasks
    int64_t buf16[MAX_BUFS][2];        // tensor-core modes: (hi, lo) fp16 images, index [0] = hi, [1] = lo
    int64_t w16[2] = {-1, -1};         // 128x128 weight images (hi, lo) of the tensor-core modes
    int64_t part_w = 0, part_b = 0, dec_part = 0, loss_part = 0;
    int n_splits_enc = 1, rows_per_enc = 512;          // row splits of the tensor-core encoder weight gradient
    int64_t part_enc_w = -1, part_enc_b = -1;          // [unit][split][128][192] fp32 / [unit][split][128]
    int64_t wenc16[2] = {-1, -1};                      // encoder weight images [n_types*128][enc_kmax] fp16 (hi, lo)
    int stack = 0;                     // the layer loop runs as the cross-layer stack kernel (tensor-core modes)
    int stack_pair = 0;                // the stack launches use the CTA-pair kernel (Bp is a multiple of 256)
    int64_t enc_sync = -1;             // work counter of the persistent encoder (k_tc_encoder_stream), zeroed by the forward prologue
    int64_t stack_sync = -1;           // dependency counters of the stack kernel (uint32 [phases][row tiles]) + error word
    int64_t stack_sync_bytes = 0;
    int64_t pad_params = -1, pad_grads = -1;   // padded plans: 128-wide fp32 parameters (every call) / gradients (training)
    int64_t total = 0;
};

constexpr int DEC_BLOCKS = 1184;     // 148 SMs x 8 resident CTAs of the 2-channel instantiation (48 registers, 8 KB of shared memory; the 8-channel one: 2 per SM): one load in flight per warp, so latency is hidden by warps
constexpr int LOSS_BLOCKS = LOSS_PARTIALS;

// returns error text ("" = ok).  widths empty: one model of width d->hidden; otherwise one model per width (d->hidden ignored)
std::string build_plan(const mshgnn_desc* d, int32_t flags, Plan& p, const std::vector<int>& widths = {});
WsLayout ws_layout(const Plan& p, int64_t B, int train, int mode, int M = 1);   // B graphs per model
bool stack_enabled();                 // cross-layer stack kernel on (default) / off (option "stack")
void set_stack_enabled(int on);
int stack_pair_mode();                // CTA-pair (cta_group::2) stack kernel: 1 = by batch size (default), 2 = always, 0 = never (option "stack_pair")
void set_stack_pair_mode(int v);
std::string describe_plan(const Plan& p);

}  // namespace mshgnn
