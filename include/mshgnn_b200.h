/* mshgnn_b200.h - C ABI of the B200-native MS-HGNN forward/backward hot path.
 *
 * The reference (lunarlab-gatech/MorphSym-HGNN) is pure Python and has no FFI: its
 * boundary for this path is the Python object protocol of
 *   src/ms_hgnn/lightning_py/hgnn_k4.py:L10-196      (GRF_HGNN_K4.__init__/forward)
 *   src/ms_hgnn/lightning_py/hgnn_c2.py:L10-189      (GRF_HGNN_C2)
 *   src/ms_hgnn/lightning_py/hgnn_k4_com.py:L10-177  (COM_HGNN_K4), hgnn_c2_com.py, hgnn.py
 *   src/ms_hgnn/lightning_py/gnnLightning.py:L124-151 (loss heads), L258-265 (optimizer)
 * This library sits under the drop-in Python mirror of those classes
 * (morphsym-hgnn_b200/ms_hgnn) and is bound with ctypes (see INTEGRATION.md).
 *
 * Conventions: every entry point returns 0 on success and a negative code on error
 * (text via mshgnn_last_error(), thread-local).  No allocation happens inside compute
 * calls: the caller passes device buffers (torch-allocated).  All compute calls enqueue
 * on the caller's CUDA stream (a cudaStream_t passed as void*) and return immediately.
 * A plan is immutable after creation and may be shared by threads; a workspace may be
 * used by one call at a time.  There is no CPU fallback: without a CUDA device every
 * compute call fails with MSHGNN_ERR_CUDA.
 */
#ifndef MSHGNN_B200_H
#define MSHGNN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSHGNN_MAX_NODE_TYPES 4
#define MSHGNN_MAX_EDGE_TYPES 16

#define MSHGNN_OK              0
#define MSHGNN_ERR_ARG        -1   /* bad argument / unsupported configuration            */
#define MSHGNN_ERR_CUDA       -2   /* CUDA runtime error (including "no device")          */
#define MSHGNN_ERR_WORKSPACE  -3   /* workspace too small                                 */

/* element types of caller buffers */
#define MSHGNN_F32 0
#define MSHGNN_F64 1
#define MSHGNN_I64 2
#define MSHGNN_F16 3   /* node features only (x_dtype of mshgnn_forward / mshgnn_backward): halves the host -> device bytes of a batch */

/* arithmetic modes */
#define MSHGNN_MODE_FP32   0   /* SIMT fp32 FMA everywhere: <=1e-4 parity mode              */
#define MSHGNN_MODE_TC     1   /* tcgen05 tensor-core path, split-fp16 operands (3 MMAs), fp32 accumulate */
#define MSHGNN_MODE_TC_1X  2   /* tcgen05, single fp16 pass (1e-3 on predictions only)      */

/* loss heads (gnnLightning.py:L124-151, gnnLightning_com.py:L96-121) */
#define MSHGNN_LOSS_MSE 0      /* mean((out - y)^2) over every output element               */
#define MSHGNN_LOSS_CE2 1      /* per-row 2-way cross-entropy, mean over rows (customMetrics.py:L6-25) */

/* parameter kinds for mshgnn_param_offset; the flat parameter order equals the reference's
 * named_parameters() order (SURVEY 3.3 state-dict names) */
#define MSHGNN_P_ENC_W   0     /* encoder.lins.<type>.weight   [H, in]   idx = node type      */
#define MSHGNN_P_ENC_B   1     /* encoder.lins.<type>.bias     [H]                            */
#define MSHGNN_P_REL_W   2     /* convs.<l>.convs.<et>.lin_rel.weight [H,H]  idx = edge type  */
#define MSHGNN_P_REL_B   3     /* convs.<l>.convs.<et>.lin_rel.bias   [H]                     */
#define MSHGNN_P_ROOT_W  4     /* convs.<l>.convs.<et>.lin_root.weight [H,H]                  */
#define MSHGNN_P_MLP_W   5     /* base_transform.{0,2}.weight  [H,H]     idx = 0 | 1          */
#define MSHGNN_P_MLP_B   6     /* base_transform.{0,2}.bias    [H]                            */
#define MSHGNN_P_DEC_W   7     /* decoder.weight [C, H]                                       */
#define MSHGNN_P_DEC_B   8     /* decoder.bias   [C]                                          */

typedef struct mshgnn_plan mshgnn_plan;

/* Static description of one model + morphology template.  Everything the reference
 * derives at construction (hgnn_k4.py:L37-144) or reads from the batch
 * (edge_index_dict, SURVEY 3.4 / Appendix A) is given here once; the library compiles it
 * into constant gather tables, so no edge_index is read on the device afterwards. */
typedef struct mshgnn_desc {
    int32_t n_node_types;                                /* <= 4, reference order (base, joint, foot)       */
    int32_t nodes_per_graph[MSHGNN_MAX_NODE_TYPES];      /* e.g. K4: 4, 12, 4                                */
    int32_t in_width[MSHGNN_MAX_NODE_TYPES];             /* feature width per type (900/300/900 ...)         */
    int32_t n_edge_types;                                /* <= 16, metadata order                            */
    int32_t edge_src_type[MSHGNN_MAX_EDGE_TYPES];
    int32_t edge_dst_type[MSHGNN_MAX_EDGE_TYPES];
    int32_t edge_mean[MSHGNN_MAX_EDGE_TYPES];            /* 1: aggr='mean' (gt/gs/center_bb)                 */
    int32_t edge_count[MSHGNN_MAX_EDGE_TYPES];           /* edges per graph                                  */
    const int32_t* edge_src[MSHGNN_MAX_EDGE_TYPES];      /* per-graph local source node index, [edge_count]  */
    const int32_t* edge_dst[MSHGNN_MAX_EDGE_TYPES];      /* per-graph local destination node index           */
    int32_t hidden;                                      /* H: 128; 1..128 with MSHGNN_PLAN_PAD_HIDDEN       */
    int32_t num_layers;                                  /* L >= 1                                           */
    int32_t morph_sym;                                   /* 1: MS-HGNN (shared base MLP + residual), 0: MI-HGNN (ReLU only) */
    int32_t mlp_type;                                    /* node type that goes through base_transform (morph_sym only) */
    int32_t decode_type;                                 /* node type the decoder reads (foot or base)       */
    int32_t out_channels;                                /* decoder width C (1, 2, 3 or 6)                   */
    const float* in_sign[MSHGNN_MAX_NODE_TYPES];         /* per type [nodes_per_graph*in_width] of +-1, NULL = ones (apply_symmetry) */
    const float* out_sign;                               /* [nodes_per_graph[decode_type]*C] of +-1, NULL = ones (ms_foot_decoder / morphological_symmetry_decoder) */
} mshgnn_desc;

/* ---- plan ------------------------------------------------------------------------- */
/* The kernels are 128 channels wide: mshgnn_plan_create takes hidden == 128 only. */
int  mshgnn_plan_create(const mshgnn_desc* desc, mshgnn_plan** plan_out);
/* flags = 0: the same as mshgnn_plan_create.  MSHGNN_PLAN_PAD_HIDDEN: hidden may be 1..128.  Such a model runs on the
 * 128-wide kernels as the model whose weights are its zero-padded copy, and gives bit for bit that model's outputs, loss,
 * input gradients and (the matching sub-blocks of its) parameter gradients.  params / grads stay in the model's own layout
 * ([H, in], [H], [H, H], [C, H] tensors, reported by mshgnn_param_count / mshgnn_param_offset).  For hidden < 128 every
 * forward first copies params into a 128-wide internal buffer in the workspace, and the backward copies the gradients back
 * out of another one: mshgnn_workspace_bytes includes both.  hidden == 128 with the flag is exactly mshgnn_plan_create. */
#define MSHGNN_PLAN_PAD_HIDDEN 1
int  mshgnn_plan_create_ex(const mshgnn_desc* desc, int32_t flags, mshgnn_plan** plan_out);
void mshgnn_plan_destroy(mshgnn_plan* plan);

/* number of fp32 elements of the flat parameter (and gradient) buffer */
int64_t mshgnn_param_count(const mshgnn_plan* plan);
/* offset/numel of one parameter tensor inside the flat buffer (at the model's hidden width) */
int  mshgnn_param_offset(const mshgnn_plan* plan, int32_t kind, int32_t layer, int32_t idx,
                         int64_t* offset_out, int64_t* numel_out);

/* bytes of device workspace needed for B graphs (train != 0 keeps activations for backward) */
int64_t mshgnn_workspace_bytes(const mshgnn_plan* plan, int64_t B, int32_t train, int32_t mode);
/* output rows = B * nodes_per_graph[decode_type], each out_channels wide */
int64_t mshgnn_out_rows(const mshgnn_plan* plan, int64_t B);

/* ---- compute (device pointers; stream = cudaStream_t) --------------------------------
 * x[t]: node features of type t, row-major [B*nodes_per_graph[t], in_width[t]], graph-major
 *       rows (row = g*nodes_per_graph[t] + local), element type x_dtype (F32 or F64).
 * params: flat fp32 parameters.  out: fp32 [mshgnn_out_rows(B), out_channels].
 * Replaces: GRF_HGNN_K4.forward hgnn_k4.py:L146-196 and its C2/COM/MI siblings. */
int mshgnn_forward(const mshgnn_plan* plan, int64_t B,
                   const void* const* x, int32_t x_dtype,
                   const float* params, float* out,
                   void* workspace, int64_t workspace_bytes,
                   int32_t train, int32_t mode, void* stream);

/* Fused loss head: writes the scalar loss to loss_out[0] and d(loss)/d(out) to dout
 * (same shape as out; dout may be NULL for evaluation).  labels: MSE -> same element count
 * as out; CE2 -> one label in {0,1} per output row.  loss_scale multiplies dout (and not
 * loss_out): pass 1/world_size for data-parallel training with a summed all-reduce.
 * Replaces: Base_Lightning.calculate_losses_step gnnLightning.py:L124-139. */
int mshgnn_loss(const mshgnn_plan* plan, int64_t B, int32_t loss_kind,
                const float* out, const void* labels, int32_t label_dtype,
                float loss_scale, float* loss_out, float* dout,
                void* workspace, int64_t workspace_bytes, void* stream);

/* Backward of mshgnn_forward(train=1) on the same workspace: writes d(loss)/d(params)
 * (every element, zeros for structurally dead branches) into grads[param_count].
 * A padded plan (hidden < 128) reads the parameters that forward copied into the workspace, not `params`.
 * grads == NULL runs the input-only backward of a frozen model: the decoder backward and the dX chain through the
 * layers (everything mshgnn_input_grad reads), without any weight-gradient launch or partial reduction.
 * Replaces: torch autograd through PyG (SURVEY 3.1 "loss.backward()"). */
int mshgnn_backward(const mshgnn_plan* plan, int64_t B,
                    const void* const* x, int32_t x_dtype,
                    const float* params, const float* dout, float* grads,
                    void* workspace, int64_t workspace_bytes,
                    int32_t mode, void* stream);

/* Same, for data-parallel training: every gradient OUTSIDE the encoder block (the encoder parameters come first in the flat
 * buffer; everything from the first convs.* offset on) is final when `layers_ready_event` (a cudaEvent_t, may be NULL) is
 * recorded on `stream` - before the encoder weight gradient, the last launch of the step, runs - so that segment can be
 * all-reduced on another stream underneath it.  Replaces: DDP's bucketed gradient hooks (gnnLightning.py:L1396-1400, devices). */
int mshgnn_backward_staged(const mshgnn_plan* plan, int64_t B,
                           const void* const* x, int32_t x_dtype,
                           const float* params, const float* dout, float* grads,
                           void* workspace, int64_t workspace_bytes,
                           int32_t mode, void* stream, void* layers_ready_event);

/* Input gradient: after mshgnn_backward / mshgnn_backward_staged (with or without grads) on the same workspace and
 * before the next mshgnn_forward on it, writes d(loss)/d(x[t]) into dx[t] - fp32 [B*nodes_per_graph[t], in_width[t]],
 * graph-major like x[t] - for every type whose dx[t] is not NULL.  Every element is written (rows of node slots that
 * cannot reach the output get exact zeros), so dx[t] may be uninitialised memory.  The result does not depend on x_dtype
 * of the forward: cast it to the features' type if needed.  params: the flat parameters of that forward.
 * Replaces: torch autograd into the node features through the encoder and apply_symmetry (hgnn_k4.py:L159-160, L198-237). */
int mshgnn_input_grad(const mshgnn_plan* plan, int64_t B, const float* params, float* const* dx,
                      void* workspace, int64_t workspace_bytes, int32_t mode, void* stream);

/* Fused Adam on flat buffers (torch.optim.Adam defaults semantics, gnnLightning.py:L258-265):
 * step is the 1-based step count after this update. */
int mshgnn_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                     int64_t n, int64_t step, float lr, float beta1, float beta2, float eps,
                     float weight_decay, void* stream);
/* plain SGD: p -= lr * g */
int mshgnn_sgd_step(float* params, const float* grads, int64_t n, float lr, void* stream);

/* ---- device-side window builder (SURVEY 8f-3) ---------------------------------------------
 * Replaces, batched on the GPU, the reference's per-sample dataset path
 *   LinTzuYaunDataset.load_data_at_dataset_seq        datasets_py/LinTzuYaunDataset.py:L66-88
 *   LinTzuYaunDataset_Morph.load_data_sorted_k4/_c2   datasets_py/LinTzuYaunDataset_Morph.py:L156-347
 *   ..._Morph.get_helper_heterogeneous_gnn(_c2)       datasets_py/LinTzuYaunDataset_Morph.py:L555-697
 *   FlexibleDataset.get_helper_heterogeneous_gnn      datasets_py/flexibleDataset.py:L537-607
 * plus torch_geometric's collate of the node features and labels (SURVEY 3.4).
 * seq: device [n_rows, seq_cols] row-major, every raw channel array side by side in dataset column order.
 * Graph g is the window of rows [starts[g], starts[g] + history_length).  A node row of type t is
 * blocks_per_node[t] blocks of block_len[t] values; block (t, node, k) - index first(t) + node*blocks + k
 * in block_col / block_sign - holds column block_col[.] of the window over time (the reference's
 * flatten('F')), z-scored per window when normalize != 0 (mean, Bessel std, NaN -> 0:
 * flexibleDataset.py:L388-396), times block_sign[.] (+-1: the datasets' apply_symmetry,
 * LinTzuYaunDataset_Morph.py:L349-408, commutes with the z-score).  block_col < 0 with block_len 1 is
 * the constant feature of a type without variables (value block_sign, 1 in the reference).
 * Labels: y[g, i] = label_seq[starts[g] + history_length - 1, label_col[i]] * label_sign[i].
 * starts is a DEVICE pointer; entries are clamped into [0, n_rows - history_length]. */
typedef struct mshgnn_window_desc {
    int32_t history_length;
    int32_t seq_cols;
    int32_t label_cols;
    int32_t n_node_types;
    int32_t nodes_per_graph[MSHGNN_MAX_NODE_TYPES];
    int32_t blocks_per_node[MSHGNN_MAX_NODE_TYPES];
    int32_t block_len[MSHGNN_MAX_NODE_TYPES];      /* history_length, or 1 for the constant feature */
    int32_t normalize;
    int32_t n_labels;
    const int32_t* block_col;                      /* host, [sum_t nodes*blocks] */
    const int32_t* block_sign;                     /* host, same shape; NULL = ones */
    const int32_t* label_col;                      /* host, [n_labels] */
    const int32_t* label_sign;                     /* host, [n_labels]; NULL = ones */
} mshgnn_window_desc;

int mshgnn_build_windows(const mshgnn_window_desc* desc, const void* seq, const void* label_seq, int32_t seq_dtype,
                         int64_t n_rows, const int64_t* starts, int64_t B, float* const* x, float* y, void* stream);

/* ---- fused step metrics (SURVEY 8f-2) -------------------------------------------------------
 * Everything Base_Lightning.calculate_losses_step derives from (y_pred, y) besides the loss gradient
 * (gnnLightning.py:L124-151, L285-348; customMetrics.py:L6-54), without a host sync:
 *   MSHGNN_LOSS_CE2: n = graphs, out [n*feet, 2] logits, labels [n, feet] in {0,1}
 *     slots 0 CE sum, 1 rows, 2 graphs whose 16-class argmax is right, 3 graphs, 4+4*leg+{0,1,2,3} = tp fp fn tn,
 *     20 CE mean (fp32-rounded), 21 16-class accuracy, 22..25 binary F1 of leg 0..3 (NaN -> 0)
 *   MSHGNN_LOSS_MSE: n = elements; slots 0 sum sq. err, 1 sum abs. err, 2 n, 20 MSE, 21 RMSE, 22 L1
 * batch[MSHGNN_METRIC_SLOTS] receives this call's values; slots 0..19 are also ADDED to epoch[] when it is not NULL
 * (torchmetrics' dist_reduce_fx="sum" states).  scratch: MSHGNN_METRIC_SCRATCH doubles of device memory. */
#define MSHGNN_METRIC_SLOTS   32
#define MSHGNN_METRIC_SCRATCH (296 * 32)
int mshgnn_step_metrics(int32_t loss_kind, int64_t n, int32_t feet, const float* out, const void* labels, int32_t label_dtype,
                        double* batch, double* epoch, double* scratch, void* stream);

/* Two more metric kinds, through mshgnn_step_metrics_ex (same batch / epoch / scratch contract as above; n = graphs):
 *   MSHGNN_METRIC_COM: COM_Base_Lightning.calculate_losses_step (gnnLightning_com.py:L70-95).  out, labels [n, n_base*6]
 *     (standardised, per base lin[3] then ang[3]); args: n_base, y_mean[6], y_std[6] (fp64, device).
 *     slots 0 sum sq. err, 1 elements, 2 sum sq. err of the lin halves, 3 of the ang halves, 4 elements of one half,
 *     5 sum over rows of the cosine similarity of the un-standardised (y * std + mean) lin 3-vectors of base 0, 6 the same
 *     for ang, 7 rows; 20 MSE, 21 RMSE, 22 MSE lin, 23 MSE ang, 24 cos_sim_lin, 25 cos_sim_ang, 26 (cos_sim_lin + cos_sim_ang) / 2.
 *     Cosine similarity is torch.nn.functional.cosine_similarity(pred, label, dim=1, eps=1e-8): each vector divided by
 *     max(norm, eps), so a zero vector scores 0.
 *   MSHGNN_METRIC_GRF_WORLD: HGNN_C2_Lightning_Reg.calculate_losses_step_worldframe (gnnLightning.py:L287-311).  out, labels
 *     [n, 12] (4 feet x 3, body frame); args: quat [n, 4] (x, y, z, w; normalised here), quat_dtype MSHGNN_F32 | MSHGNN_F64, z_only.
 *     slots 0 sum sq. err, 1 sum abs. err, 2 elements (body frame, as MSHGNN_LOSS_MSE), 3, 4, 5 the same after rotating each
 *     foot's force by R(q)^T (with z_only: over the z components 2, 5, 8, 11 only); 20 MSE, 21 RMSE, 22 L1 (body frame),
 *     23 MSE, 24 RMSE, 25 L1 (world frame).
 * Arithmetic is fp64.  MSHGNN_ERR_ARG: n_base outside 1..4 or a NULL stat for COM, NULL quaternions for world frame. */
#define MSHGNN_METRIC_COM       2
#define MSHGNN_METRIC_GRF_WORLD 3
typedef struct {
    int32_t n_base;          /* COM: bases per graph, 1..4                              */
    const double* y_mean;    /* COM: [6] standardiser mean (device)                     */
    const double* y_std;     /* COM: [6] standardiser std (device)                      */
    const void* quat;        /* GRF world frame: [n, 4] body orientation (device)       */
    int32_t quat_dtype;      /* GRF world frame: MSHGNN_F32 or MSHGNN_F64               */
    int32_t z_only;          /* GRF world frame: world-frame sums over z components only */
} mshgnn_metric_args;
int mshgnn_step_metrics_ex(int32_t kind, const mshgnn_metric_args* args, int64_t n, const float* out, const void* labels,
                           int32_t label_dtype, double* batch, double* epoch, double* scratch, void* stream);

/* JSON summary of the compiled tables (slots, liveness, gather lists); returns the bytes needed
 * (including the terminating NUL).  Host-only: usable without a GPU. */
int64_t mshgnn_plan_describe(const mshgnn_plan* plan, char* buf, int64_t cap);

/* ---- per-kernel timing (CUDA events on the launching stream) -----------------------------
 * While enabled, every kernel launch of this library is bracketed by a pair of CUDA events on the
 * stream it is launched on.  mshgnn_profile_read synchronises those events, adds the elapsed
 * milliseconds and launch counts per kernel kind into ms_out / launches_out (n entries each, n >= 19: the first n
 * kinds) and clears the record.  Used by bench.py for the roofline figures. */
#define MSHGNN_NUM_KERNEL_KINDS 21     /* n = 19 and 20 (the kinds before "dx_encoder" / "pad_params") are accepted too */
int mshgnn_profile_enable(int32_t on);
int mshgnn_profile_read(double* ms_out, int64_t* launches_out, int32_t n);
const char* mshgnn_kernel_kind_name(int32_t kind);

/* number of kernels launched by this library since process start (for gpu_launches accounting) */
/* Introspection for the parity tests: where a training-mode forward left the ReLU sign pattern it took.
 * layer = -1: encoder output; layer = l (0..L-1): slots [0, S) = ReLU of the HeteroConv output of node slot s
 * (hgnn_k4.py:L175-186), slots [S, S + n_mlp) = hidden ReLU of base_transform (hgnn_k4.py:L133-137) of MLP-type node n.
 * Layout at workspace + *byte_off: uint32 [n_slots][*rows_padded][4]; bit (c % 32) of word (c / 32) <=> pre-activation
 * of hidden channel c > 0.  Slots whose value cannot reach the output are never written.  Rows are 128 bits whatever the
 * plan's hidden width: bits c >= hidden of a padded plan are always 0. */
int mshgnn_relu_mask_offset(const mshgnn_plan* plan, int64_t B, int32_t mode, int32_t layer,
                            int64_t* byte_off, int64_t* n_slots, int64_t* rows_padded);

/* Introspection for the host tests: how a training-mode backward of B graphs splits the layer-stack weight-gradient work.
 * For layer launch l (0..L-1) writes out[4*l .. 4*l+3] = {tasks, row splits, rows per split, first partial slot}; returns L
 * (or -1).  One CTA = one task x one row split; partial slots are packed launch by launch in task order.  Host-only. */
int64_t mshgnn_dw_layout(const mshgnn_plan* plan, int64_t B, int32_t mode, int32_t* out, int64_t cap);

/* ---- batching-layout check (SURVEY 3.4) ------------------------------------------------------
 * The kernels never read edge_index (the template is compiled into the plan); this verifies, in ONE launch and without a
 * host synchronisation, that the caller's batch is that template tiled over B graphs, bit-exactly (PyG
 * Batch.from_data_list).  edge_index[e]: device int64 [2][edge_count[e] * B], row-major (row 0 sources, row 1
 * destinations), metadata order.  On a mismatch the kernel stores 1 + (edge type) into *flag - pinned host memory
 * (readable by the host at any later time) or device memory.  Replaces nothing in the reference (PyG trusts the batch);
 * it is the guard that makes "no edge_index on the device" safe. */
int mshgnn_check_edges(const mshgnn_plan* plan, int64_t B, const int64_t* const* edge_index, int32_t* flag, void* stream);

/* ---- switches and status --------------------------------------------------------------------
 * Option "stack" (default 1, environment MSHGNN_STACK=0 turns it off): run the layer loop of the tensor-core modes
 * (hgnn_k4.py:L170-186 and its backward) as ONE persistent cross-layer kernel over L2-resident row chunks instead of one
 * launch per layer.  It changes the workspace layout: query mshgnn_workspace_bytes again after switching.
 * Option "stack_pair" (MSHGNN_STACK_2CTA): the stack launches use the CTA-pair kernel (clusters of two CTAs,
 * tcgen05.mma.cta_group::2 on two row tiles at once; rows are then padded to a multiple of 256 - query the workspace size
 * again after switching): 1 (default) = for batches of >= 6144 graphs, 2 = always, 0 = never (the one-CTA stack kernel).
 * Both choose between implementations that produce identical bits (tests/test_gpu_stack.py).
 * Option "encoder" (MSHGNN_ENCODER=stream|v1|pair): kernel of the encoder forward: -1 (default) = the persistent TMA-fed kernel
 * whenever the feature tensors allow it (fp32, 16-byte rows), 0 = the same, 1 = one row tile per CTA, 2 = two row tiles per CTA;
 * "encoder_tpi" (MSHGNN_ENC_TPI): row tiles per work item of the persistent kernel, 0 = by batch size, 1, 2;
 * "encoder_dw_tma" (MSHGNN_ENC_DW=tma): feature rows of the encoder weight gradient by TMA (1) or register-staged loads (0, default).
 * All of them produce identical bits (tests/test_gpu_stack.py::test_encoder_kernels_are_bit_identical).
 * mshgnn_stack_status copies one word back (synchronising): *status_out = 1 when a dependency wait inside the last stack
 * launch on this workspace timed out (its results are then invalid); used by the tests. */
int mshgnn_set_option(const char* name, int32_t value);
int32_t mshgnn_get_option(const char* name);
int mshgnn_stack_status(const mshgnn_plan* plan, int64_t B, int32_t train, int32_t mode, const void* workspace, int32_t* status_out);
/* Diagnostics (MSHGNN_STACK_TIMING=1 selects an instrumented build of the stack kernel): byte offset in the workspace of
 * uint64 [CTA][16] cycle counters of the LAST stack launch - producer waiting for a ring slot / for a dependency, MMA
 * issuer waiting for operands / a free accumulator / a staged operand, epilogue group 0 waiting for an accumulator,
 * kernel cycles, steps.  -1 when the stack kernel is off. */
int64_t mshgnn_stack_timing_offset(const mshgnn_plan* plan, int64_t B, int32_t train, int32_t mode);

int64_t mshgnn_launch_count(void);
const char* mshgnn_last_error(void);
const char* mshgnn_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MSHGNN_B200_H */
