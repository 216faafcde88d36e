// Plan builder: morphology template + model description -> constant gather tables.
//
// What the reference does per step with index tensors (torch_geometric HeteroConv/GraphConv
// over batch.edge_index_dict, hgnn_k4.py:L102-130,170-172; SURVEY 3.3/3.4) is resolved here
// ONCE per (model, template): for every destination node slot the list of (source slot,
// weight) contributions, which layers/slots are live (the decoder only reads one node type,
// so last-layer branches into the others are dead, SURVEY 3.3-5), and the transposed pattern
// for the backward pass.
#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <sstream>
#include <utility>
#include <vector>

#include "plan.cuh"

namespace mshgnn {

static Chunk slab_chunk(int buf, int slot, int w_buf, int64_t w_off, int w16_row) {
    Chunk c{};
    c.a_kind = A_SLAB; c.a_buf = buf; c.a_slot = slot; c.K = H; c.lda = H; c.a_off = 0;
    c.w_buf = w_buf; c.w_off = (int)w_off; c.sign_off = -1; c.w16_row = w16_row;
    return c;
}

// registers the fp16 image of sum(srcs) (optionally transposed) and returns its first row in the fp16 weight tensor
static int mat16(Plan& p, const std::vector<int64_t>& srcs, bool transpose) {
    for (const auto& op : p.derive16_ops) {
        if (op.transpose != (int)transpose || op.n_src != (int)srcs.size()) continue;
        bool same = true;
        for (size_t i = 0; i < srcs.size(); ++i) same = same && op.src_off[i] == (int)srcs[i];
        if (same) return op.dst_row;
    }
    Derive16Op op{};
    op.dst_row = p.n_mats16 * H; op.transpose = transpose; op.n_src = (int)srcs.size();
    for (size_t i = 0; i < srcs.size(); ++i) op.src_off[i] = (int)srcs[i];
    p.derive16_ops.push_back(op);
    p.n_mats16++;
    return op.dst_row;
}

static Tile empty_tile() {
    Tile t{};
    t.n_chunks = 0;
    t.out_buf = -1; t.out_slot = 0; t.bias_buf = -1; t.bias_off = 0; t.relu = 0;
    t.posmask_buf = -1; t.posmask_slot = 0; t.res_buf = -1; t.res_slot = 0; t.mask_out_buf = -1; t.mask_out_slot = 0;
    t.out2_buf = -1; t.out2_slot = 0; t.out2_mask_kind = MK_NONE; t.out2_mask_buf = -1; t.out2_mask_slot = 0;
    t.priv = 0;
    return t;
}

constexpr int RD_MAX_PAIRS = 4;

// Emit reduce tasks ("units") of at most RD_MAX_PAIRS pairs each; returns false when more than 16 units result.
// Unit u takes the pairs u, u + U, u + 2U, ... (U = number of units).  Pair lists follow the template's node / edge order,
// i.e. leg by leg, so with this interleave the p-th pair of EVERY unit of every weight belongs to leg p: the CTAs of a row
// split, which all walk their pairs at the same pace, read the same few slot tiles at the same time and share them in L2
// instead of re-reading them from DRAM (ncu: 540 MB of DRAM reads per launch for 336 MB of distinct operands before).
static bool emit_units(Plan& p, const std::vector<RPair>& prs, int K, int k0, int want_colsum, int* ids, int& n_ids) {
    const size_t U = (prs.size() + RD_MAX_PAIRS - 1) / RD_MAX_PAIRS;
    for (size_t u = 0; u < U; ++u) {
        RTask T{}; T.pair_begin = (int)p.rpairs.size(); T.n_pairs = 0; T.K = K; T.k0 = k0; T.want_colsum = want_colsum;
        for (size_t i = u; i < prs.size(); i += U) { p.rpairs.push_back(prs[i]); ++T.n_pairs; }
        if (n_ids >= 16) return false;
        ids[n_ids++] = (int)p.rtasks.size();
        p.rtasks.push_back(T);
    }
    return true;
}

// ------------------------------------------------------------------------------------------------------------------
// Cross-layer stack programs (kernels_stack.cuh), derived from the per-layer tables built above: the same tiles, copied
// into one contiguous range per program, with the base_transform steps chained behind the tile that produces their input
// (forward: conv(l) of an MLP-type node -> Linear -> ReLU -> Linear + residual, hgnn_k4.py:L133-137,175-186; backward:
// dX(l) of an MLP-type node -> dpre(l-1) -> dc(l-1)), so the intermediate tiles never leave the SM in inference and are
// read back from shared memory, not from HBM, in training.
// ------------------------------------------------------------------------------------------------------------------
// activation / gradient buffers written by the phases of a stack program (as opposed to forward state a backward phase reads)
static bool is_phase_buffer(int buf) {
    return (buf >= BUF_H0 && buf < BUF_H0 + MAX_LAYERS + 1) || (buf >= BUF_DHL0 && buf < BUF_DUL0 + MAX_LAYERS);
}

static std::string build_stack_programs(Plan& p) {
    auto begin_prog = [&](Plan::Stack& st) { st.tiles.begin = (int)p.tiles.size(); st.item0 = (int)p.stack_items.size(); st.prog = StackProg{}; };
    auto begin_phase = [&](Plan::Stack& st) -> std::string {
        if (st.prog.n_phases >= STACK_MAX_PHASES) return "too many layers for the cross-layer stack kernel";
        st.prog.first_item[st.prog.n_phases] = (int)p.stack_items.size() - st.item0;
        st.prog.n_items[st.prog.n_phases] = 0;
        return "";
    };
    auto end_phase = [&](Plan::Stack& st) {
        if (st.prog.n_items[st.prog.n_phases] > 0) { st.prog.items_per_row += st.prog.n_items[st.prog.n_phases]; st.prog.n_phases++; }
    };
    // reads[i] = slots of the previous phase item i reads from global memory (operands of non-staged chunks whose buffer the
    // previous phase wrote, and residuals); filled per item, turned into dep_mask by end_prog
    std::vector<unsigned long long> reads;
    auto emit = [&](Plan::Stack& st, const std::vector<Tile>& steps) {
        StackItem it{};
        it.tile = (int)p.tiles.size() - st.tiles.begin; it.n_steps = (int)steps.size();
        const Tile& last = steps.back();
        it.out_slot = last.out_buf >= 0 ? last.out_slot : last.out2_slot;
        it.meta = 0;
        for (size_t s_ = 0; s_ < steps.size() && s_ < 4; ++s_) it.meta |= (steps[s_].n_chunks | (steps[s_].a_stage << 4)) << (8 * s_);
        unsigned long long rd = 0;
        for (const Tile& T : steps) {
            for (int c = 0; c < T.n_chunks; ++c)
                if (!(T.a_stage && c == 0) && is_phase_buffer(T.chunks[c].a_buf)) rd |= 1ull << T.chunks[c].a_slot;
            if (T.res_buf >= 0 && is_phase_buffer(T.res_buf)) rd |= 1ull << T.res_slot;
        }
        p.tiles.insert(p.tiles.end(), steps.begin(), steps.end());
        p.stack_items.push_back(it);
        reads.push_back(rd);
        st.prog.n_items[st.prog.n_phases]++;
    };
    // ping_pong: the buffers of phase p + 1's outputs are those phase p READ (inference): an item may only overwrite slot d
    // once every phase-p item that reads slot d has finished
    auto end_prog = [&](Plan::Stack& st, bool ping_pong) {
        st.tiles.count = (int)p.tiles.size() - st.tiles.begin;
        const size_t r0 = reads.size() - (p.stack_items.size() - st.item0);
        for (int ph = 0; ph < st.prog.n_phases; ++ph)
            for (int i = 0; i < st.prog.n_items[ph]; ++i) {
                StackItem& it = p.stack_items[st.item0 + st.prog.first_item[ph] + i];
                it.dep_mask = 0;
                if (ph == 0) continue;
                it.dep_mask = reads[r0 + st.prog.first_item[ph] + i];
                if (ping_pong)
                    for (int j = 0; j < st.prog.n_items[ph - 1]; ++j) {
                        const StackItem& prev = p.stack_items[st.item0 + st.prog.first_item[ph - 1] + j];
                        if (reads[r0 + st.prog.first_item[ph - 1] + j] >> it.out_slot & 1ull) it.dep_mask |= 1ull << prev.out_slot;
                    }
                // only slots the previous phase actually produces can be waited for
                unsigned long long produced = 0;
                for (int j = 0; j < st.prog.n_items[ph - 1]; ++j) produced |= 1ull << p.stack_items[st.item0 + st.prog.first_item[ph - 1] + j].out_slot;
                it.dep_mask &= produced;
            }
    };
    auto find_by_a = [&](const Launch& L, int a_buf, int a_slot) -> int {
        for (int i = 0; i < L.count; ++i) {
            const Tile& T = p.tiles[L.begin + i];
            if (T.n_chunks == 1 && T.chunks[0].a_buf == a_buf && T.chunks[0].a_slot == a_slot) return L.begin + i;
        }
        return -1;
    };

    // ---- forward (inference / training) ----
    for (int train = 0; train < 2; ++train) {
        Plan::Stack& st = train ? p.stack_train : p.stack_infer;
        begin_prog(st);
        for (int l = 0; l < p.L; ++l) {
            std::string e = begin_phase(st);
            if (!e.empty()) return e;
            const Launch& conv = train ? p.conv_train[l] : p.conv_infer[l];
            const Launch& m1 = train ? p.mlp1_train[l] : p.mlp1[l];
            for (int i = 0; i < conv.count; ++i) {
                Tile T = p.tiles[conv.begin + i];
                if (p.morph_sym && T.out_buf == BUF_CT0 + l) {
                    const int n = T.out_slot;
                    const int ia = find_by_a(m1, BUF_CT0 + l, n), ib = find_by_a(p.mlp2[l], BUF_CT0 + l, p.nm + n);
                    if (ia < 0 || ib < 0) return "internal: base_transform tiles missing for a conv tile";
                    Tile A = p.tiles[ia], Bt = p.tiles[ib];
                    T.stage_out = 1; A.a_stage = 1; A.stage_out = 1; Bt.a_stage = 1;
                    if (!train) { T.out_buf = -1; A.out_buf = -1; }     // the intermediates only exist on chip
                    emit(st, {T, A, Bt});
                } else {
                    emit(st, {T});
                }
            }
            end_phase(st);
        }
        end_prog(st, !train);
    }
    // ---- backward dX chain ----
    {
        Plan::Stack& st = p.stack_bwd;
        begin_prog(st);
        if (p.morph_sym && p.bwd_m1[p.L - 1].count > 0) {       // the decoder reads the MLP type (COM models): dh_L -> dpre -> dc_{L-1}
            std::string e = begin_phase(st);
            if (!e.empty()) return e;
            const Launch& m1 = p.bwd_m1[p.L - 1];
            for (int i = 0; i < m1.count; ++i) {
                Tile A = p.tiles[m1.begin + i];
                const int ib = find_by_a(p.bwd_m2[p.L - 1], BUF_DUL0 + p.L - 1, A.out_slot);
                if (ib < 0) return "internal: base_transform backward tiles do not pair up";
                Tile Bt = p.tiles[ib];
                A.stage_out = 1; Bt.a_stage = 1;
                emit(st, {A, Bt});
            }
            end_phase(st);
        }
        for (int l = p.L - 1; l >= 0; --l) {
            std::string e = begin_phase(st);
            if (!e.empty()) return e;
            const Launch& dx = p.bwd_dx[l];
            for (int i = 0; i < dx.count; ++i) {
                Tile T = p.tiles[dx.begin + i];
                int ia = -1;
                if (p.morph_sym && l >= 1 && T.out_buf == BUF_DHL0 + l && T.out2_buf < 0) ia = find_by_a(p.bwd_m1[l - 1], BUF_DHL0 + l, T.out_slot);
                if (ia >= 0) {
                    Tile A = p.tiles[ia];
                    const int ib = find_by_a(p.bwd_m2[l - 1], BUF_DUL0 + l - 1, A.out_slot);
                    if (ib < 0) return "internal: base_transform backward tiles do not pair up";
                    Tile Bt = p.tiles[ib];
                    T.stage_out = 1; A.a_stage = 1; A.stage_out = 1; Bt.a_stage = 1;
                    emit(st, {T, A, Bt});
                } else {
                    // dh of a joint / foot node is read back ONLY as the pass-through residual of the same node one layer down (the
                    // MMA operands are the masked dc images; only base nodes feed dh into base_transform's backward).  Such a dh is
                    // kept as fp32 in a thread-private layout (kernels_stack.cuh): written straight from the epilogue's registers,
                    // read back by one bulk copy - no (hi, lo) split, no second in-place pass through the staging tiles, and the
                    // tile is left with ONE staged output (dc).  dh_L comes from the decoder kernel as images.
                    if (p.morph_sym) {
                        const int slot = T.out_buf >= 0 ? T.out_slot : T.out2_slot;
                        const bool base = p.slot_type[slot] == p.mlp_type;
                        if (!base && T.out_buf == BUF_DHL0 + l && T.out2_buf >= 0) T.priv |= TILE_OUT_PRIV;
                        if (!base && T.res_buf == BUF_DHL0 + l + 1 && l + 1 < p.L) T.priv |= TILE_RES_PRIV;
                    }
                    emit(st, {T});
                }
            }
            end_phase(st);
        }
        end_prog(st, false);
        // every base_transform backward tile must have been chained somewhere
        int chained = 0, want = 0;
        for (int i = 0; i < st.tiles.count; ++i) chained += p.tiles[st.tiles.begin + i].a_stage;
        for (int l = 0; l < p.L; ++l) want += p.bwd_m1[l].count + p.bwd_m2[l].count;
        const int heads = (p.morph_sym && p.bwd_m1[p.L - 1].count > 0) ? p.bwd_m1[p.L - 1].count : 0;     // pre-phase m1 tiles read global memory
        if (chained != want - heads) return "internal: base_transform backward tiles left out of the stack program";
    }
    return "";
}

// Offsets of every parameter tensor at hidden width `h` (reference named_parameters() order).
static ParamLayout param_layout(const Plan& p, int64_t h) {
    ParamLayout y;
    int64_t o = 0;
    for (int t = 0; t < p.n_types; ++t) { y.enc_w[t] = o; o += h * p.in_w[t]; y.enc_b[t] = o; o += h; }
    y.rel_w.assign(p.L * p.n_etypes, 0); y.rel_b = y.rel_w; y.root_w = y.rel_w;
    for (int l = 0; l < p.L; ++l)
        for (int e = 0; e < p.n_etypes; ++e) {
            const int i = l * p.n_etypes + e;
            y.rel_w[i] = o; o += h * h; y.rel_b[i] = o; o += h; y.root_w[i] = o; o += h * h;
        }
    if (p.morph_sym)
        for (int i = 0; i < 2; ++i) { y.mlp_w[i] = o; o += h * h; y.mlp_b[i] = o; o += h; }
    y.dec_w = o; o += p.C * h; y.dec_b = o; o += p.C;
    y.n = o;
    return y;
}

std::string build_plan(const mshgnn_desc* d, int32_t flags, Plan& p, const std::vector<int>& widths) {
    char err[256];
    if (!d) return "desc is NULL";
    if (flags & ~MSHGNN_PLAN_PAD_HIDDEN) { snprintf(err, sizeof err, "unknown plan flags 0x%x", (unsigned)flags); return err; }
    if (widths.empty()) {
        if (!(flags & MSHGNN_PLAN_PAD_HIDDEN) && d->hidden != H) {
            snprintf(err, sizeof err, "hidden=%d unsupported: this build is specialised for H=128 (MSHGNN_PLAN_PAD_HIDDEN runs 1..128)", d->hidden);
            return err;
        }
        if (d->hidden < 1 || d->hidden > H) { snprintf(err, sizeof err, "hidden=%d unsupported: padded plans take 1..128 hidden channels", d->hidden); return err; }
        p.hidden.assign(1, d->hidden);
    } else {
        for (size_t m = 0; m < widths.size(); ++m)
            if (widths[m] < 1 || widths[m] > H) {
                snprintf(err, sizeof err, "model %zu: hidden=%d unsupported: model batches take 1..128 hidden channels", m, widths[m]);
                return err;
            }
        p.hidden = widths;
    }
    p.n_models = (int)p.hidden.size();
    p.padded = false;
    for (int h : p.hidden) p.padded = p.padded || h != H;
    if (d->n_node_types < 1 || d->n_node_types > MSHGNN_MAX_NODE_TYPES) return "n_node_types out of range";
    if (d->n_edge_types < 1 || d->n_edge_types > MSHGNN_MAX_EDGE_TYPES) return "n_edge_types out of range";
    if (d->num_layers < 1 || d->num_layers > MAX_LAYERS) return "num_layers out of range (1..15)";
    if (d->decode_type < 0 || d->decode_type >= d->n_node_types) return "decode_type out of range";
    if (d->out_channels < 1 || d->out_channels > 8) return "out_channels out of range (1..8)";
    if (d->morph_sym && (d->mlp_type < 0 || d->mlp_type >= d->n_node_types)) return "mlp_type out of range";

    p.n_types = d->n_node_types; p.n_etypes = d->n_edge_types; p.L = d->num_layers;
    p.morph_sym = d->morph_sym ? 1 : 0; p.mlp_type = d->morph_sym ? d->mlp_type : -1;
    p.dec_type = d->decode_type; p.C = d->out_channels;
    p.S = 0;
    for (int t = 0; t < p.n_types; ++t) {
        if (d->nodes_per_graph[t] < 1 || d->nodes_per_graph[t] > 16) return "nodes_per_graph out of range (1..16)";
        if (d->in_width[t] < 1) return "in_width must be >= 1";
        p.nodes[t] = d->nodes_per_graph[t]; p.in_w[t] = d->in_width[t];
        p.type_base[t] = p.S; p.S += p.nodes[t];
        for (int n = 0; n < p.nodes[t]; ++n) { p.slot_type.push_back(t); p.slot_local.push_back(n); }
    }
    if (p.S > 48) return "too many nodes per graph";
    p.nm = p.morph_sym ? p.nodes[p.mlp_type] : 0;

    std::vector<char> has_in(p.n_types, 0);
    for (int e = 0; e < p.n_etypes; ++e) {
        const int st = d->edge_src_type[e], dt = d->edge_dst_type[e];
        if (st < 0 || st >= p.n_types || dt < 0 || dt >= p.n_types) return "edge type endpoint out of range";
        p.e_src_t[e] = st; p.e_dst_t[e] = dt; p.e_mean[e] = d->edge_mean[e] ? 1 : 0;
        has_in[dt] = 1;
        if (d->edge_count[e] < 0 || (d->edge_count[e] > 0 && (!d->edge_src[e] || !d->edge_dst[e]))) return "edge list missing";
        p.e_src[e].assign(d->edge_src[e], d->edge_src[e] + d->edge_count[e]);
        p.e_dst[e].assign(d->edge_dst[e], d->edge_dst[e] + d->edge_count[e]);
        std::vector<int> deg(p.nodes[dt], 0);
        for (int i = 0; i < d->edge_count[e]; ++i) {
            if (p.e_src[e][i] < 0 || p.e_src[e][i] >= p.nodes[st] || p.e_dst[e][i] < 0 || p.e_dst[e][i] >= p.nodes[dt])
                return "edge endpoint out of range for its node type";
            deg[p.e_dst[e][i]]++;
        }
        if (p.e_mean[e])
            for (int n = 0; n < p.nodes[dt]; ++n)
                if (deg[n] > 1) {
                    snprintf(err, sizeof err, "edge type %d: aggr='mean' with in-degree %d > 1 is not supported "
                             "(all reference templates have in-degree 1 on mean relations)", e, deg[n]);
                    return err;
                }
    }
    for (int t = 0; t < p.n_types; ++t)
        if (!has_in[t]) return "every node type must be the destination of at least one edge type";

    // ---------------- parameter layout: reference named_parameters() order ----------------
    {
        const ParamLayout in = param_layout(p, H);
        for (int t = 0; t < p.n_types; ++t) { p.off_enc_w[t] = in.enc_w[t]; p.off_enc_b[t] = in.enc_b[t]; }
        p.off_rel_w = in.rel_w; p.off_rel_b = in.rel_b; p.off_root_w = in.root_w;
        for (int i = 0; i < 2; ++i) { p.off_mlp_w[i] = in.mlp_w[i]; p.off_mlp_b[i] = in.mlp_b[i]; }
        p.off_dec_w = in.dec_w; p.off_dec_b = in.dec_b;
        p.n_params = in.n;
        if (in.n > (int64_t)1 << 30) return "parameter count too large";
        p.ext_base.assign(1, 0);
        for (int m = 0; m < p.n_models; ++m) {
            p.ext.push_back(p.hidden[m] != H ? param_layout(p, p.hidden[m]) : in);
            p.ext_base.push_back(p.ext_base.back() + p.ext.back().n);
        }
    }
    if (p.padded) {
        // The caller's [h, in], [h], [h, h], [C, h] tensors are the top-left blocks of the 128-wide ones.  Every model's encoder
        // segments come first: the backward compacts the rest before the encoder weight gradient runs, then the encoder block.
        auto seg = [&](int64_t e, int64_t i, int rows, int cols, int rows_i, int cols_i) { p.pad_segs.push_back(PadSeg{e, i, rows, cols, rows_i, cols_i}); };
        for (int m = 0; m < p.n_models; ++m) {
            const ParamLayout& y = p.ext[m];
            const int64_t e0 = p.ext_base[m], i0 = m * p.n_params;
            const int h = p.hidden[m];
            for (int t = 0; t < p.n_types; ++t) {
                seg(e0 + y.enc_w[t], i0 + p.off_enc_w[t], h, p.in_w[t], H, p.in_w[t]);
                seg(e0 + y.enc_b[t], i0 + p.off_enc_b[t], 1, h, 1, H);
            }
        }
        p.n_pad_enc = (int)p.pad_segs.size();
        for (int m = 0; m < p.n_models; ++m) {
            const ParamLayout& y = p.ext[m];
            const int64_t e0 = p.ext_base[m], i0 = m * p.n_params;
            const int h = p.hidden[m];
            for (int i = 0; i < p.L * p.n_etypes; ++i) {
                seg(e0 + y.rel_w[i], i0 + p.off_rel_w[i], h, h, H, H);
                seg(e0 + y.rel_b[i], i0 + p.off_rel_b[i], 1, h, 1, H);
                seg(e0 + y.root_w[i], i0 + p.off_root_w[i], h, h, H, H);
            }
            if (p.morph_sym)
                for (int i = 0; i < 2; ++i) { seg(e0 + y.mlp_w[i], i0 + p.off_mlp_w[i], h, h, H, H); seg(e0 + y.mlp_b[i], i0 + p.off_mlp_b[i], 1, h, 1, H); }
            seg(e0 + y.dec_w, i0 + p.off_dec_w, p.C, h, p.C, H);
            seg(e0 + y.dec_b, i0 + p.off_dec_b, 1, p.C, 1, p.C);
        }
    }

    // ---------------- derived weights ----------------
    int64_t q = 0;
    auto add_op = [&](int64_t dst, int rows, int cols, int tr, std::vector<int64_t> srcs) {
        DeriveOp op{}; op.dst_off = (int)dst; op.rows = rows; op.cols = cols; op.transpose = tr;
        op.n_src = (int)srcs.size();
        for (size_t i = 0; i < srcs.size(); ++i) op.src_off[i] = (int)srcs[i];
        p.derive_ops.push_back(op);
    };
    for (int t = 0; t < p.n_types; ++t) {
        p.der_encT[t] = q; add_op(q, H, p.in_w[t], 1, {p.off_enc_w[t]}); q += (int64_t)H * p.in_w[t];
    }
    p.der_relT.assign(p.L * p.n_etypes, -1);
    p.der_rootT.assign(p.L * p.n_types, -1); p.der_root = p.der_rootT; p.der_bias = p.der_rootT;
    for (int l = 0; l < p.L; ++l) {
        for (int e = 0; e < p.n_etypes; ++e) {
            p.der_relT[l * p.n_etypes + e] = q; add_op(q, H, H, 1, {p.off_rel_w[l * p.n_etypes + e]}); q += H * H;
        }
        for (int t = 0; t < p.n_types; ++t) {
            std::vector<int64_t> roots, biases;
            for (int e = 0; e < p.n_etypes; ++e)
                if (p.e_dst_t[e] == t) { roots.push_back(p.off_root_w[l * p.n_etypes + e]); biases.push_back(p.off_rel_b[l * p.n_etypes + e]); }
            if (roots.size() > 4) return "more than 4 edge types into one node type is not supported";
            p.der_rootT[l * p.n_types + t] = q; add_op(q, H, H, 1, roots); q += H * H;
            p.der_root[l * p.n_types + t] = q;  add_op(q, H, H, 0, roots); q += H * H;
            p.der_bias[l * p.n_types + t] = q;  add_op(q, 1, H, 0, biases); q += H;
        }
    }
    if (p.morph_sym)
        for (int i = 0; i < 2; ++i) { p.der_mlpT[i] = q; add_op(q, H, H, 1, {p.off_mlp_w[i]}); q += H * H; }
    p.n_derived = q;
    // bias sums ([1 x H] ops) first: the tensor-core modes read nothing else from the derived buffer (their weights are
    // the fp16 images of k_derive16), so they run only this prefix
    std::stable_partition(p.derive_ops.begin(), p.derive_ops.end(), [](const DeriveOp& o) { return o.rows == 1; });
    p.n_derive_bias = 0;
    for (const DeriveOp& o : p.derive_ops) p.n_derive_bias += o.rows == 1;

    // ---------------- signs ----------------
    p.sign_off_slot.assign(p.S, -1);
    for (int t = 0; t < p.n_types; ++t) {
        if (!d->in_sign[t]) continue;
        for (int n = 0; n < p.nodes[t]; ++n) {
            p.sign_off_slot[p.slot_of(t, n)] = (int)p.signs.size();
            for (int k = 0; k < p.in_w[t]; ++k) p.signs.push_back(d->in_sign[t][(int64_t)n * p.in_w[t] + k]);
            while (p.signs.size() % 4) p.signs.push_back(1.f);
        }
    }
    if (d->out_sign) {
        p.sign_off_out = (int)p.signs.size();
        for (int i = 0; i < p.nodes[p.dec_type] * p.C; ++i) p.signs.push_back(d->out_sign[i]);
    }
    if (p.signs.empty()) p.signs.push_back(1.f);

    auto roots_of = [&](int l, int t) {
        std::vector<int64_t> r;
        for (int e = 0; e < p.n_etypes; ++e)
            if (p.e_dst_t[e] == t) r.push_back(p.off_root_w[l * p.n_etypes + e]);
        return r;
    };

    // ---------------- forward contribution lists ----------------
    // contrib[d] = list of (src slot, edge type); the root term is implicit.
    struct Contrib { int src, e; };
    std::vector<std::vector<Contrib>> contrib(p.S);
    for (int e = 0; e < p.n_etypes; ++e)
        for (size_t i = 0; i < p.e_src[e].size(); ++i)
            contrib[p.slot_of(p.e_dst_t[e], p.e_dst[e][i])].push_back({p.slot_of(p.e_src_t[e], p.e_src[e][i]), e});
    for (int s = 0; s < p.S; ++s)
        if ((int)contrib[s].size() + 1 > MAX_CHUNKS) return "a node has too many in-edges (max 7)";
    std::vector<std::vector<Contrib>> outgoing(p.S);   // outgoing[s] = (dst slot, e)
    for (int dslot = 0; dslot < p.S; ++dslot)
        for (auto& c : contrib[dslot]) outgoing[c.src].push_back({dslot, c.e});
    for (int s = 0; s < p.S; ++s)
        if ((int)outgoing[s].size() + 1 > MAX_CHUNKS) return "a node has too many out-edges (max 7)";

    // ---------------- liveness: need[l][s] <=> h_l[s] influences the output ----------------
    p.need.assign(p.L + 1, std::vector<char>(p.S, 0));
    for (int n = 0; n < p.nodes[p.dec_type]; ++n) p.need[p.L][p.slot_of(p.dec_type, n)] = 1;
    for (int l = p.L - 1; l >= 0; --l)
        for (int dslot = 0; dslot < p.S; ++dslot) {
            if (!p.need[l + 1][dslot]) continue;
            p.need[l][dslot] = 1;                              // root term (and residual)
            for (auto& c : contrib[dslot]) p.need[l][c.src] = 1;
        }

    // ---------------- decoder ----------------
    memset(&p.dec, 0, sizeof p.dec);
    p.dec.n_dec = p.nodes[p.dec_type]; p.dec.C = p.C;
    for (int n = 0; n < p.dec.n_dec; ++n) p.dec.slots[n] = p.slot_of(p.dec_type, n);
    p.dec.w_off = (int)p.off_dec_w; p.dec.b_off = (int)p.off_dec_b; p.dec.sign_off = p.sign_off_out;

    // ---------------- forward tiles ----------------
    auto push_launch = [&](std::vector<Tile>& v) { Launch L{(int)p.tiles.size(), (int)v.size()}; p.tiles.insert(p.tiles.end(), v.begin(), v.end()); return L; };
    {
        std::vector<Tile> v;
        for (int s = 0; s < p.S; ++s) {
            if (!p.need[0][s]) continue;
            const int t = p.slot_type[s], n = p.slot_local[s];
            Tile T = empty_tile();
            Chunk c{};
            c.a_kind = A_EXT; c.a_buf = BUF_X0 + t; c.a_slot = 0; c.K = p.in_w[t]; c.lda = p.nodes[t] * p.in_w[t];
            c.a_off = n * p.in_w[t]; c.w_buf = BUF_DERIVED; c.w_off = (int)p.der_encT[t]; c.sign_off = p.sign_off_slot[s];
            c.w16_row = t * H;   // tensor-core encoder: first row of this type's [128][enc_kmax] fp16 weight image
            T.chunks[T.n_chunks++] = c;
            T.bias_buf = BUF_PARAMS; T.bias_off = (int)p.off_enc_b[t]; T.relu = 1;
            T.out_buf = BUF_H0; T.out_slot = s;
            v.push_back(T);
        }
        p.enc_launch = push_launch(v);
        for (auto& T : v) { T.mask_out_buf = BUF_MASKE; T.mask_out_slot = T.out_slot; }
        p.enc_train = push_launch(v);
    }
    for (int l = 0; l < p.L; ++l) {
        std::vector<Tile> conv, m1, m2;
        for (int dslot = 0; dslot < p.S; ++dslot) {
            if (!p.need[l + 1][dslot]) continue;
            const int t = p.slot_type[dslot], n = p.slot_local[dslot];
            Tile T = empty_tile();
            for (auto& c : contrib[dslot])
                T.chunks[T.n_chunks++] = slab_chunk(BUF_H0 + l, c.src, BUF_DERIVED, p.der_relT[l * p.n_etypes + c.e],
                                                    mat16(p, {p.off_rel_w[l * p.n_etypes + c.e]}, false));
            T.chunks[T.n_chunks++] = slab_chunk(BUF_H0 + l, dslot, BUF_DERIVED, p.der_rootT[l * p.n_types + t], mat16(p, roots_of(l, t), false));
            T.bias_buf = BUF_DERIVED; T.bias_off = (int)p.der_bias[l * p.n_types + t];
            if (p.morph_sym && t == p.mlp_type) {
                // conv -> c_base ; base_transform: Linear -> ReLU -> Linear ; + residual (hgnn_k4.py:L133-137,175-186)
                T.relu = 0; T.out_buf = BUF_CT0 + l; T.out_slot = n;
                conv.push_back(T);
                Tile A = empty_tile();
                A.chunks[A.n_chunks++] = slab_chunk(BUF_CT0 + l, n, BUF_DERIVED, p.der_mlpT[0], mat16(p, {p.off_mlp_w[0]}, false));
                A.bias_buf = BUF_PARAMS; A.bias_off = (int)p.off_mlp_b[0]; A.relu = 1;
                A.out_buf = BUF_CT0 + l; A.out_slot = p.nm + n;
                m1.push_back(A);
                Tile Bt = empty_tile();
                Bt.chunks[Bt.n_chunks++] = slab_chunk(BUF_CT0 + l, p.nm + n, BUF_DERIVED, p.der_mlpT[1], mat16(p, {p.off_mlp_w[1]}, false));
                Bt.bias_buf = BUF_PARAMS; Bt.bias_off = (int)p.off_mlp_b[1]; Bt.relu = 0;
                Bt.res_buf = BUF_H0 + l; Bt.res_slot = dslot;
                Bt.out_buf = BUF_H0 + l + 1; Bt.out_slot = dslot;
                m2.push_back(Bt);
            } else {
                T.relu = 1; T.out_buf = BUF_H0 + l + 1; T.out_slot = dslot;
                if (p.morph_sym) { T.res_buf = BUF_H0 + l; T.res_slot = dslot; }
                conv.push_back(T);
            }
        }
        // inference copy (no ReLU bitmask), training copy (bitmask for MS joint/foot rows)
        p.conv_infer.push_back(push_launch(conv));
        for (auto& T : conv)
            if (T.relu) { T.mask_out_buf = BUF_MASK0 + l; T.mask_out_slot = T.out_slot; }
        p.conv_train.push_back(push_launch(conv));
        p.mlp1.push_back(push_launch(m1));
        for (auto& T : m1) { T.mask_out_buf = BUF_MASK0 + l; T.mask_out_slot = p.S + (T.out_slot - p.nm); }
        p.mlp1_train.push_back(push_launch(m1));
        p.mlp2.push_back(push_launch(m2));
    }

    // ---------------- backward tiles + weight-gradient tasks ----------------
    p.bwd_m1.resize(p.L); p.bwd_m2.resize(p.L); p.bwd_dx.resize(p.L); p.dw_layer.resize(p.L);
    std::vector<int> mlp_tasks[2];
    for (int l = p.L - 1; l >= 0; --l) {
        // per-layer buffer ids (plan.cuh): the per-layer launch sequence aliases them onto ping-pong buffers
        const int DHn = BUF_DHL0 + l + 1, DHo = BUF_DHL0 + l;
        const int DCc = BUF_DCL0 + l, DCp = BUF_DCL0 + l - 1;   // dc_l lives in DCc, dc_{l-1} goes to DCp
        const int DUc = BUF_DUL0 + l;
        std::vector<Tile> b1, b2, dx;
        if (p.morph_sym)
            for (int n = 0; n < p.nm; ++n) {
                const int s = p.slot_of(p.mlp_type, n);
                if (!p.need[l + 1][s]) continue;
                Tile A = empty_tile();   // dpre = (du * W2) (*) (t > 0)
                A.chunks[A.n_chunks++] = slab_chunk(DHn, s, BUF_PARAMS, p.off_mlp_w[1], mat16(p, {p.off_mlp_w[1]}, true));
                A.posmask_buf = BUF_MASK0 + l; A.posmask_slot = p.S + n;
                A.out_buf = DUc; A.out_slot = n;
                b1.push_back(A);
                Tile Bt = empty_tile();  // dc_base = dpre * W1
                Bt.chunks[Bt.n_chunks++] = slab_chunk(DUc, n, BUF_PARAMS, p.off_mlp_w[0], mat16(p, {p.off_mlp_w[0]}, true));
                Bt.out_buf = DCc; Bt.out_slot = s;
                b2.push_back(Bt);
            }
        for (int s = 0; s < p.S; ++s) {
            if (!p.need[l][s]) continue;
            const int t = p.slot_type[s];
            Tile T = empty_tile();
            for (auto& og : outgoing[s])
                if (p.need[l + 1][og.src])   // og.src holds the destination slot here
                    T.chunks[T.n_chunks++] = slab_chunk(DCc, og.src, BUF_PARAMS, p.off_rel_w[l * p.n_etypes + og.e],
                                                        mat16(p, {p.off_rel_w[l * p.n_etypes + og.e]}, true));
            if (p.need[l + 1][s]) {
                T.chunks[T.n_chunks++] = slab_chunk(DCc, s, BUF_DERIVED, p.der_root[l * p.n_types + t], mat16(p, roots_of(l, t), true));
                if (p.morph_sym) { T.res_buf = DHn; T.res_slot = s; }
            }
            if (l == 0) {
                T.out2_buf = DCp; T.out2_slot = s; T.out2_mask_kind = MK_BITS; T.out2_mask_buf = BUF_MASKE; T.out2_mask_slot = s;
            } else if (p.morph_sym) {
                T.out_buf = DHo; T.out_slot = s;
                if (t != p.mlp_type) {
                    T.out2_buf = DCp; T.out2_slot = s; T.out2_mask_kind = MK_BITS; T.out2_mask_buf = BUF_MASK0 + l - 1; T.out2_mask_slot = s;
                }
            } else {
                T.out2_buf = DCp; T.out2_slot = s; T.out2_mask_kind = MK_BITS; T.out2_mask_buf = BUF_MASK0 + l - 1; T.out2_mask_slot = s;
            }
            dx.push_back(T);
        }
        p.bwd_m1[l] = push_launch(b1); p.bwd_m2[l] = push_launch(b2); p.bwd_dx[l] = push_launch(dx);

        // ---- weight-gradient tasks of layer l (units of <= RD_MAX_PAIRS pairs so all CTAs carry equal work) ----
        Launch lt{(int)p.rtasks.size(), 0};
        auto slab_pair = [&](int dbuf, int dslot, int abuf, int aslot) {
            RPair r{}; r.d_buf = dbuf; r.d_slot = dslot; r.a_kind = A_SLAB; r.a_buf = abuf; r.a_slot = aslot; r.lda = H; r.a_off = 0; r.sign_off = -1;
            return r;
        };
        for (int e = 0; e < p.n_etypes; ++e) {          // lin_rel weights
            std::vector<RPair> prs;
            for (size_t i = 0; i < p.e_src[e].size(); ++i) {
                const int dslot = p.slot_of(p.e_dst_t[e], p.e_dst[e][i]);
                if (!p.need[l + 1][dslot]) continue;
                prs.push_back(slab_pair(DCc, dslot, BUF_H0 + l, p.slot_of(p.e_src_t[e], p.e_src[e][i])));
            }
            if (prs.empty()) continue;
            OutGroup g{}; g.kind = 0; g.n_outs = 1; g.outs[0] = (int)p.off_rel_w[l * p.n_etypes + e]; g.K = H; g.k0 = 0; g.scale = 1.f;
            if (!emit_units(p, prs, H, 0, 0, g.tasks, g.n_tasks)) return "too many weight-gradient units for one tensor";
            p.groups.push_back(g);
        }
        for (int t = 0; t < p.n_types; ++t) {           // lin_root weights + lin_rel biases (shared by all edge types into t)
            std::vector<RPair> prs;
            for (int n = 0; n < p.nodes[t]; ++n) {
                const int s = p.slot_of(t, n);
                if (p.need[l + 1][s]) prs.push_back(slab_pair(DCc, s, BUF_H0 + l, s));
            }
            if (prs.empty()) continue;
            OutGroup gw{}; gw.kind = 0; gw.K = H; gw.k0 = 0; gw.scale = 1.f;
            if (!emit_units(p, prs, H, 0, 1, gw.tasks, gw.n_tasks)) return "too many weight-gradient units for one tensor";
            OutGroup gb = gw; gb.kind = 1;
            for (int e = 0; e < p.n_etypes; ++e)
                if (p.e_dst_t[e] == t) {
                    gw.outs[gw.n_outs++] = (int)p.off_root_w[l * p.n_etypes + e];
                    gb.outs[gb.n_outs++] = (int)p.off_rel_b[l * p.n_etypes + e];
                }
            p.groups.push_back(gw); p.groups.push_back(gb);
        }
        if (p.morph_sym) {                               // shared base_transform: tasks per layer, one group at the end
            std::vector<RPair> p1, p2;
            for (int n = 0; n < p.nm; ++n) {
                const int s = p.slot_of(p.mlp_type, n);
                if (!p.need[l + 1][s]) continue;
                p1.push_back(slab_pair(DUc, n, BUF_CT0 + l, n));
                p2.push_back(slab_pair(DHn, s, BUF_CT0 + l, p.nm + n));
            }
            if (!p1.empty()) {
                int ids[16], n_ids = 0;
                if (!emit_units(p, p1, H, 0, 1, ids, n_ids)) return "too many weight-gradient units for one tensor";
                mlp_tasks[0].insert(mlp_tasks[0].end(), ids, ids + n_ids);
                n_ids = 0;
                if (!emit_units(p, p2, H, 0, 1, ids, n_ids)) return "too many weight-gradient units for one tensor";
                mlp_tasks[1].insert(mlp_tasks[1].end(), ids, ids + n_ids);
            }
        }
        lt.count = (int)p.rtasks.size() - lt.begin;
        p.dw_layer[l] = lt;
    }
    if (p.morph_sym)
        for (int i = 0; i < 2; ++i) {
            if (mlp_tasks[i].empty()) continue;
            // the shared MLP accumulates over layers: chunk the task list into groups of <= 16 that ADD into the output
            if (mlp_tasks[i].size() > 16) return "base_transform gradient spans more than 16 units";
            OutGroup gw{}; gw.kind = 0; gw.K = H; gw.k0 = 0; gw.scale = 1.f; gw.n_outs = 1; gw.outs[0] = (int)p.off_mlp_w[i];
            for (int tk : mlp_tasks[i]) gw.tasks[gw.n_tasks++] = tk;
            OutGroup gb = gw; gb.kind = 1; gb.outs[0] = (int)p.off_mlp_b[i];
            p.groups.push_back(gw); p.groups.push_back(gb);
        }
    p.n_groups_layers = (int)p.groups.size();
    // ---- encoder weight gradients: dW_enc[t] = sum_slots dpre0[s]^T (x[s] * sign[s]) ----
    p.dw_enc.begin = (int)p.rtasks.size();
    for (int t = 0; t < p.n_types; ++t) {
        std::vector<RPair> prs;
        for (int n = 0; n < p.nodes[t]; ++n) {
            const int s = p.slot_of(t, n);
            if (!p.need[0][s]) continue;
            RPair r{}; r.d_buf = BUF_DCL0 - 1; r.d_slot = s; r.a_kind = A_EXT; r.a_buf = BUF_X0 + t; r.a_slot = 0;
            r.lda = p.nodes[t] * p.in_w[t]; r.a_off = n * p.in_w[t]; r.sign_off = p.sign_off_slot[s];
            prs.push_back(r);
        }
        if (prs.empty()) continue;
        for (int k0 = 0; k0 < p.in_w[t]; k0 += H) {
            OutGroup g{}; g.kind = 0; g.n_outs = 1; g.outs[0] = (int)p.off_enc_w[t]; g.K = p.in_w[t]; g.k0 = k0; g.scale = 1.f;
            if (!emit_units(p, prs, p.in_w[t], k0, k0 == 0, g.tasks, g.n_tasks)) return "too many weight-gradient units for one tensor";
            p.groups.push_back(g);
            if (k0 == 0) { OutGroup gb = g; gb.kind = 1; gb.outs[0] = (int)p.off_enc_b[t]; p.groups.push_back(gb); }
        }
    }
    p.dw_enc.count = (int)p.rtasks.size() - p.dw_enc.begin;
    // ---- tensor-core encoder weight-gradient units: (type, 192-column range, group of <= 4 slots) ----
    p.enc_kmax = 64;
    for (int t = 0; t < p.n_types; ++t) if (round_up(p.in_w[t], 64) > p.enc_kmax) p.enc_kmax = (int)round_up(p.in_w[t], 64);
    for (int t = 0; t < p.n_types; ++t) {
        std::vector<int> slots;
        for (int n = 0; n < p.nodes[t]; ++n) if (p.need[0][p.slot_of(t, n)]) slots.push_back(n);
        if (slots.empty()) continue;
        for (int k0 = 0; k0 < p.in_w[t]; k0 += 192) {
            EncDwGroup g{};
            g.first = (int)p.enc_units.size(); g.K = p.in_w[t]; g.k0 = k0;
            g.width = p.in_w[t] - k0 < 192 ? p.in_w[t] - k0 : 192;
            g.w_off = (int)p.off_enc_w[t]; g.b_off = k0 == 0 ? (int)p.off_enc_b[t] : -1;
            for (size_t b = 0; b < slots.size(); b += 4) {
                EncDwUnit u{};
                u.x_buf = BUF_X0 + t; u.lda = p.nodes[t] * p.in_w[t]; u.K = p.in_w[t]; u.k0 = k0; u.nkb = (g.width + 63) / 64;
                u.want_colsum = k0 == 0;
                for (size_t i = b; i < slots.size() && i < b + 4; ++i) {
                    const int n = slots[i], s = p.slot_of(t, n);
                    u.d_slot[u.n_slots] = s; u.a_off[u.n_slots] = n * p.in_w[t]; u.sign_off[u.n_slots] = p.sign_off_slot[s];
                    u.n_slots++;
                }
                p.enc_units.push_back(u);
            }
            g.count = (int)p.enc_units.size() - g.first;
            p.enc_groups.push_back(g);
        }
    }
    // ---- input-gradient units: one per node slot ----
    for (int t = 0; t < p.n_types; ++t)
        for (int n = 0; n < p.nodes[t]; ++n) {
            const int s = p.slot_of(t, n);
            DxUnit u{};
            u.type = t; u.slot = s; u.node = n; u.K = p.in_w[t]; u.n_kb = (p.in_w[t] + 63) / 64;
            u.sign_off = p.sign_off_slot[s]; u.live = p.need[0][s] ? 1 : 0;
            p.dx_units.push_back(u);
        }
    { std::string e = build_stack_programs(p); if (!e.empty()) return e; }
    return "";
}

static std::atomic<int> g_stack_on{1};
bool stack_enabled() { return g_stack_on.load(std::memory_order_relaxed) != 0; }
void set_stack_enabled(int on) { g_stack_on.store(on ? 1 : 0, std::memory_order_relaxed); }

// CTA-pair variant of the stack kernel (kernels_stack2.cuh): 1 (default) = for batches of >= STACK_PAIR_MIN_GRAPHS graphs, 2 = always,
// 0 = never (option "stack_pair").  Below ~6 K graphs a phase of a row chunk has fewer pair items than there are
// CTA pairs to feed (8 pairs x 20 items against 74 pairs at 2048 graphs) and the one-CTA kernel is 5-10 % faster
// (2048 graphs: 0.155 / 0.155 ms against 0.159 / 0.171; 4096: 0.214 / 0.251 against 0.215 / 0.268; 16384: 0.81 / 1.03 against 0.77 / 0.975).
constexpr int64_t STACK_PAIR_MIN_GRAPHS = 6144;
static std::atomic<int> g_stack_pair{1};
int stack_pair_mode() { return g_stack_pair.load(std::memory_order_relaxed); }
void set_stack_pair_mode(int v) { g_stack_pair.store(v < 0 ? 0 : (v > 2 ? 2 : v), std::memory_order_relaxed); }

// Row split of a weight-gradient launch of `units` CTAs per split (one unit x one row split each, one CTA per SM): a CTA takes
// time ~ rows + a fixed ~96 rows' worth, and the launch ceil(units x splits / 148) waves of that.  Starting from `rows0`, whose
// cost counts `keep` times, a candidate of [lo, hi] rows (multiples of 64, at most 64 splits) is taken when its cost is below
// `gain` times the best so far.
static int64_t fit_split_rows(int64_t B, int64_t units, int64_t rows0, double keep, double gain, int64_t lo, int64_t hi) {
    auto cost = [&](int64_t rows) {
        const int64_t ns = (B + rows - 1) / rows;
        return (double)((units * ns + 147) / 148) * (double)(rows + 96);
    };
    int64_t best = rows0;
    double best_c = keep * cost(rows0);
    for (int64_t rows = lo; rows <= hi; rows += 64) {
        if ((B + rows - 1) / rows > 64) continue;
        const double c = cost(rows);
        if (c < gain * best_c) { best_c = c; best = rows; }
    }
    return best;
}

// Every split below is a function of the per-model batch B alone: model m of a model batch reduces its rows exactly as a
// single-model call on its B graphs does, so its gradients are bit for bit the same.
WsLayout ws_layout(const Plan& p, int64_t B, int train, int mode, int M) {
    const bool tc = mode != MSHGNN_MODE_FP32;
    WsLayout w{};
    w.M = M < 1 ? 1 : M;
    w.stack = tc && stack_enabled() && p.stack_infer.prog.n_phases > 0;
    w.stack_pair = w.stack && (stack_pair_mode() == 2 || (stack_pair_mode() == 1 && (int64_t)w.M * B >= STACK_PAIR_MIN_GRAPHS));
    w.Bm = round_up(B < 1 ? 1 : B, w.stack_pair ? 2 * TILE_M : TILE_M);      // the CTA-pair kernel walks row tiles two at a time
    w.Bp = (int64_t)w.M * w.Bm;
    int ns = (int)((B + 511) / 512);
    w.n_splits = ns < 1 ? 1 : (ns > 64 ? 64 : ns);
    {   // tcgen05 reduce-GEMM: ~1024 rows per split (fp32 accumulation in TMEM, splits summed in double), no empty split.
        // Row range per CTA decides the L2 reuse: the CTAs resident together (148) cover 148 / n_tasks splits, and every
        // dC / A slot tile of those rows is read by ~3 pairs at different times.  With 2048-row splits that working set was
        // 336 MB (> 126 MB L2) and ncu counted 607 MB of DRAM reads per launch for 300 MB of operands.
        const int64_t dw_rows = 1024;
        int64_t target = (B + dw_rows - 1) / dw_rows;
        // small batches: still give every SM a CTA (tasks x splits >= ~148), down to 64-row splits
        int tasks = 1;
        for (size_t l = 0; l < p.dw_layer.size(); ++l) tasks = p.dw_layer[l].count > tasks ? p.dw_layer[l].count : tasks;
        const int64_t fill = (148 + tasks - 1) / tasks, most = (B + 63) / 64;
        if (target < fill) target = fill < most ? fill : most;
        target = target < 1 ? 1 : (target > 64 ? 64 : target);
        w.rows_per_tc = (int)round_up((B + target - 1) / target, 64);
        w.n_splits_tc = (int)((B + w.rows_per_tc - 1) / w.rows_per_tc);
        // Per layer launch: the pruned last layers have 2 / 5 / 8 / 11 tasks instead of 17 (dead branches), so the default 16
        // splits left them at 32 / 80 / 128 / 176 CTAs - a quarter-filled wave, or one full wave plus a 19 % one (ncu: 57 / 58 /
        // 61 / 114 us against 121 us for the full 272-CTA layer).  Fit each layer's split under the same row cap; keep the
        // default unless the model gains > 10 %.
        const int64_t cap = dw_rows > w.rows_per_tc ? dw_rows : w.rows_per_tc;
        for (int l = 0; l < MAX_LAYERS; ++l) { w.dw_ns[l] = w.n_splits_tc; w.dw_rows[l] = w.rows_per_tc; }
        int64_t all_tasks = 0;
        for (size_t l = 0; l < p.dw_layer.size() && l < (size_t)MAX_LAYERS; ++l) {
            all_tasks += p.dw_layer[l].count;
            w.dw_rows[l] = (int)fit_split_rows(B, p.dw_layer[l].count, w.rows_per_tc, 0.9, 1.0, 64, cap);
            w.dw_ns[l] = (int)((B + w.dw_rows[l] - 1) / w.dw_rows[l]);
        }
        // Stack mode: the dX chain of every layer has already run when the weight gradients start, so ALL layers' tasks go
        // into ONE launch (K4: 94 tasks) with one row split count fitted to whole waves by the same cost model - 8 launches
        // fewer, and at small batches (2048 graphs: 136 CTAs of 256 rows per layer launch) CTAs long enough to amortise
        // their fixed prologue / partial write-out (94 x 3 splits of 704 rows).
        if (w.stack && train) {
            const int64_t best = fit_split_rows(B, all_tasks, w.rows_per_tc, 1.0, 1.0, 64, round_up(B < 2048 ? B : 2048, 64));
            for (size_t l = 0; l < p.dw_layer.size() && l < (size_t)MAX_LAYERS; ++l) { w.dw_rows[l] = (int)best; w.dw_ns[l] = (int)((B + best - 1) / best); }
        }
    }
    {   // partial slots, packed launch by launch in task order (the SIMT kernels use one split count for every task)
        std::vector<std::pair<int, int>> seg;          // (first task, split count)
        for (size_t l = 0; l < p.dw_layer.size() && l < (size_t)MAX_LAYERS; ++l)
            if (p.dw_layer[l].count > 0) seg.push_back({p.dw_layer[l].begin, tc ? w.dw_ns[l] : w.n_splits});
        if (p.dw_enc.count > 0) seg.push_back({p.dw_enc.begin, tc ? 0 : w.n_splits});   // the tensor-core encoder gradient has its own partials
        std::sort(seg.begin(), seg.end());
        w.segs.n = 0;
        int base = 0;
        for (size_t i = 0; i < seg.size() && i < (size_t)MAX_PART_SEGS; ++i) {
            const int end = i + 1 < seg.size() ? seg[i + 1].first : (int)p.rtasks.size();
            w.segs.begin[i] = seg[i].first; w.segs.ns[i] = seg[i].second; w.segs.base[i] = base;
            base += (end - seg[i].first) * seg[i].second;
            w.segs.begin[i + 1] = end;
            w.segs.n = (int)i + 1;
        }
        w.part_slots = base > 0 ? base : 1;
        for (int l = 0; l < MAX_LAYERS; ++l) w.dw_slot0[l] = 0;
        for (size_t l = 0; l < p.dw_layer.size() && l < (size_t)MAX_LAYERS; ++l)
            for (int i = 0; i < w.segs.n; ++i)
                if (w.segs.begin[i] == p.dw_layer[l].begin && p.dw_layer[l].count > 0) w.dw_slot0[l] = w.segs.base[i];
    }
    int64_t o = 0;
    auto take = [&](int64_t bytes) { int64_t at = o; o += round_up(bytes, 256); return at; };
    const int64_t slab = (int64_t)p.S * w.Bp * H * 4;
    const int64_t ctb = (int64_t)2 * p.nm * w.Bp * H * 4;
    for (int id = 0; id < MAX_BUFS; ++id) w.buf[id] = w.buf16[id][0] = w.buf16[id][1] = -1;
    w.part_w = w.part_b = w.dec_part = -1;
    w.buf[BUF_DERIVED] = take(w.M * p.n_derived * 4);
    // fp32 slabs exist in MODE_FP32 only: the tensor-core modes keep every activation / gradient as (hi, lo) fp16 images
    if (train) {
        if (!tc) {
            for (int l = 0; l <= p.L; ++l) w.buf[BUF_H0 + l] = take(slab);
            if (p.morph_sym)
                for (int l = 0; l < p.L; ++l) w.buf[BUF_CT0 + l] = take(ctb);
        }
        for (int l = 0; l < p.L; ++l) w.buf[BUF_MASK0 + l] = take((int64_t)(p.S + p.nm) * w.Bp * 16);
        w.buf[BUF_MASKE] = take((int64_t)p.S * w.Bp * 16);
        if (!tc) {      // the per-layer backward ids alias two ping-pong slabs
            int64_t dh[2], dc[2], du = -1;
            dh[0] = take(slab); dh[1] = take(slab); dc[0] = take(slab); dc[1] = take(slab);
            if (p.morph_sym) du = take((int64_t)p.nm * w.Bp * H * 4);
            for (int l = 0; l <= p.L; ++l) w.buf[BUF_DHL0 + l] = dh[l & 1];
            for (int l = -1; l < p.L; ++l) w.buf[BUF_DCL0 + l] = dc[(l + 2) & 1];
            for (int l = 0; l < p.L; ++l) w.buf[BUF_DUL0 + l] = du;
        }
        w.part_w = take(w.M * w.part_slots * H * H * 4);
        w.part_b = take(w.M * w.part_slots * H * 4);
        w.dec_part = take((int64_t)w.M * DEC_BLOCKS * (DEC_MAXC * H + DEC_MAXC) * 4);
    } else if (!tc) {
        const int64_t a = take(slab), b = take(slab);
        for (int l = 0; l <= p.L; ++l) w.buf[BUF_H0 + l] = (l & 1) ? b : a;
        if (p.morph_sym) { const int64_t c = take(ctb); for (int l = 0; l < p.L; ++l) w.buf[BUF_CT0 + l] = c; }
    }
    if (tc) {
        for (int i = 0; i < 2; ++i) w.w16[i] = take((int64_t)w.M * p.n_mats16 * H * H * 2);
        if (train) {
            for (int l = 0; l <= p.L; ++l) for (int i = 0; i < 2; ++i) w.buf16[BUF_H0 + l][i] = take(slab / 2);
            if (p.morph_sym)
                for (int l = 0; l < p.L; ++l) for (int i = 0; i < 2; ++i) w.buf16[BUF_CT0 + l][i] = take(ctb / 2);
            if (!w.stack) {      // the per-layer launch sequence: backward ids alias two ping-pong images, as in MODE_FP32
                int64_t dh[2][2], dc[2][2], du[2] = {-1, -1};
                for (int b = 0; b < 2; ++b) for (int i = 0; i < 2; ++i) { dh[b][i] = take(slab / 2); dc[b][i] = take(slab / 2); }
                if (p.morph_sym) for (int i = 0; i < 2; ++i) du[i] = take((int64_t)p.nm * w.Bp * H * 2);
                for (int i = 0; i < 2; ++i) {
                    for (int l = 0; l <= p.L; ++l) w.buf16[BUF_DHL0 + l][i] = dh[l & 1][i];
                    for (int l = -1; l < p.L; ++l) w.buf16[BUF_DCL0 + l][i] = dc[(l + 2) & 1][i];
                    for (int l = 0; l < p.L; ++l) w.buf16[BUF_DUL0 + l][i] = du[i];
                }
            } else {
                // the dX chain of all layers runs in ONE launch ahead of the weight-gradient kernels: every layer keeps its own
                // dh / dc / du images (dh_l only where a residual or base_transform reads it: MS-HGNN models)
                for (int l = 0; l <= p.L; ++l) for (int i = 0; i < 2; ++i) {
                    if (p.morph_sym && l >= 1) w.buf16[BUF_DHL0 + l][i] = take(slab / 2);
                    w.buf16[BUF_DCL0 + l - 1][i] = take(slab / 2);       // dc_{-1} (encoder dpre) .. dc_{L-1}
                }
                if (p.morph_sym) for (int l = 0; l < p.L; ++l) for (int i = 0; i < 2; ++i) w.buf16[BUF_DUL0 + l][i] = take((int64_t)p.nm * w.Bp * H * 2);
            }
        } else {
            int64_t a[2], b[2], c[2] = {-1, -1};
            for (int i = 0; i < 2; ++i) { a[i] = take(slab / 2); b[i] = take(slab / 2); }
            if (p.morph_sym) for (int i = 0; i < 2; ++i) c[i] = take(ctb / 2);
            for (int l = 0; l <= p.L; ++l) for (int i = 0; i < 2; ++i) w.buf16[BUF_H0 + l][i] = (l & 1) ? b[i] : a[i];
            for (int l = 0; l < p.L; ++l) for (int i = 0; i < 2; ++i) w.buf16[BUF_CT0 + l][i] = c[i];
        }
    }
    if (tc) {
        for (int i = 0; i < 2; ++i) w.wenc16[i] = take((int64_t)w.M * p.n_types * H * p.enc_kmax * 2);
        w.enc_sync = take(256);
        if (train) {
            // row splits of the encoder weight gradient, fitted to whole waves like the layer-stack ones (16 units for the K4 model:
            // 512-row splits gave 64 CTAs on 148 SMs at 2048 graphs); each step must gain 3 %
            w.rows_per_enc = (int)fit_split_rows(B, (int64_t)p.enc_units.size(), 512, 1.0, 0.97, 128, 1024);
            w.n_splits_enc = (int)((B + w.rows_per_enc - 1) / w.rows_per_enc);
            w.part_enc_w = take((int64_t)w.M * p.enc_units.size() * w.n_splits_enc * H * 192 * 4);
            w.part_enc_b = take((int64_t)w.M * p.enc_units.size() * w.n_splits_enc * H * 4);
        }
    }
    if (w.stack) {
        w.stack_sync_bytes = ((int64_t)(p.L + 2) * (w.Bp / TILE_M) * p.S + 64) * 4;      // per (phase, row tile, node slot) completion counters + work counter + error word
        w.stack_sync = take(w.stack_sync_bytes);
    }
    if (p.padded) {
        w.pad_params = take(w.M * p.n_params * 4);
        if (train) w.pad_grads = take(w.M * p.n_params * 4);
    }
    w.loss_part = take((int64_t)w.M * LOSS_BLOCKS * 8);      // last: mshgnn_loss finds its partials at the end of the caller's workspace
    w.total = o;
    return w;
}

std::string describe_plan(const Plan& p) {
    std::ostringstream os;
    os << "{\"S\":" << p.S << ",\"L\":" << p.L << ",\"hidden\":" << p.hidden[0];
    if (p.n_models > 1) {
        os << ",\"hidden_models\":[";
        for (int m = 0; m < p.n_models; ++m) os << (m ? "," : "") << p.hidden[m];
        os << "]";
    }
    os << ",\"kernel_hidden\":" << H << ",\"n_params\":" << p.ext_base.back() << ",\"n_derived\":" << p.n_derived
       << ",\"n_tiles\":" << p.tiles.size() << ",\"n_rtasks\":" << p.rtasks.size() << ",\"n_rpairs\":" << p.rpairs.size()
       << ",\"n_groups\":" << p.groups.size() << ",\"n_mats16\":" << p.n_mats16 << ",\"enc_kmax\":" << p.enc_kmax
       << ",\"n_types\":" << p.n_types << ",\"need\":[";
    for (int l = 0; l <= p.L; ++l) {
        os << (l ? "," : "") << "[";
        for (int s = 0; s < p.S; ++s) os << (s ? "," : "") << (int)p.need[l][s];
        os << "]";
    }
    os << "],\"conv\":[";
    for (int l = 0; l < p.L; ++l) {
        os << (l ? "," : "") << "[";
        const Launch& La = p.conv_infer[l];
        for (int i = 0; i < La.count; ++i) {
            const Tile& T = p.tiles[La.begin + i];
            os << (i ? "," : "") << "{\"out_buf\":" << T.out_buf << ",\"out_slot\":" << T.out_slot << ",\"relu\":" << T.relu
               << ",\"res\":" << T.res_buf << ",\"src\":[";
            for (int c = 0; c < T.n_chunks; ++c) os << (c ? "," : "") << "[" << T.chunks[c].a_slot << "," << T.chunks[c].w_off << "]";
            os << "]}";
        }
        os << "]";
    }
    os << "],\"mac_rows_fwd\":";
    int64_t rows = 0;
    for (int l = 0; l < p.L; ++l) {
        for (int i = 0; i < p.conv_infer[l].count; ++i) rows += p.tiles[p.conv_infer[l].begin + i].n_chunks;
        rows += p.mlp1[l].count + p.mlp2[l].count;
    }
    os << rows << "}";
    return os.str();
}

}  // namespace mshgnn
