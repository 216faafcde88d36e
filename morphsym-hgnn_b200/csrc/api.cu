// C ABI of libmshgnn_b200.so (see include/mshgnn_b200.h): launch sequencing of the hot path.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <vector>

#include "kernels_simt.cuh"
#include "kernels_tc.cuh"
#include "kernels_enc.cuh"
#include "kernels_dx.cuh"
#include "kernels_stack.cuh"
#include "kernels_stack2.cuh"
#include "kernels_pad.cuh"
#include "plan.cuh"
#include "windows.cuh"
#include "metrics.cuh"

using namespace mshgnn;

struct mshgnn_plan {
    Plan p;
};

namespace {

thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                     \
    do {                                                                                   \
        cudaError_t _e = (expr);                                                           \
        if (_e != cudaSuccess)                                                             \
            return fail(MSHGNN_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

// ---- per-kernel event profiling ----
enum Kind : int { K_DERIVE = 0, K_ENC_FWD, K_CONV_FWD, K_MLP_FWD, K_DEC_FWD, K_LOSS, K_DEC_BWD, K_MLP_BWD, K_DX_BWD,
                  K_DW_LAYER, K_DW_ENC, K_REDUCE, K_OPTIM, K_MEMSET, K_WINDOWS, K_METRICS, K_STACK_FWD, K_STACK_BWD, K_EDGES, K_DX_ENC, K_PAD, K_NKINDS };
static_assert(K_NKINDS == MSHGNN_NUM_KERNEL_KINDS, "kernel kind table out of sync with the header");
constexpr int K_NKINDS_V1 = 19;      // kinds before dx_encoder: mshgnn_profile_read still accepts n = 19 (and 20) from callers built against older headers
const char* const kKindNames[MSHGNN_NUM_KERNEL_KINDS] = {
    "derive_weights", "encoder_fwd", "conv_fwd", "base_mlp_fwd", "decoder_fwd", "loss",
    "decoder_bwd", "base_mlp_bwd", "dx_bwd", "dw_layers", "dw_encoder",
    "reduce_partials", "optimizer", "memset", "window_builder", "step_metrics", "stack_fwd", "stack_bwd", "check_edges", "dx_encoder", "pad_params"};
struct ProfRec { int kind; cudaEvent_t a, b; };
std::mutex g_prof_mu;
bool g_prof_on = false;
std::vector<ProfRec> g_prof;
std::vector<cudaEvent_t> g_prof_pool;

struct ProfScope {
    cudaStream_t st; cudaEvent_t a = nullptr, b = nullptr; int kind; bool on;
    ProfScope(int k, cudaStream_t s) : st(s), kind(k), on(g_prof_on) {
        if (!on) return;
        std::lock_guard<std::mutex> lk(g_prof_mu);
        auto get = [&]() { cudaEvent_t e; if (!g_prof_pool.empty()) { e = g_prof_pool.back(); g_prof_pool.pop_back(); } else cudaEventCreate(&e); return e; };
        a = get(); b = get();
        cudaEventRecord(a, st);
    }
    ~ProfScope() {
        if (!on) return;
        cudaEventRecord(b, st);
        std::lock_guard<std::mutex> lk(g_prof_mu);
        g_prof.push_back({kind, a, b});
    }
};

#define LAUNCH_CHECK()                                                                     \
    do {                                                                                   \
        g_launches.fetch_add(1, std::memory_order_relaxed);                                \
        cudaError_t _e = cudaGetLastError();                                               \
        if (_e != cudaSuccess)                                                             \
            return fail(MSHGNN_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

template <typename T>
int upload(const Plan& p, const std::vector<T>& v, T** d) {
    *d = nullptr;
    if (v.empty()) return 0;
    CUDA_TRY(cudaMalloc((void**)d, v.size() * sizeof(T)));
    p.d_allocs.push_back(*d);
    CUDA_TRY(cudaMemcpy(*d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return 0;
}

int ensure_uploaded(const Plan& p) {
    std::lock_guard<std::mutex> lk(p.mu);
    int dev = -1;
    CUDA_TRY(cudaGetDevice(&dev));
    if (p.uploaded) {
        if (dev != p.device) return fail(MSHGNN_ERR_ARG, "plan tables live on device %d but the current device is %d", p.device, dev);
        return 0;
    }
    int rc;
    if ((rc = upload(p, p.tiles, &p.d_tiles))) return rc;
    if ((rc = upload(p, p.stack_items, &p.d_stack_items))) return rc;
    {
        std::vector<int> tpl;
        for (int e = 0; e < p.n_etypes; ++e) { tpl.insert(tpl.end(), p.e_src[e].begin(), p.e_src[e].end()); tpl.insert(tpl.end(), p.e_dst[e].begin(), p.e_dst[e].end()); }
        if (tpl.empty()) tpl.push_back(0);
        if ((rc = upload(p, tpl, &p.d_edge_tpl))) return rc;
    }
    if ((rc = upload(p, p.rtasks, &p.d_rtasks))) return rc;
    if ((rc = upload(p, p.rpairs, &p.d_rpairs))) return rc;
    if ((rc = upload(p, p.groups, &p.d_groups))) return rc;
    if ((rc = upload(p, p.derive_ops, &p.d_derive))) return rc;
    if ((rc = upload(p, p.derive16_ops, &p.d_derive16))) return rc;
    if ((rc = upload(p, p.signs, &p.d_signs))) return rc;
    if ((rc = upload(p, p.enc_units, &p.d_enc_units))) return rc;
    if ((rc = upload(p, p.enc_groups, &p.d_enc_groups))) return rc;
    if ((rc = upload(p, p.dx_units, &p.d_dx_units))) return rc;
    if ((rc = upload(p, p.pad_segs, &p.d_pad_segs))) return rc;
    p.device = dev;
    p.uploaded = true;
    return 0;
}

// device pointers of the workspace buffers (ws_layout placed them); params, grads and the feature tensors are the caller's
void fill_bufs(const Plan& p, const WsLayout& w, char* ws, BufTable& bt) {
    for (int id = 0; id < MAX_BUFS; ++id) bt.p[id] = w.buf[id] < 0 ? nullptr : ws + w.buf[id];
    bt.p[BUF_SIGNS] = p.d_signs;
}

// first 256-byte row of every fp16 image relative to the workspace base (one TMA map then covers all of them)
void fill_rows16(const WsLayout& w, BufRows& br) {
    auto row = [](int64_t off) { return off < 0 ? 0 : (int)(off / 256); };
    for (int id = 0; id < MAX_BUFS; ++id) { br.hi[id] = row(w.buf16[id][0]); br.lo[id] = row(w.buf16[id][1]); }
    br.w_hi = row(w.w16[0]); br.w_lo = row(w.w16[1]);
}

// image i (0 = hi, 1 = lo) of a buffer id, NULL when the layout has none
__half* image16(char* ws, const WsLayout& w, int id, int i) { return w.buf16[id][i] < 0 ? nullptr : (__half*)(ws + w.buf16[id][i]); }

int launch_rowgemm(int kind, const Plan& p, const Launch& L, const BufTable& bt, int64_t B, int64_t Bp, int x_f64, cudaStream_t st) {
    if (L.count == 0) return 0;
    ProfScope ps(kind, st);
    dim3 grid((unsigned)(Bp / TILE_M), (unsigned)L.count);
    k_rowgemm<<<grid, 256, 0, st>>>(p.d_tiles + L.begin, bt, B, Bp, x_f64);
    LAUNCH_CHECK();
    return 0;
}

// ---- tensor-core launches ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// cuTensorMapEncodeTiled with unit element strides; `what` names the tensor in the error text
int encode_map(CUtensorMap* m, CUtensorMapDataType type, cuuint32_t rank, const void* base, const cuuint64_t* dims, const cuuint64_t* strides,
               const cuuint32_t* box, CUtensorMapSwizzle sw, const char* what) {
    static EncodeTiledFn enc = nullptr;
    if (!enc) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || !ptr) return fail(MSHGNN_ERR_CUDA, "cuTensorMapEncodeTiled is not available in this driver");
        enc = (EncodeTiledFn)ptr;
    }
    // cuTensorMapEncodeTiled is a driver call and needs a context current on THIS thread.  The runtime binds the primary
    // context lazily: a thread that has not yet made a context-binding runtime call - PyTorch's autograd worker when the
    // caching allocator serves every allocation of its first backward from cached blocks - fails here with
    // CUDA_ERROR_INVALID_CONTEXT (201).  cudaFree(0) binds it; once per thread.
    static thread_local bool ctx_bound = false;
    if (!ctx_bound) { CUDA_TRY(cudaFree(0)); ctx_bound = true; }
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(m, type, rank, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(MSHGNN_ERR_CUDA, "cuTensorMapEncodeTiled%s failed with CUresult %d", what, (int)r);
    return 0;
}

// [rows, cols] fp16 row-major tensor viewed through a (box_cols x box_rows) box with the given swizzle
int make_map_2d(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int box_cols, int box_rows, CUtensorMapSwizzle sw) {
    if (!base || rows < 1) return fail(MSHGNN_ERR_ARG, "internal: bad fp16 tensor for a TMA map");
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
    const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    return encode_map(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, base, dims, strides, box, sw, "");
}

// The caller's fp32 feature tensor x[B * nodes, K] of one node type as a (K, nodes, B) tensor, box = 64 columns x 1 node x 128 graphs:
// one TMA request fetches the 256-byte fragments of a K block of 128 consecutive graphs of one node slot (k_tc_encoder_stream).
// The input gradient (k_tc_encoder_dx) stores through the same view: box 32 columns x 1 x 128 graphs, SWIZZLE_128B.
int make_map_x3d(CUtensorMap* m, const void* base, int64_t B, int nodes, int K, int box_rows = 128, int box_cols = 64,
                 CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_NONE) {
    const cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)nodes, (cuuint64_t)B};
    const cuuint64_t strides[2] = {(cuuint64_t)K * 4, (cuuint64_t)nodes * K * 4};
    const cuuint32_t box[3] = {(cuuint32_t)box_cols, 1, (cuuint32_t)box_rows};
    return encode_map(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, sw, " (features)");
}

// The whole workspace as one [total/256 rows][128 fp16] tensor: every (hi, lo) image of every buffer (and the 128x128
// weight images) is a row range of it, so three maps serve every tensor-core launch of a call.
struct WsMaps {
    TcMaps tc;            // .k: 32 x 128 SWIZZLE_64B (operand K blocks), .o: 64 x 128 SWIZZLE_128B (epilogue tiles)
    CUtensorMap dw;       // 64 x 64 SWIZZLE_128B (MN-major operands of the weight-gradient kernels)
};
int make_ws_maps(WsMaps* m, const void* ws, const WsLayout& w) {
    if (w.total / 256 > 0x7fffffffLL) return fail(MSHGNN_ERR_ARG, "workspace too large for one TMA map");
    int rc;
    if ((rc = make_map_2d(&m->tc.k, ws, w.total / 256, H, TC_KB, 128, CU_TENSOR_MAP_SWIZZLE_64B))) return rc;
    if ((rc = make_map_2d(&m->tc.o, ws, w.total / 256, H, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    if ((rc = make_map_2d(&m->dw, ws, w.total / 256, H, 64, DW_KB, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    return 0;
}

// per-device state: a process may drive several GPUs (one plan / model per device)
constexpr int MAX_DEVICES = 64;
int sm_count(int* out) {
    static std::atomic<int> n[MAX_DEVICES];
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    int v = dev < MAX_DEVICES ? n[dev].load(std::memory_order_relaxed) : 0;
    if (!v) {
        CUDA_TRY(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev));
        if (dev < MAX_DEVICES) n[dev].store(v, std::memory_order_relaxed);
    }
    *out = v;
    return 0;
}
// true the first time it is called on the current device for this flag set (cudaFuncSetAttribute is per device)
bool first_on_device(std::atomic<bool> (&flags)[MAX_DEVICES]) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEVICES) return true;
    return !flags[dev].exchange(true);
}

// encoder kernel choice: -1 = default (persistent TMA-fed kernel when the inputs allow it), 0 persistent, 1 one tile per CTA, 2 two tiles per CTA;
// rows tiles per item of the persistent kernel: 0 = by batch size, 1, 2 (mshgnn_set_option "encoder" / "encoder_tpi"; same-process A/B and bit-identity tests)
static std::atomic<int> g_encoder_kernel{-1}, g_encoder_tpi{0}, g_encoder_dw_tma{-1};

int launch_tc_encoder(const Plan& p, const Launch& L, const WsLayout& w, const BufTable& bt, const BufRows& br, const WsMaps& wm, char* ws,
                      const float* params, int64_t B, int xf64, int split, cudaStream_t st) {
    if (L.count == 0) return 0;
    static std::atomic<bool> attr_set[64];
    // a model batch runs the two-tile kernel, the one that knows which model a row tile belongs to (the kernels give identical bits)
    const int opt = g_encoder_kernel.load();
    const int which = w.M > 1 ? 2 : (opt >= 0 ? opt : 0);
    if (first_on_device(attr_set)) {
        CUDA_TRY(cudaFuncSetAttribute(k_tc_encoder, cudaFuncAttributeMaxDynamicSharedMemorySize, ENC_SMEM_BYTES));
        CUDA_TRY(cudaFuncSetAttribute(k_tc_encoder_pair, cudaFuncAttributeMaxDynamicSharedMemorySize, ENCP_SMEM_BYTES));
        CUDA_TRY(cudaFuncSetAttribute(k_tc_encoder_stream, cudaFuncAttributeMaxDynamicSharedMemorySize, ENQ_SMEM_BYTES));
    }
    __half* e_hi = (__half*)(ws + w.wenc16[0]);
    __half* e_lo = (__half*)(ws + w.wenc16[1]);
    EncMaps maps;
    int rc;
    if ((rc = make_map_2d(&maps.w_hi, e_hi, (int64_t)w.M * p.n_types * H, p.enc_kmax, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    if ((rc = make_map_2d(&maps.w_lo, e_lo, (int64_t)w.M * p.n_types * H, p.enc_kmax, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    maps.o = wm.tc.o;
    // the persistent kernel copies row fragments with cp.async.bulk: fp32 features, every 64-column fragment 16-byte aligned
    bool stream_ok = xf64 == 0 && L.count <= ENQ_MAX_SLOTS;
    for (int i = 0; i < L.count && stream_ok; ++i) {
        const Chunk& ch = p.tiles[L.begin + i].chunks[0];
        stream_ok = ch.a_buf >= BUF_X0 && ch.a_buf < BUF_X0 + p.n_types && enq_rows_ok(bt.p[ch.a_buf], ch.K, ch.sign_off);
    }
    ProfScope ps(K_ENC_FWD, st);
    const unsigned n_row_tiles = (unsigned)(w.Bp / TILE_M);
    if (which == 1) k_tc_encoder<<<dim3(n_row_tiles, (unsigned)L.count), ENC_THREADS, ENC_SMEM_BYTES, st>>>(maps, p.d_tiles + L.begin, bt, br, B, w.Bp, xf64, split);
    else if (which == 2 || !stream_ok) {
        const unsigned pairs = (unsigned)(w.M * ((w.Bm / TILE_M + 1) / 2));     // per model: its row-tile pairs
        k_tc_encoder_pair<<<dim3(pairs, (unsigned)L.count), ENC_THREADS, ENCP_SMEM_BYTES, st>>>(maps, p.d_tiles + L.begin, bt, br, B, w.Bp, xf64, split, /*enc_prefetch*/ 0,
                                                                                          w.Bm, p.n_types * H, p.n_params);
    } else {
        // persistent kernel: one CTA per SM draws (node slot, row-tile pair) items from the counter the forward prologue zeroed
        int n_sm = 0;
        if ((rc = sm_count(&n_sm))) return rc;
        // two row tiles per item (they share every weight stage) only when that leaves every SM several items: at 2048 graphs 64 long and
        // 96 short pair items on 148 SMs would make two long items the critical path (1.5 x the balanced time); single tiles balance
        const int opt_tpi = g_encoder_tpi.load();
        const int tpi = opt_tpi ? opt_tpi : ((int64_t)L.count * ((n_row_tiles + 1) / 2) >= 4 * (int64_t)n_sm ? 2 : 1);
        const int64_t n_items = (int64_t)L.count * ((n_row_tiles + tpi - 1) / tpi);
        const unsigned grid = (unsigned)(n_items < n_sm ? n_items : n_sm);
        EnqMaps em;
        em.w_hi = maps.w_hi; em.w_lo = maps.w_lo; em.o = maps.o;
        for (int t = 0; t < p.n_types; ++t) {
            if (p.in_w[t] % 4 || (reinterpret_cast<uintptr_t>(bt.p[BUF_X0 + t]) & 15)) { em.x[t] = maps.o; continue; }      // no slot of this launch reads it (stream_ok)
            if ((rc = make_map_x3d(&em.x[t], bt.p[BUF_X0 + t], B, p.nodes[t], p.in_w[t]))) return rc;
        }
        for (int t = p.n_types; t < 4; ++t) em.x[t] = maps.o;
        k_tc_encoder_stream<<<grid, ENQ_THREADS, ENQ_SMEM_BYTES, st>>>(em, p.d_tiles + L.begin, L.count, (int)BUF_X0, bt, br, B, w.Bp, split, (uint32_t*)(ws + w.enc_sync), tpi,
                                                                       /*pf*/ 0, /*dbg*/ 0);
    }
    LAUNCH_CHECK();
    return 0;
}

int launch_tc_rowgemm(int kind, const Plan& p, const Launch& L, const BufTable& bt, const BufRows& br, const WsMaps& wm,
                      int64_t B, int64_t Bp, int split, cudaStream_t st) {
    if (L.count == 0) return 0;
    static std::atomic<bool> attr_set[64];
    if (first_on_device(attr_set)) {
        CUDA_TRY(cudaFuncSetAttribute(k_tc_rowgemm, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_BYTES));
        CUDA_TRY(cudaFuncSetAttribute(k_tc_rowgemm_persistent, cudaFuncAttributeMaxDynamicSharedMemorySize, PK_SMEM_BYTES));
        CUDA_TRY(cudaFuncSetAttribute(k_tc_rowgemm_pair, cudaFuncAttributeMaxDynamicSharedMemorySize, PP_SMEM_BYTES));
    }
    for (int i = 0; i < L.count; ++i)
        for (int c = 0; c < p.tiles[L.begin + i].n_chunks; ++c)
            if (p.tiles[L.begin + i].chunks[c].a_kind != A_SLAB)
                return fail(MSHGNN_ERR_ARG, "internal: a tensor-core row-GEMM launch must read slab buffers");
    ProfScope ps(kind, st);
    if (L.count > PK_MAX_TILES) {
        dim3 grid((unsigned)L.count, (unsigned)(Bp / TILE_M));
        k_tc_rowgemm<<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(wm.tc, p.d_tiles + L.begin, bt, br, B, Bp, split);
    } else {
        int n_sm = 0, rc;
        if ((rc = sm_count(&n_sm))) return rc;
        // two row tiles per item (shared weight stages) only when that still leaves every SM >= 4 items: short launches
        // (base MLP: 4-8 output tiles) lose more to wave quantisation than they gain from the smaller operand stream
        const bool pair = Bp >= 2 * TILE_M && (int64_t)L.count * ((Bp / TILE_M + 1) / 2) >= 4 * (int64_t)n_sm;
        const int64_t n_items = (int64_t)L.count * (pair ? (Bp / TILE_M + 1) / 2 : Bp / TILE_M);
        if (n_items > 0x7fffffffLL) return fail(MSHGNN_ERR_ARG, "batch too large for one row-GEMM launch");
        const unsigned grid = (unsigned)(n_items < n_sm ? n_items : n_sm);
        // programmatic stream serialization: the prologue of this grid overlaps the tail of the previous kernel (the
        // kernel itself waits with griddepcontrol.wait before touching anything that kernel wrote)
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(PK_THREADS); cfg.dynamicSmemBytes = pair ? PP_SMEM_BYTES : PK_SMEM_BYTES; cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = g_prof_on ? 0 : 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        const Tile* d_tiles = p.d_tiles + L.begin;
        const int n_tiles = L.count, n_it = (int)n_items;
        if (pair) CUDA_TRY(cudaLaunchKernelEx(&cfg, k_tc_rowgemm_pair, wm.tc, d_tiles, n_tiles, n_it, bt, br, B, Bp, split));
        else CUDA_TRY(cudaLaunchKernelEx(&cfg, k_tc_rowgemm_persistent, wm.tc, d_tiles, n_tiles, n_it, bt, br, B, Bp, split));
    }
    LAUNCH_CHECK();
    return 0;
}

int launch_tc_dw(int kind, const Plan& p, int layer, const Launch& L, const WsLayout& w, const BufRows& br, const WsMaps& wm, int64_t B, int split,
                 float* part_w, float* part_b, cudaStream_t st) {
    if (L.count == 0) return 0;
    static std::atomic<bool> attr_set[64];
    if (first_on_device(attr_set)) CUDA_TRY(cudaFuncSetAttribute(k_tc_reducegemm, cudaFuncAttributeMaxDynamicSharedMemorySize, DW_SMEM_BYTES));
    for (int i = 0; i < L.count; ++i) {
        const RTask& T = p.rtasks[L.begin + i];
        if (T.n_pairs > DW_MAX_PAIRS) return fail(MSHGNN_ERR_ARG, "internal: weight-gradient task with more than %d pairs", DW_MAX_PAIRS);
        for (int j = 0; j < T.n_pairs; ++j)
            if (p.rpairs[T.pair_begin + j].a_kind != A_SLAB) return fail(MSHGNN_ERR_ARG, "internal: tensor-core weight-gradient task must read slabs");
    }
    ProfScope ps(kind, st);
    dim3 grid((unsigned)L.count, (unsigned)(w.M * w.dw_ns[layer]));          // per model: the wave-fitted row splits of this layer (ws_layout)
    k_tc_reducegemm<<<grid, TC_THREADS, DW_SMEM_BYTES, st>>>(wm.dw, p.d_rtasks, p.d_rpairs, L.begin, br, B, w.Bp, w.dw_rows[layer], w.dw_slot0[layer],
                                                             split, part_w, part_b, w.Bm, w.dw_ns[layer], w.part_slots);
    LAUNCH_CHECK();
    return 0;
}

// ---- cross-layer stack kernel (kernels_stack.cuh) ----
// Item order of the stack kernel (kernels_stack.cuh): row chunks of RC row tiles, walked phase by phase.
// RC trades the two things the kernel is sensitive to (cycle counters of an instrumented build, profiles/r2_stack_timing.txt, 16384 graphs, K4 Mini Cheetah):
//   * dependency distance: the items of layer l + 1 of a row tile are handed out RC x (items per row tile and layer) items
//     after those of layer l; below ~2 x 148 items in flight + the latency of the slowest item (a base_transform chain) the
//     scheduler warps wait (RC = 24: 22 % of the kernel in queue waits, RC = 32: 9 %, RC = 48: 7 %);
//   * L2 residency: a chunk's input and output slabs of one layer are RC x 2 x S x 128 x 512 B (RC = 32: 84 MB of 126 MB).
// The diagonal wavefront (uniform distance D x items per slot) was measured 5 % slower at equal footprint (all layers'
// weights and buffers are live at once); the host always selects the chunked order.
int stack_rows_per_chunk(const Plan& p) {
    const int64_t per_row_tile = (int64_t)2 * p.S * TILE_M * H * 4;
    int rc = (int)((int64_t)84 * 1024 * 1024 / per_row_tile);
    return rc < 16 ? 16 : (rc > 64 ? 64 : rc);
}

int stack_sync_reset(const WsLayout& w, char* ws, cudaStream_t st) {
    if (!w.stack) return 0;
    ProfScope ps(K_MEMSET, st);
    CUDA_TRY(cudaMemsetAsync(ws + w.stack_sync, 0, (size_t)w.stack_sync_bytes, st));
    return 0;
}

int launch_stack(int kind, const Plan& p, const Plan::Stack& sp, const WsLayout& w, const BufTable& bt, const BufRows& br, const WsMaps& wm,
                 char* ws, int64_t B, int split, cudaStream_t st) {
    if (sp.prog.n_phases == 0) return 0;
    static std::atomic<bool> attr_set[64];
    if (first_on_device(attr_set)) {
        CUDA_TRY(cudaFuncSetAttribute(k_tc_stack<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SK_SMEM_BYTES));
        CUDA_TRY(cudaFuncSetAttribute(k_tc_stack<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SK_SMEM_BYTES));
    }
    bool has_priv = false;               // thread-private fp32 tensors in this program (kernels_stack.cuh): selects the PRIV instantiation
    for (int i = 0; i < sp.tiles.count; ++i) {
        const Tile& T = p.tiles[sp.tiles.begin + i];
        has_priv = has_priv || T.priv != 0;
        for (int c = 0; c < T.n_chunks; ++c)
            if (T.chunks[c].a_kind != A_SLAB) return fail(MSHGNN_ERR_ARG, "internal: a stack program must read slab buffers");
    }
    int n_prog_items = 0;
    for (int ph = 0; ph < sp.prog.n_phases; ++ph) n_prog_items = std::max(n_prog_items, sp.prog.first_item[ph] + sp.prog.n_items[ph]);
    for (int i = 0; i < n_prog_items; ++i) {
        const StackItem& it = p.stack_items[sp.item0 + i];
        int chunks = 0;
        for (int st_ = 0; st_ < it.n_steps; ++st_) chunks += p.tiles[sp.tiles.begin + it.tile + st_].n_chunks;
        if (chunks > SK_QCHUNKS || it.n_steps > SK_QSTEPS) return fail(MSHGNN_ERR_ARG, "internal: stack item with %d chunks / %d steps (queue holds %d / %d)", chunks, it.n_steps, SK_QCHUNKS, SK_QSTEPS);
    }
    StackArgs a;
    a.prog = sp.prog;
    a.n_row_tiles = (int)(w.Bp / TILE_M);
    const int64_t n_total = (int64_t)a.n_row_tiles * sp.prog.items_per_row;
    if (n_total > 0x7fffffffLL) return fail(MSHGNN_ERR_ARG, "batch too large for one stack launch");
    a.n_total = (int)n_total;
    a.split = split; a.B = B; a.Bp = w.Bp; a.n_slots = p.S;
    a.tiles_m = (int)(w.Bm / TILE_M); a.w16_rows = p.n_mats16 * H; a.n_params = (int)p.n_params; a.n_derived = (int)p.n_derived;
    a.sync = (uint32_t*)(ws + w.stack_sync);
    a.err = (uint32_t*)(ws + w.stack_sync + w.stack_sync_bytes - 4);
    a.next = (uint32_t*)(ws + w.stack_sync + w.stack_sync_bytes - 8);
    a.ws = ws;
    a.debug = 0;
    if ((int64_t)sp.prog.n_phases * a.n_row_tiles * p.S + 2 > w.stack_sync_bytes / 4) return fail(MSHGNN_ERR_WORKSPACE, "internal: stack counters do not fit");
    int n_sm = 0, rc;
    if ((rc = sm_count(&n_sm))) return rc;
    // an item drawn long before it runs delays its dependents: the scheduler warp stays one item ahead of the producer
    a.lookahead = 1;
    a.chunked = 1;
    a.delay = stack_rows_per_chunk(p);
    if (w.stack_pair) {
        // CTA-pair kernel: items are (phase, row-tile pair, node slot); one cluster of two CTAs per TPC
        if (a.n_row_tiles & 1) return fail(MSHGNN_ERR_ARG, "internal: the CTA-pair stack kernel needs an even number of row tiles");
        static std::atomic<bool> attr2_set[64];
        static std::atomic<int> max_clusters[64];
        int dev = 0;
        CUDA_TRY(cudaGetDevice(&dev));
        if (first_on_device(attr2_set)) {
            CUDA_TRY(cudaFuncSetAttribute(k_tc_stack2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, S2_SMEM_BYTES));
            CUDA_TRY(cudaFuncSetAttribute(k_tc_stack2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, S2_SMEM_BYTES));
        }
        const int64_t n_pairs_total = (int64_t)(a.n_row_tiles / 2) * sp.prog.items_per_row;
        a.n_total = (int)n_pairs_total;
        a.delay = std::max(a.delay / 2, 1);
        cudaLaunchConfig_t cfg = {};
        cfg.blockDim = dim3(SK_THREADS); cfg.dynamicSmemBytes = S2_SMEM_BYTES; cfg.stream = st;
        cudaLaunchAttribute at[2];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[1].val.programmaticStreamSerializationAllowed = g_prof_on ? 0 : 1;
        cfg.attrs = at; cfg.numAttrs = 2;
        int mc = dev < 64 ? max_clusters[dev].load(std::memory_order_relaxed) : 0;
        if (!mc) {
            cfg.gridDim = dim3((unsigned)n_sm);
            CUDA_TRY(cudaOccupancyMaxActiveClusters(&mc, k_tc_stack2<true>, &cfg));
            if (mc < 1) return fail(MSHGNN_ERR_CUDA, "the CTA-pair stack kernel does not fit on this device (0 active clusters)");
            if (dev < 64) max_clusters[dev].store(mc, std::memory_order_relaxed);
        }
        const int64_t clusters = n_pairs_total < mc ? n_pairs_total : mc;
        cfg.gridDim = dim3((unsigned)(2 * clusters));
        const Tile* d_tiles = p.d_tiles + sp.tiles.begin;
        const StackItem* d_items = p.d_stack_items + sp.item0;
        ProfScope ps(kind, st);
        if (has_priv) CUDA_TRY(cudaLaunchKernelEx(&cfg, k_tc_stack2<true>, wm.tc, wm.dw, d_tiles, d_items, a, bt, br));
        else CUDA_TRY(cudaLaunchKernelEx(&cfg, k_tc_stack2<false>, wm.tc, wm.dw, d_tiles, d_items, a, bt, br));
        LAUNCH_CHECK();
        return 0;
    }
    ProfScope ps(kind, st);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(n_total < n_sm ? n_total : n_sm)); cfg.blockDim = dim3(SK_THREADS); cfg.dynamicSmemBytes = SK_SMEM_BYTES; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = g_prof_on ? 0 : 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    const Tile* d_tiles = p.d_tiles + sp.tiles.begin;
    const StackItem* d_items = p.d_stack_items + sp.item0;
    if (has_priv) CUDA_TRY(cudaLaunchKernelEx(&cfg, k_tc_stack<true>, wm.tc, d_tiles, d_items, a, bt, br));
    else CUDA_TRY(cudaLaunchKernelEx(&cfg, k_tc_stack<false>, wm.tc, d_tiles, d_items, a, bt, br));
    LAUNCH_CHECK();
    return 0;
}

// Grid z and per-model strides of the pad / compaction kernels for a call on M models: a plan of one model repeats its table
// for every model (z = M), a mixed plan's table already covers every model with absolute offsets (z = 1, strides 0).
struct PadGrid { unsigned z; int64_t ext_n, in_n; };
PadGrid pad_grid(const Plan& p, int M) {
    if (p.n_models > 1) return {1u, 0, 0};
    return {(unsigned)M, p.ext_base.back(), p.n_params};
}
unsigned pad_grid_y(int count) { return (unsigned)std::min(count, PAD_MAX_GRID_Y); }

// padded plans: caller's gradients of the tensors segs [first, first + count) from the internal 128-wide gradient buffer
int compact_grads(const Plan& p, int M, int first, int count, const float* in, float* ext, cudaStream_t st) {
    if (count == 0) return 0;
    const PadGrid g = pad_grid(p, M);
    ProfScope ps(K_PAD, st);
    k_compact_grads<<<dim3(PAD_BLOCKS_X, pad_grid_y(count), g.z), 256, 0, st>>>(p.d_pad_segs + first, count, in, ext, g.in_n, g.ext_n);
    LAUNCH_CHECK();
    return 0;
}

// Tensor-core modes carry every backward quantity multiplied by a power of two G ~ #output rows so that the fp16 (hi, lo)
// images of dL/dh stay in the normal range; the weight-gradient reductions and the input gradient multiply by 1/G (exact).
float grad_scale(const Plan& p, int64_t B) {
    int e = 0;
    std::frexp((double)(B * p.dec.n_dec), &e);
    return (float)std::ldexp(1.0, e - 1);
}

int check_plan_mode(const mshgnn_plan* plan, int32_t mode) {
    if (!plan) return fail(MSHGNN_ERR_ARG, "plan is NULL");
    if (mode != MSHGNN_MODE_FP32 && mode != MSHGNN_MODE_TC && mode != MSHGNN_MODE_TC_1X) return fail(MSHGNN_ERR_ARG, "unknown mode %d", mode);
    return 0;
}

// What forward, backward and input_grad share for one call on a workspace.  open_call checks the workspace and lays it out;
// bind_call, after the entry point's own checks, uploads the plan and resolves every buffer the kernels address.
struct Call {
    const Plan* p = nullptr;
    WsLayout w;
    char* ws = nullptr;
    bool tc = false;
    int split = 0;                     // MSHGNN_MODE_TC: (hi, lo) products; MSHGNN_MODE_TC_1X: hi products only
    float G = 1.f;                     // grad_scale in the tensor-core modes
    const float* params = nullptr;     // the kernels' parameters and gradients: a padded plan's 128-wide workspace buffers
    float* grads = nullptr;
    BufTable bt;
    BufRows br;
    WsMaps wm;                         // tensor-core modes
};

// What a model batch of M models supports; checked before the device is touched
int check_models(const Plan& p, int64_t M, int64_t B, int32_t mode) {
    if (M < 1) return fail(MSHGNN_ERR_ARG, "M must be >= 1 (got %lld)", (long long)M);
    if (p.n_models > 1 && M != p.n_models)
        return fail(MSHGNN_ERR_ARG, "the plan describes a model batch of %d models: M must be %d (got %lld)", p.n_models, p.n_models, (long long)M);
    if (B < 1) return fail(MSHGNN_ERR_ARG, "B must be >= 1 (got %lld)", (long long)B);
    if (M == 1) return 0;
    if (mode == MSHGNN_MODE_FP32) return fail(MSHGNN_ERR_ARG, "model batches (M = %lld) run in the tensor-core modes only", (long long)M);
    if (!stack_enabled() || p.stack_infer.prog.n_phases == 0) return fail(MSHGNN_ERR_ARG, "model batches (M = %lld) need the cross-layer stack kernel (option 'stack')", (long long)M);
    if (M * std::max(p.n_params, p.n_derived) > 0x7fffffffLL || M * p.n_mats16 * H > 0x7fffffffLL || M * B > 0x7fffffffLL)
        return fail(MSHGNN_ERR_ARG, "model batch of %lld models too large", (long long)M);
    // grid.y / grid.z of the per-model launches: M x (up to 64 row splits) for the weight-gradient kernels, M elsewhere
    if (M > 65535 / 64) return fail(MSHGNN_ERR_ARG, "model batch of %lld models: at most %d models per call", (long long)M, 65535 / 64);
    return 0;
}

int open_call(Call& c, const mshgnn_plan* plan, int64_t M, int64_t B, int train, int32_t mode, void* ws, int64_t ws_bytes) {
    const Plan& p = plan->p;
    int rc;
    if ((rc = check_models(p, M, B, mode))) return rc;      // before ws_layout, which needs B >= 1
    c.p = &p;
    c.w = ws_layout(p, B, train, mode, (int)M);
    if (!ws) return fail(MSHGNN_ERR_ARG, "workspace is NULL");
    if (ws_bytes < c.w.total) return fail(MSHGNN_ERR_WORKSPACE, "workspace too small: %lld < %lld bytes", (long long)ws_bytes, (long long)c.w.total);
    if (reinterpret_cast<uintptr_t>(ws) & 255) return fail(MSHGNN_ERR_ARG, "workspace must be 256-byte aligned");
    c.ws = (char*)ws;
    c.tc = mode != MSHGNN_MODE_FP32;
    c.split = mode == MSHGNN_MODE_TC;
    c.G = c.tc ? grad_scale(p, B) : 1.f;
    return 0;
}

// x: the caller's feature tensors (NULL: the call reads none)
int bind_call(Call& c, const float* params, float* grads, const void* const* x) {
    const Plan& p = *c.p;
    int rc;
    if ((rc = ensure_uploaded(p))) return rc;
    if (p.padded) {     // the forward's 128-wide zero-padded parameter copy; gradients go to the 128-wide buffer, then compacted
        params = (const float*)(c.ws + c.w.pad_params);
        if (grads) grads = (float*)(c.ws + c.w.pad_grads);
    }
    c.params = params;
    c.grads = grads;
    fill_bufs(p, c.w, c.ws, c.bt);
    c.bt.p[BUF_PARAMS] = (void*)params;
    c.bt.p[BUF_GRADS] = grads;
    for (int t = 0; x && t < p.n_types; ++t) {
        if (!x[t]) return fail(MSHGNN_ERR_ARG, "x[%d] is NULL", t);
        c.bt.p[BUF_X0 + t] = (void*)x[t];
    }
    fill_rows16(c.w, c.br);
    if (c.tc && (rc = make_ws_maps(&c.wm, c.ws, c.w))) return rc;
    return 0;
}

// tensor-core encoder weight gradient: split partials of every unit, then their reduction into the gradient buffer
int launch_tc_encoder_dw(const Call& c, int64_t B, int xf64, cudaStream_t st) {
    const Plan& p = *c.p;
    const WsLayout& w = c.w;
    const BufTable& bt = c.bt;
    static std::atomic<bool> attr_set[64];
    if (first_on_device(attr_set)) {
        CUDA_TRY(cudaFuncSetAttribute(k_tc_encoder_dw<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, EDW_SMEM_BYTES));
        CUDA_TRY(cudaFuncSetAttribute(k_tc_encoder_dw<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, EDW_SMEM_BYTES));
    }
    // x rows by TMA (raw fp32 into the X operand area, converted in place) when every feature tensor allows it: fp32, 16-byte rows
    // (measured, same box: 0.258-0.270 ms against 0.246-0.251 ms for the register-staged loaders - here the loads of a step are issued
    // BEFORE its stage is free and nothing is pipelined across register sets, so the scoreboard effect of kernels_enc.cuh costs
    // little, while a landing zone inside the stage serialises copy -> conversion -> MMA per stage.  Off unless option "encoder_dw_tma" is 1.)
    bool xt = xf64 == 0 && w.M == 1 && g_encoder_dw_tma.load() > 0;
    for (const EncDwUnit& eu : p.enc_units)
        if (xt) xt = eu.x_buf >= BUF_X0 && eu.x_buf < BUF_X0 + p.n_types && enq_rows_ok(bt.p[eu.x_buf], eu.K, 0);
    EncXMaps xm;
    int rc;
    for (int t = 0; t < 4; ++t) {
        if (xt && t < p.n_types && p.in_w[t] % 4 == 0 && (reinterpret_cast<uintptr_t>(bt.p[BUF_X0 + t]) & 15) == 0) {
            if ((rc = make_map_x3d(&xm.x[t], bt.p[BUF_X0 + t], B, p.nodes[t], p.in_w[t], 64))) return rc;
        } else xm.x[t] = c.wm.dw;
    }
    float* pe_w = (float*)(c.ws + w.part_enc_w);
    float* pe_b = (float*)(c.ws + w.part_enc_b);
    {
        ProfScope ps(K_DW_ENC, st);
        dim3 grid((unsigned)p.enc_units.size(), (unsigned)(w.M * w.n_splits_enc));
        if (xt) k_tc_encoder_dw<true><<<grid, ENC_THREADS, EDW_SMEM_BYTES, st>>>(c.wm.dw, xm, (int)BUF_X0, p.d_enc_units, bt, c.br, B, w.Bp, w.rows_per_enc, w.n_splits_enc, xf64,
                                                                                 c.split, pe_w, pe_b, w.Bm);
        else k_tc_encoder_dw<false><<<grid, ENC_THREADS, EDW_SMEM_BYTES, st>>>(c.wm.dw, xm, (int)BUF_X0, p.d_enc_units, bt, c.br, B, w.Bp, w.rows_per_enc, w.n_splits_enc, xf64,
                                                                               c.split, pe_w, pe_b, w.Bm);
        LAUNCH_CHECK();
    }
    {
        ProfScope ps(K_REDUCE, st);
        dim3 grid((unsigned)p.enc_groups.size(), 48, (unsigned)w.M);
        k_reduce_enc<<<grid, 256, 0, st>>>(p.d_enc_groups, pe_w, pe_b, w.n_splits_enc, c.grads, 1.f / c.G, (int)p.enc_units.size(), p.n_params);
        LAUNCH_CHECK();
    }
    return 0;
}

// What the per-model optimizer entry points share: argument checks and the per-model table (lr, ranges, active flags).
int opt_models_table(const float* params, const float* grads, int32_t M, const int64_t* offsets, const float* lr, OptModels& t, int64_t* most) {
    if (!params || !grads || !offsets || !lr) return fail(MSHGNN_ERR_ARG, "NULL argument");
    if (M < 1 || M > OPT_MAX_MODELS) return fail(MSHGNN_ERR_ARG, "M must be in 1..%d (got %d)", OPT_MAX_MODELS, M);
    if (offsets[0] < 0) return fail(MSHGNN_ERR_ARG, "offsets[0] must be >= 0");
    memset(&t, 0, sizeof t);
    *most = 0;
    for (int m = 0; m <= M; ++m) {
        if (m > 0 && offsets[m] < offsets[m - 1]) return fail(MSHGNN_ERR_ARG, "offsets must not decrease (model %d)", m - 1);
        t.off[m] = offsets[m];
        if (m > 0) *most = std::max(*most, offsets[m] - offsets[m - 1]);
    }
    for (int m = 0; m < M; ++m) t.lr[m] = lr[m];
    return 0;
}

// grid of the per-model optimizer kernels: one row of CTAs per model, together about as many CTAs as k_adam's launch
dim3 opt_models_grid(int32_t M, int64_t most) {
    int64_t bx = std::min<int64_t>((most + 255) / 256, (148 * 8 + M - 1) / M);
    return dim3((unsigned)std::max<int64_t>(bx, 1), (unsigned)M);
}

}  // namespace

extern "C" {

int mshgnn_plan_create_ex(const mshgnn_desc* desc, int32_t flags, mshgnn_plan** plan_out) {
    if (!plan_out) return fail(MSHGNN_ERR_ARG, "plan_out is NULL");
    *plan_out = nullptr;
    mshgnn_plan* pl = new (std::nothrow) mshgnn_plan();
    if (!pl) return fail(MSHGNN_ERR_ARG, "out of host memory");
    std::string e = build_plan(desc, flags, pl->p);
    if (!e.empty()) { delete pl; return fail(MSHGNN_ERR_ARG, "%s", e.c_str()); }
    *plan_out = pl;
    return 0;
}

int mshgnn_plan_create(const mshgnn_desc* desc, mshgnn_plan** plan_out) { return mshgnn_plan_create_ex(desc, 0, plan_out); }

int mshgnn_plan_create_models(const mshgnn_desc* desc, int32_t M, const int32_t* hidden, mshgnn_plan** plan_out) {
    if (!plan_out) return fail(MSHGNN_ERR_ARG, "plan_out is NULL");
    *plan_out = nullptr;
    if (M < 1 || M > OPT_MAX_MODELS) return fail(MSHGNN_ERR_ARG, "M must be in 1..%d (got %d)", OPT_MAX_MODELS, M);
    if (!hidden) return fail(MSHGNN_ERR_ARG, "hidden is NULL");
    mshgnn_plan* pl = new (std::nothrow) mshgnn_plan();
    if (!pl) return fail(MSHGNN_ERR_ARG, "out of host memory");
    std::string e = build_plan(desc, 0, pl->p, std::vector<int>(hidden, hidden + M));
    if (!e.empty()) { delete pl; return fail(MSHGNN_ERR_ARG, "%s", e.c_str()); }
    *plan_out = pl;
    return 0;
}

void mshgnn_plan_destroy(mshgnn_plan* plan) {
    if (!plan) return;
    Plan& p = plan->p;
    for (void* d : p.d_allocs) cudaFree(d);
    delete plan;
}

int64_t mshgnn_param_count(const mshgnn_plan* plan) { return plan ? plan->p.ext_base.back() : -1; }

int mshgnn_param_offset(const mshgnn_plan* plan, int32_t kind, int32_t layer, int32_t idx, int64_t* off, int64_t* numel) {
    if (plan && plan->p.n_models > 1)
        return fail(MSHGNN_ERR_ARG, "the plan describes %d models: use mshgnn_param_offset_model", plan->p.n_models);
    return mshgnn_param_offset_model(plan, 0, kind, layer, idx, off, numel);
}

int mshgnn_param_offset_model(const mshgnn_plan* plan, int32_t m, int32_t kind, int32_t layer, int32_t idx, int64_t* off, int64_t* numel) {
    if (!plan || !off || !numel) return fail(MSHGNN_ERR_ARG, "NULL argument");
    const Plan& p = plan->p;
    if (m < 0 || m >= p.n_models) return fail(MSHGNN_ERR_ARG, "model %d out of range (the plan describes %d)", m, p.n_models);
    const ParamLayout& y = p.ext[m];      // the caller's layout of model m, at its width h, from the model's start
    const int64_t h = p.hidden[m];
    const int64_t base = p.ext_base[m];
    auto lay_ok = [&]() { return layer >= 0 && layer < p.L && idx >= 0 && idx < p.n_etypes; };
    switch (kind) {
        case MSHGNN_P_ENC_W: if (idx < 0 || idx >= p.n_types) break; *off = base + y.enc_w[idx]; *numel = h * p.in_w[idx]; return 0;
        case MSHGNN_P_ENC_B: if (idx < 0 || idx >= p.n_types) break; *off = base + y.enc_b[idx]; *numel = h; return 0;
        case MSHGNN_P_REL_W: if (!lay_ok()) break; *off = base + y.rel_w[layer * p.n_etypes + idx]; *numel = h * h; return 0;
        case MSHGNN_P_REL_B: if (!lay_ok()) break; *off = base + y.rel_b[layer * p.n_etypes + idx]; *numel = h; return 0;
        case MSHGNN_P_ROOT_W: if (!lay_ok()) break; *off = base + y.root_w[layer * p.n_etypes + idx]; *numel = h * h; return 0;
        case MSHGNN_P_MLP_W: if (!p.morph_sym || idx < 0 || idx > 1) break; *off = base + y.mlp_w[idx]; *numel = h * h; return 0;
        case MSHGNN_P_MLP_B: if (!p.morph_sym || idx < 0 || idx > 1) break; *off = base + y.mlp_b[idx]; *numel = h; return 0;
        case MSHGNN_P_DEC_W: *off = base + y.dec_w; *numel = p.C * h; return 0;
        case MSHGNN_P_DEC_B: *off = base + y.dec_b; *numel = p.C; return 0;
        default: break;
    }
    return fail(MSHGNN_ERR_ARG, "no such parameter (kind=%d layer=%d idx=%d)", kind, layer, idx);
}

int64_t mshgnn_workspace_bytes(const mshgnn_plan* plan, int64_t B, int32_t train, int32_t mode) {
    return mshgnn_workspace_bytes_models(plan, 1, B, train, mode);
}

int64_t mshgnn_workspace_bytes_models(const mshgnn_plan* plan, int64_t M, int64_t B, int32_t train, int32_t mode) {
    if (!plan || M < 1 || B < 1) return -1;
    if ((M > 1 || plan->p.n_models > 1) && (check_plan_mode(plan, mode) || check_models(plan->p, M, B, mode))) return -1;
    const WsLayout w = ws_layout(plan->p, B, train, mode, (int)M);
    if (train && mode != MSHGNN_MODE_FP32 && getenv("MSHGNN_DEBUG_LAYOUT")) {   // weight-gradient row splits per layer launch
        fprintf(stderr, "mshgnn layout M=%d B=%lld Bm=%lld: dW default %d x %d rows, %lld partial slots;", w.M, (long long)B, (long long)w.Bm,
                w.n_splits_tc, w.rows_per_tc, (long long)w.part_slots);
        for (size_t l = 0; l < plan->p.dw_layer.size(); ++l) fprintf(stderr, " L%zu[%d tasks]: %d x %d", l, plan->p.dw_layer[l].count, w.dw_ns[l], w.dw_rows[l]);
        fprintf(stderr, "; segments");
        for (int i = 0; i < w.segs.n; ++i) fprintf(stderr, " [tasks %d..%d) x %d @ slot %d", w.segs.begin[i], w.segs.begin[i + 1], w.segs.ns[i], w.segs.base[i]);
        fprintf(stderr, "\n");
    }
    return w.total;
}

int64_t mshgnn_dw_layout(const mshgnn_plan* plan, int64_t B, int32_t mode, int32_t* out, int64_t cap) {
    if (!plan || B < 1 || !out) return -1;
    const Plan& p = plan->p;
    const WsLayout w = ws_layout(p, B, 1, mode);
    const bool tc = mode != MSHGNN_MODE_FP32;
    for (int l = 0; l < p.L && 4 * (int64_t)l + 3 < cap; ++l) {
        out[4 * l] = p.dw_layer[l].count;
        out[4 * l + 1] = tc ? w.dw_ns[l] : w.n_splits;
        out[4 * l + 2] = tc ? w.dw_rows[l] : (int32_t)round_up((B + w.n_splits - 1) / w.n_splits, RG_BK);   // as k_reducegemm rounds it
        out[4 * l + 3] = w.dw_slot0[l];
    }
    return p.L;
}

int64_t mshgnn_out_rows(const mshgnn_plan* plan, int64_t B) { return plan ? B * plan->p.nodes[plan->p.dec_type] : -1; }

int64_t mshgnn_plan_describe(const mshgnn_plan* plan, char* buf, int64_t cap) {
    if (!plan) return -1;
    const std::string s = describe_plan(plan->p);
    if (buf && cap > 0) {
        const int64_t n = (int64_t)s.size() < cap - 1 ? (int64_t)s.size() : cap - 1;
        memcpy(buf, s.data(), n);
        buf[n] = 0;
    }
    return (int64_t)s.size() + 1;
}

int mshgnn_forward(const mshgnn_plan* plan, int64_t B, const void* const* x, int32_t x_dtype, const float* params,
                   float* out, void* workspace, int64_t workspace_bytes, int32_t train, int32_t mode, void* stream) {
    return mshgnn_forward_models(plan, 1, B, x, x_dtype, params, out, workspace, workspace_bytes, train, mode, stream);
}

int mshgnn_forward_models(const mshgnn_plan* plan, int64_t M, int64_t B, const void* const* x, int32_t x_dtype, const float* params,
                          float* out, void* workspace, int64_t workspace_bytes, int32_t train, int32_t mode, void* stream) {
    int rc;
    if ((rc = check_plan_mode(plan, mode))) return rc;
    const Plan& p = plan->p;
    if (x_dtype != MSHGNN_F32 && x_dtype != MSHGNN_F64 && x_dtype != MSHGNN_F16) return fail(MSHGNN_ERR_ARG, "x_dtype must be F32, F64 or F16");
    if (!x || !params || !out) return fail(MSHGNN_ERR_ARG, "NULL argument");
    Call c;
    if ((rc = open_call(c, plan, M, B, train, mode, workspace, workspace_bytes))) return rc;
    for (int t = 0; t < p.n_types; ++t)      // before the device is touched
        if (!x[t]) return fail(MSHGNN_ERR_ARG, "x[%d] is NULL", t);
    if ((rc = bind_call(c, params, nullptr, x))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const WsLayout& w = c.w;
    const BufTable& bt = c.bt;
    if (p.padded) {     // every kernel below reads the 128-wide zero-padded copy
        const PadGrid g = pad_grid(p, w.M);
        const int n_segs = (int)p.pad_segs.size();
        ProfScope ps(K_PAD, st);
        k_pad_params<<<dim3(PAD_BLOCKS_X, pad_grid_y(n_segs), g.z), 256, 0, st>>>(p.d_pad_segs, n_segs, params, (float*)c.params, g.ext_n, g.in_n);
        LAUNCH_CHECK();
    }
    params = c.params;
    const int xf64 = x_dtype == MSHGNN_F64 ? 1 : (x_dtype == MSHGNN_F16 ? 2 : 0);      // element-type code of the kernels (ld_x)

    if (!c.tc) {
        {   // derived weights (transposes, root sums, bias sums) from the current parameters
            ProfScope ps(K_DERIVE, st);
            const unsigned n_ops = (unsigned)p.derive_ops.size();
            if (n_ops > 0) {
                dim3 grid(16, n_ops);
                k_derive<<<grid, 256, 0, st>>>(p.d_derive, params, (float*)bt.p[BUF_DERIVED]);
                LAUNCH_CHECK();
            }
        }
        if ((rc = launch_rowgemm(K_ENC_FWD, p, train ? p.enc_train : p.enc_launch, bt, B, w.Bp, xf64, st))) return rc;
        for (int l = 0; l < p.L; ++l) {
            if ((rc = launch_rowgemm(K_CONV_FWD, p, train ? p.conv_train[l] : p.conv_infer[l], bt, B, w.Bp, 0, st))) return rc;
            if ((rc = launch_rowgemm(K_MLP_FWD, p, (train ? p.mlp1_train[l] : p.mlp1[l]), bt, B, w.Bp, 0, st))) return rc;
            if ((rc = launch_rowgemm(K_MLP_FWD, p, p.mlp2[l], bt, B, w.Bp, 0, st))) return rc;
        }
    } else {
        // tensor-core path: every activation lives as a (hi, lo) fp16 image pair only; TMA in, TMA out
        const BufRows& br = c.br;
        const WsMaps& wm = c.wm;
        __half* w_hi = (__half*)((char*)workspace + w.w16[0]);
        __half* w_lo = (__half*)((char*)workspace + w.w16[1]);
        const int split = c.split;
        {   // bias sums, (hi, lo) weight images, encoder weight image, stack counters: one launch (k_fwd_prologue)
            ProfScope ps(K_DERIVE, st);
            FwdPrologue fp;
            fp.ops = p.d_derive; fp.n_bias = p.n_derive_bias;
            fp.ops16 = p.d_derive16; fp.n16 = (int)p.derive16_ops.size();
            fp.ed.n_types = p.n_types;
            for (int t = 0; t < p.n_types; ++t) { fp.ed.w_off[t] = p.off_enc_w[t]; fp.ed.K[t] = p.in_w[t]; }
            fp.kmax = p.enc_kmax;
            fp.zero = w.stack ? (uint32_t*)((char*)workspace + w.stack_sync) : nullptr;
            fp.zero_words = w.stack ? w.stack_sync_bytes / 4 : 0;
            fp.zero_blocks = w.stack ? 16 : 0;
            fp.enc_sync = (uint32_t*)((char*)workspace + w.enc_sync);
            fp.n_params = p.n_params; fp.n_derived = p.n_derived;
            const unsigned blocks = (unsigned)(fp.n_bias + 8 * fp.n16 + 64 * p.n_types + fp.zero_blocks);
            k_fwd_prologue<<<dim3(blocks, (unsigned)w.M), 256, 0, st>>>(fp, params, (float*)bt.p[BUF_DERIVED], w_hi, w_lo, (__half*)((char*)workspace + w.wenc16[0]),
                                                    (__half*)((char*)workspace + w.wenc16[1]));
            LAUNCH_CHECK();
        }
        if ((rc = launch_tc_encoder(p, train ? p.enc_train : p.enc_launch, w, bt, br, wm, (char*)workspace, params, B, xf64, split, st))) return rc;
        if (w.stack) {
            // all layers (conv + chained base_transform) in one persistent launch over L2-resident row chunks
            if ((rc = launch_stack(K_STACK_FWD, p, train ? p.stack_train : p.stack_infer, w, bt, br, wm, (char*)workspace, B, split, st))) return rc;
        } else
        for (int l = 0; l < p.L; ++l) {
            if ((rc = launch_tc_rowgemm(K_CONV_FWD, p, train ? p.conv_train[l] : p.conv_infer[l], bt, br, wm, B, w.Bp, split, st))) return rc;
            if ((rc = launch_tc_rowgemm(K_MLP_FWD, p, train ? p.mlp1_train[l] : p.mlp1[l], bt, br, wm, B, w.Bp, split, st))) return rc;
            if ((rc = launch_tc_rowgemm(K_MLP_FWD, p, p.mlp2[l], bt, br, wm, B, w.Bp, split, st))) return rc;
        }
    }
    {
        const int64_t rows = B * p.dec.n_dec;
        int blocks = (int)((rows + 7) / 8);
        if (blocks > 148 * 8) blocks = 148 * 8;
        ProfScope ps(K_DEC_FWD, st);
#define MSHGNN_DEC_FWD(CM) k_decoder_fwd<CM><<<dim3(blocks, (unsigned)w.M), 256, 0, st>>>(p.dec, (const float*)bt.p[BUF_H0 + p.L], image16(c.ws, w, BUF_H0 + p.L, 0), \
                                              image16(c.ws, w, BUF_H0 + p.L, 1), params, p.d_signs, out, B, w.Bp, w.Bm, p.n_params)
        if (p.dec.C <= 2) MSHGNN_DEC_FWD(2); else if (p.dec.C <= 4) MSHGNN_DEC_FWD(4); else MSHGNN_DEC_FWD(8);
#undef MSHGNN_DEC_FWD
        LAUNCH_CHECK();
    }
    return 0;
}

int mshgnn_loss(const mshgnn_plan* plan, int64_t B, int32_t loss_kind, const float* out, const void* labels,
                int32_t label_dtype, float loss_scale, float* loss_out, float* dout, void* workspace,
                int64_t workspace_bytes, void* stream) {
    return mshgnn_loss_models(plan, 1, B, loss_kind, out, labels, label_dtype, loss_scale, loss_out, dout, workspace, workspace_bytes, stream);
}

int mshgnn_loss_models(const mshgnn_plan* plan, int64_t M, int64_t B, int32_t loss_kind, const float* out, const void* labels,
                       int32_t label_dtype, float loss_scale, float* loss_out, float* dout, void* workspace,
                       int64_t workspace_bytes, void* stream) {
    if (!plan) return fail(MSHGNN_ERR_ARG, "plan is NULL");
    const Plan& p = plan->p;
    if (!out || !labels || !loss_out || !workspace) return fail(MSHGNN_ERR_ARG, "NULL argument");
    if (B < 1) return fail(MSHGNN_ERR_ARG, "B must be >= 1");
    if (M < 1 || M > 65535) return fail(MSHGNN_ERR_ARG, "M must be in 1..65535 (got %lld)", (long long)M);
    if (p.n_models > 1 && M != p.n_models)
        return fail(MSHGNN_ERR_ARG, "the plan describes a model batch of %d models: M must be %d (got %lld)", p.n_models, p.n_models, (long long)M);
    if (label_dtype < 0 || label_dtype > 2) return fail(MSHGNN_ERR_ARG, "bad label_dtype");
    if (loss_kind == MSHGNN_LOSS_CE2 && p.C != 2) return fail(MSHGNN_ERR_ARG, "CE2 loss needs out_channels == 2");
    if (loss_kind != MSHGNN_LOSS_CE2 && loss_kind != MSHGNN_LOSS_MSE) return fail(MSHGNN_ERR_ARG, "bad loss_kind");
    if (workspace_bytes < M * LOSS_BLOCKS * 8) return fail(MSHGNN_ERR_WORKSPACE, "workspace too small for the loss partials");
    cudaStream_t st = (cudaStream_t)stream;
    // the loss partials (LOSS_BLOCKS per model) live in the last 256-aligned M*LOSS_BLOCKS*8 bytes of the workspace
    double* partial = (double*)((char*)workspace + ((workspace_bytes - M * LOSS_BLOCKS * 8) & ~(int64_t)255));
    const int64_t rows = B * p.dec.n_dec;
    const int64_t n = loss_kind == MSHGNN_LOSS_MSE ? rows * p.C : rows;
    int blocks = (int)((n + 255) / 256);
    if (blocks > LOSS_BLOCKS) blocks = LOSS_BLOCKS;
    ProfScope ps(K_LOSS, st);
    k_loss_partial<<<dim3(blocks, (unsigned)M), 256, 0, st>>>(loss_kind, out, labels, label_dtype, n, loss_scale / (float)n, dout, partial);
    LAUNCH_CHECK();
    k_loss_final<<<(unsigned)M, 32, 0, st>>>(partial, blocks, 1.0 / (double)n, loss_kind == MSHGNN_LOSS_CE2, loss_out);
    LAUNCH_CHECK();
    return 0;
}

int mshgnn_backward(const mshgnn_plan* plan, int64_t B, const void* const* x, int32_t x_dtype, const float* params,
                    const float* dout, float* grads, void* workspace, int64_t workspace_bytes, int32_t mode, void* stream) {
    return mshgnn_backward_staged(plan, B, x, x_dtype, params, dout, grads, workspace, workspace_bytes, mode, stream, nullptr);
}

int mshgnn_backward_staged(const mshgnn_plan* plan, int64_t B, const void* const* x, int32_t x_dtype, const float* params,
                           const float* dout, float* grads, void* workspace, int64_t workspace_bytes, int32_t mode, void* stream,
                           void* layers_ready_event) {
    return mshgnn_backward_models(plan, 1, B, x, x_dtype, params, dout, grads, workspace, workspace_bytes, mode, stream, layers_ready_event);
}

int mshgnn_backward_models(const mshgnn_plan* plan, int64_t M, int64_t B, const void* const* x, int32_t x_dtype, const float* params,
                           const float* dout, float* grads, void* workspace, int64_t workspace_bytes, int32_t mode, void* stream,
                           void* layers_ready_event) {
    int rc;
    if ((rc = check_plan_mode(plan, mode))) return rc;
    const Plan& p = plan->p;
    if (x_dtype != MSHGNN_F32 && x_dtype != MSHGNN_F64 && x_dtype != MSHGNN_F16) return fail(MSHGNN_ERR_ARG, "x_dtype must be F32, F64 or F16");
    if (!x || !params || !dout) return fail(MSHGNN_ERR_ARG, "NULL argument");
    const bool want_dw = grads != nullptr;      // NULL: input-only backward (the dX chain for mshgnn_input_grad, no weight gradient)
    Call c;
    if ((rc = open_call(c, plan, M, B, 1, mode, workspace, workspace_bytes))) return rc;
    if ((rc = bind_call(c, params, grads, x))) return rc;
    float* const grads_out = grads;             // padded plans: the caller's gradients, compacted from c.grads
    grads = c.grads;
    params = c.params;
    cudaStream_t st = (cudaStream_t)stream;
    const WsLayout& w = c.w;
    const BufTable& bt = c.bt;
    const BufRows& br = c.br;
    const WsMaps& wm = c.wm;
    char* ws = c.ws;
    const bool tc = c.tc;
    const int split = c.split;
    const float G = c.G;
    const int xf64 = x_dtype == MSHGNN_F64 ? 1 : (x_dtype == MSHGNN_F16 ? 2 : 0);      // element-type code of the kernels (ld_x)
    float* part_w = (float*)(ws + w.part_w);
    float* part_b = (float*)(ws + w.part_b);
    float* dec_part = (float*)(ws + w.dec_part);

    if (!want_dw) {
        if ((rc = stack_sync_reset(w, ws, st))) return rc;
    } else if (w.stack && (reinterpret_cast<uintptr_t>(grads) & 15) == 0) {
        ProfScope ps(K_MEMSET, st);
        const int64_t n_all = w.M * p.n_params, n4 = n_all / 4;
        k_bwd_prologue<<<296, 256, 0, st>>>((float4*)grads, n4, grads + n4 * 4, (int)(n_all - n4 * 4), (uint32_t*)(ws + w.stack_sync), w.stack_sync_bytes / 4);
        LAUNCH_CHECK();
    } else {
        { ProfScope ps(K_MEMSET, st); CUDA_TRY(cudaMemsetAsync(grads, 0, (size_t)w.M * p.n_params * 4, st)); }
        if ((rc = stack_sync_reset(w, ws, st))) return rc;
    }

    {   // decoder backward: dH_L on the decoded slots (+ masked copy = dc_{L-1}), dW_dec, db_dec
        const int L = p.L;
        const bool want_dh = p.morph_sym, want_dc = !p.morph_sym || p.dec_type != p.mlp_type;
        const int dhb = BUF_DHL0 + L, dcb = BUF_DCL0 + L - 1;
        // fp32 mode writes the slabs, the tensor-core modes the (hi, lo) images (the layout has only one of them)
        float* dh = want_dh ? (float*)bt.p[dhb] : nullptr;
        float* dc = want_dc ? (float*)bt.p[dcb] : nullptr;
        const int mk = want_dc ? MK_BITS : MK_NONE;
        const void* mbuf = want_dc ? bt.p[BUF_MASK0 + L - 1] : nullptr;
        ProfScope ps(K_DEC_BWD, st);
#define MSHGNN_DEC_BWD(CM) k_decoder_bwd<CM><<<dim3(DEC_BLOCKS, (unsigned)w.M), 256, 0, st>>>(p.dec, (const float*)bt.p[BUF_H0 + L], image16(ws, w, BUF_H0 + L, 0), \
                                                  image16(ws, w, BUF_H0 + L, 1), params, p.d_signs, dout, dh, dc, mk, mbuf, dec_part, B, w.Bp, G, \
                                                  want_dh ? image16(ws, w, dhb, 0) : nullptr, want_dh ? image16(ws, w, dhb, 1) : nullptr, \
                                                  want_dc ? image16(ws, w, dcb, 0) : nullptr, want_dc ? image16(ws, w, dcb, 1) : nullptr, w.Bm, p.n_params)
        if (p.dec.C <= 2) MSHGNN_DEC_BWD(2); else if (p.dec.C <= 4) MSHGNN_DEC_BWD(4); else MSHGNN_DEC_BWD(8);
#undef MSHGNN_DEC_BWD
        LAUNCH_CHECK();
        if (want_dw) {
            k_decoder_bwd_reduce<<<dim3(p.dec.C * H + p.dec.C, (unsigned)w.M), 256, 0, st>>>(p.dec, dec_part, DEC_BLOCKS, grads, 1.f / G, p.n_params);
            LAUNCH_CHECK();
        }
    }
    // layer-stack groups were produced with the split count of the kernel that ran them, encoder groups with the SIMT one
    const int ngl = p.n_groups_layers, nge = (int)p.groups.size() - ngl;
    auto reduce_layers = [&]() -> int {
        if (ngl > 0 && want_dw) {
            // 64 blocks per group = one element per thread: the groups of the shared base_transform weights sum up to 16 tasks x
            // 16..64 splits per element, and that serial chain (not the 117 MB of partials) sets the launch time.  (Four lanes per
            // element over the splits of a task, combined through shared memory, was measured: 2x SLOWER - the chain that matters is
            // the one over the TASKS of a group, one load round trip each.)
            dim3 grid((unsigned)ngl, 64, (unsigned)w.M);
            ProfScope ps(K_REDUCE, st);
            k_reduce_partials<<<grid, 256, 0, st>>>(p.d_groups, part_w, part_b, w.segs, grads, 1.f / G, w.part_slots, p.n_params);
            LAUNCH_CHECK();
        }
        return 0;
    };
    if (tc) {
        if (w.stack) {
            // the whole dX chain (with the base_transform backward chained on chip) in one launch over per-layer dh / dc / du
            // images, then the weight gradients of every layer (they only read what the chain and the forward pass stored)
            if ((rc = launch_stack(K_STACK_BWD, p, p.stack_bwd, w, bt, br, wm, ws, B, split, st))) return rc;
            if (want_dw) {
                // tasks are laid out layer L-1 first, contiguously: one launch covers them all (ws_layout fitted one split count)
                Launch all{p.dw_layer[p.L - 1].begin, 0};
                for (int l = 0; l < p.L; ++l) all.count += p.dw_layer[l].count;
                if ((rc = launch_tc_dw(K_DW_LAYER, p, p.L - 1, all, w, br, wm, B, split, part_w, part_b, st))) return rc;
            }
        } else {
            for (int l = p.L - 1; l >= 0; --l) {
                if ((rc = launch_tc_rowgemm(K_MLP_BWD, p, p.bwd_m1[l], bt, br, wm, B, w.Bp, split, st))) return rc;
                if ((rc = launch_tc_rowgemm(K_MLP_BWD, p, p.bwd_m2[l], bt, br, wm, B, w.Bp, split, st))) return rc;
                if (want_dw && (rc = launch_tc_dw(K_DW_LAYER, p, l, p.dw_layer[l], w, br, wm, B, split, part_w, part_b, st))) return rc;
                if ((rc = launch_tc_rowgemm(K_DX_BWD, p, p.bwd_dx[l], bt, br, wm, B, w.Bp, split, st))) return rc;
            }
        }
        // Every gradient outside the encoder is final here - before the encoder weight gradient, the last 8 % of the step, has
        // even started: the caller's event lets a data-parallel trainer all-reduce that 7.5 MB segment underneath it.
        if ((rc = reduce_layers())) return rc;
        if (p.padded && want_dw && (rc = compact_grads(p, w.M, p.n_pad_enc, (int)p.pad_segs.size() - p.n_pad_enc, grads, grads_out, st))) return rc;
        if (layers_ready_event) CUDA_TRY(cudaEventRecord((cudaEvent_t)layers_ready_event, st));
        if (!p.enc_units.empty() && want_dw && (rc = launch_tc_encoder_dw(c, B, xf64, st))) return rc;
        if (p.padded && want_dw && (rc = compact_grads(p, w.M, 0, p.n_pad_enc, grads, grads_out, st))) return rc;
    } else {
        auto launch_dw = [&](int kind, const Launch& L) -> int {
            if (L.count == 0 || !want_dw) return 0;
            ProfScope ps(kind, st);
            dim3 grid((unsigned)L.count, (unsigned)w.n_splits);
            k_reducegemm<<<grid, 256, 0, st>>>(p.d_rtasks, p.d_rpairs, L.begin, bt, B, w.Bp, xf64, w.n_splits, part_w, part_b);
            LAUNCH_CHECK();
            return 0;
        };
        for (int l = p.L - 1; l >= 0; --l) {
            if ((rc = launch_rowgemm(K_MLP_BWD, p, p.bwd_m1[l], bt, B, w.Bp, 0, st))) return rc;
            if ((rc = launch_rowgemm(K_MLP_BWD, p, p.bwd_m2[l], bt, B, w.Bp, 0, st))) return rc;
            if ((rc = launch_dw(K_DW_LAYER, p.dw_layer[l]))) return rc;
            if ((rc = launch_rowgemm(K_DX_BWD, p, p.bwd_dx[l], bt, B, w.Bp, 0, st))) return rc;
        }
        if ((rc = launch_dw(K_DW_ENC, p.dw_enc))) return rc;
        if ((rc = reduce_layers())) return rc;
        if (nge > 0 && want_dw) {
            dim3 grid((unsigned)nge, 32);
            ProfScope ps(K_REDUCE, st);
            k_reduce_partials<<<grid, 256, 0, st>>>(p.d_groups + ngl, part_w, part_b, w.segs, grads, 1.f / G, w.part_slots, p.n_params);
            LAUNCH_CHECK();
        }
        if (p.padded && want_dw && (rc = compact_grads(p, w.M, 0, (int)p.pad_segs.size(), grads, grads_out, st))) return rc;
        if (layers_ready_event) CUDA_TRY(cudaEventRecord((cudaEvent_t)layers_ready_event, st));
    }
    return 0;
}

int mshgnn_input_grad(const mshgnn_plan* plan, int64_t B, const float* params, float* const* dx, void* workspace, int64_t workspace_bytes,
                      int32_t mode, void* stream) {
    int rc;
    if ((rc = check_plan_mode(plan, mode))) return rc;
    const Plan& p = plan->p;
    if (!params || !dx) return fail(MSHGNN_ERR_ARG, "NULL argument");
    Call c;
    if ((rc = open_call(c, plan, 1, B, 1, mode, workspace, workspace_bytes))) return rc;
    DxOut o;
    memset(&o, 0, sizeof o);
    unsigned n_kb = 1;
    bool any = false;
    for (int t = 0; t < p.n_types; ++t) {
        if (dx[t] && (reinterpret_cast<uintptr_t>(dx[t]) & 3)) return fail(MSHGNN_ERR_ARG, "dx[%d] must be 4-byte aligned", t);
        o.p[t] = dx[t]; o.nodes[t] = p.nodes[t]; o.w_off[t] = p.off_enc_w[t];
        n_kb = std::max(n_kb, (unsigned)((p.in_w[t] + 63) / 64));
        any = any || dx[t];
    }
    if (!any) return 0;
    if ((rc = bind_call(c, params, nullptr, nullptr))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const WsLayout& w = c.w;
    const unsigned n_units = (unsigned)p.dx_units.size();
    if (!c.tc) {      // c.params: a padded plan's 128-wide copy (o.w_off is in that layout)
        ProfScope ps(K_DX_ENC, st);
        k_encoder_dx<<<dim3((unsigned)((B + 15) / 16), n_units, n_kb), 256, 0, st>>>(p.d_dx_units, o, (const float*)c.bt.p[BUF_DCL0 - 1], c.params, p.d_signs, B, w.Bp);
        LAUNCH_CHECK();
        return 0;
    }
    // tensor-core modes: dpre0 as (hi, lo) images, the encoder weight image of the forward prologue (x 2^8), G of the backward
    static std::atomic<bool> attr_set[64];
    if (first_on_device(attr_set)) CUDA_TRY(cudaFuncSetAttribute(k_tc_encoder_dx, cudaFuncAttributeMaxDynamicSharedMemorySize, DX_SMEM_BYTES));
    DxMaps maps;
    maps.a = c.wm.tc.o;
    if ((rc = make_map_2d(&maps.w_hi, c.ws + w.wenc16[0], (int64_t)p.n_types * H, p.enc_kmax, 64, 64, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    if ((rc = make_map_2d(&maps.w_lo, c.ws + w.wenc16[1], (int64_t)p.n_types * H, p.enc_kmax, 64, 64, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    for (int t = 0; t < 4; ++t) {
        maps.x[t] = c.wm.tc.o;
        if (t < p.n_types && dx[t] && enq_rows_ok(dx[t], p.in_w[t], -1)) {
            if ((rc = make_map_x3d(&maps.x[t], dx[t], B, p.nodes[t], p.in_w[t], 128, 32, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
            o.tma |= 1 << t;
        }
    }
    const float scale = TC_W_UNSCALE / c.G;      // 1 / (G 2^8)
    ProfScope ps(K_DX_ENC, st);
    k_tc_encoder_dx<<<dim3((unsigned)(w.Bp / TILE_M), n_units), DX_THREADS, DX_SMEM_BYTES, st>>>(maps, p.d_dx_units, o, p.d_signs, c.br.hi[BUF_DC1_ID],
                                                                                               c.br.lo[BUF_DC1_ID], B, w.Bp, c.split, scale);
    LAUNCH_CHECK();
    return 0;
}

int mshgnn_adam_step(float* params,const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, int64_t step,
                     float lr, float beta1, float beta2, float eps, float weight_decay, void* stream) {
    if (!params || !grads || !exp_avg || !exp_avg_sq || n < 1 || step < 1) return fail(MSHGNN_ERR_ARG, "bad argument");
    const float bc1 = 1.f - (float)std::pow((double)beta1, (double)step);
    const float bc2s = (float)std::sqrt(1.0 - std::pow((double)beta2, (double)step));
    int blocks = (int)((n + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    ProfScope ps(K_OPTIM, (cudaStream_t)stream);
    k_adam<<<blocks, 256, 0, (cudaStream_t)stream>>>(params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, bc1, bc2s);
    LAUNCH_CHECK();
    return 0;
}

int mshgnn_sgd_step(float* params, const float* grads, int64_t n, float lr, void* stream) {
    if (!params || !grads || n < 1) return fail(MSHGNN_ERR_ARG, "bad argument");
    int blocks = (int)((n + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    ProfScope ps(K_OPTIM, (cudaStream_t)stream);
    k_sgd<<<blocks, 256, 0, (cudaStream_t)stream>>>(params, grads, n, lr);
    LAUNCH_CHECK();
    return 0;
}

int mshgnn_adam_step_models(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int32_t M, const int64_t* offsets,
                            const int64_t* step, const float* lr, float beta1, float beta2, float eps, float weight_decay, void* stream) {
    OptModels t;
    int64_t most = 0;
    int rc;
    if ((rc = opt_models_table(params, grads, M, offsets, lr, t, &most))) return rc;
    if (!exp_avg || !exp_avg_sq || !step) return fail(MSHGNN_ERR_ARG, "NULL argument");
    for (int m = 0; m < M; ++m) {
        if (step[m] < 0) return fail(MSHGNN_ERR_ARG, "step[%d] must be >= 0 (got %lld)", m, (long long)step[m]);
        t.active[m] = step[m] > 0;
        if (!t.active[m]) continue;
        t.bc1[m] = 1.f - (float)std::pow((double)beta1, (double)step[m]);           // as mshgnn_adam_step
        t.bc2s[m] = (float)std::sqrt(1.0 - std::pow((double)beta2, (double)step[m]));
    }
    ProfScope ps(K_OPTIM, (cudaStream_t)stream);
    k_adam_models<<<opt_models_grid(M, most), 256, 0, (cudaStream_t)stream>>>(params, grads, exp_avg, exp_avg_sq, t, beta1, beta2, eps, weight_decay);
    LAUNCH_CHECK();
    return 0;
}

int mshgnn_sgd_step_models(float* params, const float* grads, int32_t M, const int64_t* offsets, const float* lr, const int32_t* active,
                           void* stream) {
    OptModels t;
    int64_t most = 0;
    int rc;
    if ((rc = opt_models_table(params, grads, M, offsets, lr, t, &most))) return rc;
    for (int m = 0; m < M; ++m) t.active[m] = !active || active[m] != 0;
    ProfScope ps(K_OPTIM, (cudaStream_t)stream);
    k_sgd_models<<<opt_models_grid(M, most), 256, 0, (cudaStream_t)stream>>>(params, grads, t);
    LAUNCH_CHECK();
    return 0;
}

int mshgnn_build_windows(const mshgnn_window_desc* d, const void* seq, const void* label_seq, int32_t seq_dtype, int64_t n_rows,
                         const int64_t* starts, int64_t B, float* const* x, float* y, void* stream) {
    if (!d || !seq || !starts || !x || B < 1) return fail(MSHGNN_ERR_ARG, "bad argument");
    if (seq_dtype != MSHGNN_F32 && seq_dtype != MSHGNN_F64) return fail(MSHGNN_ERR_ARG, "seq_dtype must be F32 or F64");
    const int T = d->history_length, C = d->seq_cols;
    if (T < 1 || (d->normalize && T < 2)) return fail(MSHGNN_ERR_ARG, "history_length %d unsupported (normalisation needs >= 2 rows)", T);
    if (C < 1 || C > WIN_MAX_COLS) return fail(MSHGNN_ERR_ARG, "seq_cols %d outside [1, %d]", C, WIN_MAX_COLS);
    if (n_rows < T) return fail(MSHGNN_ERR_ARG, "sequence has %lld rows, fewer than history_length %d", (long long)n_rows, T);
    if (d->n_node_types < 1 || d->n_node_types > 4) return fail(MSHGNN_ERR_ARG, "n_node_types out of range");
    if (d->n_labels < 0 || d->n_labels > WIN_MAX_LABELS) return fail(MSHGNN_ERR_ARG, "n_labels out of range");
    if (y && d->n_labels > 0 && (!label_seq || d->label_cols < 1 || !d->label_col)) return fail(MSHGNN_ERR_ARG, "labels requested without a label sequence");
    WindowTable tb;
    memset(&tb, 0, sizeof tb);
    tb.T = T; tb.C = C; tb.CL = d->label_cols; tb.n_types = d->n_node_types; tb.normalize = d->normalize != 0;
    tb.n_labels = y ? d->n_labels : 0;
    WindowPtrs out;
    memset(&out, 0, sizeof out);
    int nb = 0;
    for (int t = 0; t < d->n_node_types; ++t) {
        const int nodes = d->nodes_per_graph[t], blocks = d->blocks_per_node[t], len = d->block_len[t];
        if (nodes < 0 || blocks < 0 || (nodes * blocks > 0 && len != T && len != 1)) return fail(MSHGNN_ERR_ARG, "type %d: bad block shape", t);
        if (nodes * blocks > 0 && !x[t]) return fail(MSHGNN_ERR_ARG, "type %d: null output", t);
        tb.nodes[t] = nodes; tb.blocks[t] = blocks > 0 ? blocks : 1; tb.blen[t] = len; tb.first_block[t] = nb;
        out.x[t] = x[t];
        if (nb + nodes * blocks > WIN_MAX_BLOCKS) return fail(MSHGNN_ERR_ARG, "more than %d feature blocks per graph", WIN_MAX_BLOCKS);
        for (int i = 0; i < nodes * blocks; ++i) {
            const int c = d->block_col[nb + i], sg = d->block_sign ? d->block_sign[nb + i] : 1;
            if (c >= C) return fail(MSHGNN_ERR_ARG, "block %d reads column %d of a %d-column sequence", nb + i, c, C);
            if (c >= 0 && len != T) return fail(MSHGNN_ERR_ARG, "type %d: a constant-length block cannot read a column", t);
            if (sg < -127 || sg > 127) return fail(MSHGNN_ERR_ARG, "block factor out of range");
            tb.col[nb + i] = (int16_t)(c < 0 ? -1 : c); tb.sign[nb + i] = (int8_t)sg;
            if (c >= 0) tb.col_used[c] = 1;
        }
        nb += nodes * blocks;
    }
    tb.n_blocks = nb;
    for (int i = 0; i < tb.n_labels; ++i) {
        const int c = d->label_col[i];
        if (c < 0 || c >= d->label_cols) return fail(MSHGNN_ERR_ARG, "label column out of range");
        tb.label_col[i] = (int16_t)c; tb.label_sign[i] = (int8_t)(d->label_sign ? d->label_sign[i] : 1);
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int Tp = T | 1;
    const size_t esz = seq_dtype == MSHGNN_F64 ? 8 : 4;
    const int vw = (int)(16 / esz);
    const int Cp = (C + vw - 1) / vw * vw;
    if (Cp / vw > WIN_THREADS) return fail(MSHGNN_ERR_ARG, "seq_cols exceeds the CTA size");
    const int nrg = std::min(WIN_THREADS / (Cp / vw), WIN_MAX_RG);
    // z-scored window [C][T|1] floats, also the scratch of the statistics partials [row groups][Cp][2] doubles
    const size_t nz_bytes = (std::max((size_t)C * Tp * 4, (size_t)nrg * Cp * 16) + 127) / 128 * 128;
    const size_t smem = nz_bytes + (size_t)T * Cp * esz;
    if (smem > 200 * 1024) return fail(MSHGNN_ERR_ARG, "window of %d x %d does not fit in shared memory", T, C);
    // one bulk async copy per window needs 16-byte aligned window starts and sizes
    const int bulk = ((size_t)C * esz) % 16 == 0 && ((uintptr_t)seq % 16) == 0 && ((size_t)T * C * esz) < (1u << 20);
    int dev = 0, sms = 148;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (220 * 1024) / (smem + 1024)));
    const int grid = (int)std::min<int64_t>(B, (int64_t)sms * per_sm);
    ProfScope ps(K_WINDOWS, st);
    if (seq_dtype == MSHGNN_F64) {
        CUDA_TRY(cudaFuncSetAttribute(k_build_windows<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_build_windows<double><<<grid, WIN_THREADS, smem, st>>>(tb, (const double*)seq, (const double*)label_seq, n_rows, starts, B, out, y, bulk, (int)nz_bytes);
    } else {
        CUDA_TRY(cudaFuncSetAttribute(k_build_windows<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_build_windows<float><<<grid, WIN_THREADS, smem, st>>>(tb, (const float*)seq, (const float*)label_seq, n_rows, starts, B, out, y, bulk, (int)nz_bytes);
    }
    LAUNCH_CHECK();
    return 0;
}

int mshgnn_step_metrics(int32_t loss_kind, int64_t n, int32_t feet, const float* out, const void* labels, int32_t label_dtype,
                        double* batch, double* epoch, double* scratch, void* stream) {
    if (!out || !labels || !batch || !scratch || n < 1) return fail(MSHGNN_ERR_ARG, "bad argument");
    if (loss_kind != MSHGNN_LOSS_MSE && loss_kind != MSHGNN_LOSS_CE2) return fail(MSHGNN_ERR_ARG, "bad loss_kind");
    if (loss_kind == MSHGNN_LOSS_CE2 && (feet < 1 || feet > 4)) return fail(MSHGNN_ERR_ARG, "classification metrics need 1..4 rows per graph");
    if (label_dtype < 0 || label_dtype > 2) return fail(MSHGNN_ERR_ARG, "bad label_dtype");
    cudaStream_t st = (cudaStream_t)stream;
    int blocks = (int)((n + 255) / 256);
    if (blocks > MET_BLOCKS) blocks = MET_BLOCKS;
    ProfScope ps(K_METRICS, st);
    k_metrics_partial<<<blocks, 256, 0, st>>>(loss_kind, feet, out, labels, label_dtype, n, scratch);
    LAUNCH_CHECK();
    k_metrics_final<<<1, 32, 0, st>>>(loss_kind, scratch, blocks, batch, epoch);
    LAUNCH_CHECK();
    return 0;
}

int mshgnn_step_metrics_ex(int32_t kind, const mshgnn_metric_args* args, int64_t n, const float* out, const void* labels,
                           int32_t label_dtype, double* batch, double* epoch, double* scratch, void* stream) {
    if (!args || !out || !labels || !batch || !scratch || n < 1) return fail(MSHGNN_ERR_ARG, "bad argument");
    if (kind != MSHGNN_METRIC_COM && kind != MSHGNN_METRIC_GRF_WORLD) return fail(MSHGNN_ERR_ARG, "bad metric kind");
    if (label_dtype < 0 || label_dtype > 2) return fail(MSHGNN_ERR_ARG, "bad label_dtype");
    if (kind == MSHGNN_METRIC_COM) {
        if (args->n_base < 1 || args->n_base > 4) return fail(MSHGNN_ERR_ARG, "COM metrics need n_base in 1..4");
        if (!args->y_mean || !args->y_std) return fail(MSHGNN_ERR_ARG, "COM metrics need y_mean and y_std");
    } else {
        if (!args->quat) return fail(MSHGNN_ERR_ARG, "world-frame GRF metrics need the quaternions");
        if (args->quat_dtype != MSHGNN_F32 && args->quat_dtype != MSHGNN_F64) return fail(MSHGNN_ERR_ARG, "bad quat_dtype");
    }
    cudaStream_t st = (cudaStream_t)stream;
    int blocks = (int)((n + 255) / 256);
    if (blocks > MET_BLOCKS) blocks = MET_BLOCKS;
    ProfScope ps(K_METRICS, st);
    k_metrics_partial_ex<<<blocks, 256, 0, st>>>(kind, *args, out, labels, label_dtype, n, scratch);
    LAUNCH_CHECK();
    k_metrics_final<<<1, 32, 0, st>>>(kind, scratch, blocks, batch, epoch);
    LAUNCH_CHECK();
    return 0;
}

int mshgnn_profile_enable(int32_t on) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof_on = on != 0;
    return 0;
}

int mshgnn_profile_read(double* ms_out, int64_t* launches_out, int32_t n) {
    if (!ms_out || !launches_out || n < K_NKINDS_V1) return fail(MSHGNN_ERR_ARG, "bad argument");
    std::vector<ProfRec> recs;
    {
        std::lock_guard<std::mutex> lk(g_prof_mu);
        recs.swap(g_prof);
    }
    for (int i = 0; i < n; ++i) { ms_out[i] = 0.0; launches_out[i] = 0; }
    for (auto& r : recs) {
        CUDA_TRY(cudaEventSynchronize(r.b));
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, r.a, r.b));
        if (r.kind < n) { ms_out[r.kind] += ms; launches_out[r.kind] += 1; }
    }
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (auto& r : recs) { g_prof_pool.push_back(r.a); g_prof_pool.push_back(r.b); }
    return 0;
}

const char* mshgnn_kernel_kind_name(int32_t kind) {
    return (kind >= 0 && kind < MSHGNN_NUM_KERNEL_KINDS) ? kKindNames[kind] : "";
}

int mshgnn_relu_mask_offset(const mshgnn_plan* plan, int64_t B, int32_t mode, int32_t layer, int64_t* byte_off, int64_t* n_slots,
                            int64_t* rows_padded) {
    if (!plan || !byte_off || !n_slots || !rows_padded || B < 1) return fail(MSHGNN_ERR_ARG, "bad argument");
    const Plan& p = plan->p;
    if (layer < -1 || layer >= p.L) return fail(MSHGNN_ERR_ARG, "layer out of range");
    const WsLayout w = ws_layout(p, B, 1, mode);
    *byte_off = w.buf[layer < 0 ? BUF_MASKE : BUF_MASK0 + layer];
    *n_slots = layer < 0 ? p.S : p.S + p.nm;
    *rows_padded = w.Bp;
    return 0;
}

int mshgnn_check_edges(const mshgnn_plan* plan, int64_t B, const int64_t* const* edge_index, int32_t* flag, void* stream) {
    if (!plan || !edge_index || !flag || B < 1) return fail(MSHGNN_ERR_ARG, "bad argument");
    const Plan& p = plan->p;
    int rc;
    if ((rc = ensure_uploaded(p))) return rc;
    EdgeCheck ec;
    memset(&ec, 0, sizeof ec);
    ec.n_etypes = p.n_etypes;
    int off = 0;
    int64_t most = 0;
    for (int e = 0; e < p.n_etypes; ++e) {
        ec.E[e] = (int)p.e_src[e].size();
        ec.n_src[e] = p.nodes[p.e_src_t[e]]; ec.n_dst[e] = p.nodes[p.e_dst_t[e]];
        ec.tpl_off[e] = off; off += 2 * ec.E[e];
        if (ec.E[e] > 0 && !edge_index[e]) return fail(MSHGNN_ERR_ARG, "edge_index[%d] is NULL", e);
        ec.ei[e] = (const long long*)edge_index[e];
        most = std::max<int64_t>(most, (int64_t)ec.E[e] * B);
    }
    if (most == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned blocks = (unsigned)std::min<int64_t>((most + 1023) / 1024, 148 * 4);
    ProfScope ps(K_EDGES, st);
    k_check_edges<<<dim3(blocks, (unsigned)p.n_etypes), 256, 0, st>>>(ec, p.d_edge_tpl, (long long)B, flag);
    LAUNCH_CHECK();
    return 0;
}

int mshgnn_set_option(const char* name, int32_t value) {
    if (!name) return fail(MSHGNN_ERR_ARG, "option name is NULL");
    if (!strcmp(name, "stack")) { set_stack_enabled(value); return 0; }
    if (!strcmp(name, "stack_pair")) { set_stack_pair_mode(value); return 0; }
    if (!strcmp(name, "encoder")) { g_encoder_kernel.store(value < 0 || value > 2 ? -1 : value); return 0; }
    if (!strcmp(name, "encoder_tpi")) { g_encoder_tpi.store(value == 1 || value == 2 ? value : 0); return 0; }
    if (!strcmp(name, "encoder_dw_tma")) { g_encoder_dw_tma.store(value < 0 ? -1 : (value ? 1 : 0)); return 0; }
    return fail(MSHGNN_ERR_ARG, "unknown option '%s'", name);
}

int32_t mshgnn_get_option(const char* name) {
    if (name && !strcmp(name, "stack")) return stack_enabled() ? 1 : 0;
    if (name && !strcmp(name, "stack_pair")) return stack_pair_mode();
    if (name && !strcmp(name, "encoder")) return g_encoder_kernel.load();
    if (name && !strcmp(name, "encoder_tpi")) return g_encoder_tpi.load();
    if (name && !strcmp(name, "encoder_dw_tma")) return g_encoder_dw_tma.load();
    return -1;
}

int mshgnn_stack_status(const mshgnn_plan* plan, int64_t B, int32_t train, int32_t mode, const void* workspace, int32_t* status_out) {
    if (!plan || !workspace || !status_out || B < 1) return fail(MSHGNN_ERR_ARG, "bad argument");
    const WsLayout w = ws_layout(plan->p, B, train, mode);
    *status_out = 0;
    if (!w.stack) return 0;
    uint32_t word = 0;      // last word of the counter region: set by a stack launch whose dependency wait timed out
    CUDA_TRY(cudaMemcpy(&word, (const char*)workspace + w.stack_sync + w.stack_sync_bytes - 4, 4, cudaMemcpyDeviceToHost));
    *status_out = word ? 1 : 0;
    return 0;
}

int64_t mshgnn_launch_count(void) { return g_launches.load(); }
const char* mshgnn_last_error(void) { return g_err; }
const char* mshgnn_version(void) { return "mshgnn_b200 0.1 (sm_100a)"; }

}  // extern "C"
