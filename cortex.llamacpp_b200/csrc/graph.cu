// graph.cu -- op dispatch and graph execution behind b200_graph_compute().
//
// Replaces ggml_cuda_compute_forward (ggml-cuda.cu:2100-2332), ggml_backend_cuda_device_supports_op
// (:2959-3258) and the CUDA-graph capture/update logic of ggml_backend_cuda_graph_compute (:2432-2788).
// The caller (ggml-b200.cpp or a test) hands over a flat list of b200_op; we
//   1. optionally fuse adjacent ops (RMS_NORM+MUL, SILU+MUL) when the intermediate is not observable,
//   2. run them on the context's stream, or
//   3. when cuda_graphs is on and the very same op list (pointers, shapes, params) was seen before,
//      replay the captured cudaGraphExec instead of re-launching ~10 kernels per layer.
#include "common.cuh"
#include "gemv.h"
#include <string.h>
#include <algorithm>

// A decode step of llama.cpp differs from the previous one ONLY in where the new K/V rows are stored (the CPY destinations are
// views of the cache at kv_head, llama-graph.cpp:1375-1397).  The reference patches those kernel parameters into its captured
// graph every token (maintain_cuda_graph, ggml-cuda.cu:2544-2587); here the cache key ignores them and the captured rope+store
// kernels read their destinations from a small device table that is refreshed with one 16 B/layer copy before each replay.
struct GraphCacheEntry {
    std::vector<b200_op> key;                       // op list with the KV-store destinations zeroed
    std::vector<int> kv_idx;                        // op indices of the KV-store candidates (CPY f32 -> 1-D cache view)
    std::vector<void *> kv_ptrs;                    // their destinations at first sighting (exact-match fallback)
    bool indirect = false;                          // every candidate is absorbed by a fused rope+store node: table indirection
    std::vector<std::pair<int, int>> node_kv;       // per rope+store node: op indices of its K and V store
    void **dev_table = nullptr;                     // [2 * nodes] device pointers
    cudaGraphExec_t exec = nullptr;
    int hits = 0;
};
struct GraphCache {
    std::vector<GraphCacheEntry> entries;
    std::vector<b200_op> scratch_key;               // reused per call
    std::vector<int> scratch_idx;
};

void graph_cache_free(b200_ctx *ctx) {
    if (!ctx->graph_cache) return;
    for (auto &e : ctx->graph_cache->entries) { if (e.exec) cudaGraphExecDestroy(e.exec); if (e.dev_table) cudaFree(e.dev_table); }
    delete ctx->graph_cache;
    ctx->graph_cache = nullptr;
}

static int dispatch(b200_ctx *ctx, const b200_op *op) {
    if (ctx->fa_map_valid && op->dst.data) {       // an op that writes into the attention mask drops its live-tile map (fattn.cu)
        const uintptr_t lo = (uintptr_t)op->dst.data;
        if (lo < ctx->fa_map_mask_end && lo + (size_t)op->dst.nb[3] * (size_t)(op->dst.ne[3] > 0 ? op->dst.ne[3] : 1) > ctx->fa_map_mask) ctx->fa_map_valid = false;
    }
    switch (op->op) {
        case B200_OP_NONE: return B200_OK;
        case B200_OP_MUL_MAT: return op_mul_mat(ctx, op);
        case B200_OP_MUL_MAT_ID: return op_mul_mat_id(ctx, op);
        case B200_OP_FLASH_ATTN_EXT: return op_flash_attn_ext(ctx, op);
        case B200_OP_ALLREDUCE: return op_allreduce(ctx, op);
        default: return op_glue(ctx, op);
    }
}

extern "C" int b200_supports_op(int device, const b200_op *op) {
    (void)device;
    if (!op) return 0;
    // a row-split tensor's `data` is the host-side b200_split: only op_mul_mat_split reads it, as the weight of a MUL_MAT
    for (int i = 0; i < op->n_src && i < B200_MAX_SRC; i++)
        if ((op->src[i].flags & B200_TENSOR_FLAG_SPLIT) && (op->op != B200_OP_MUL_MAT || i != 0)) return 0;
    if (op->dst.flags & B200_TENSOR_FLAG_SPLIT) return 0;
    switch (op->op) {
        case B200_OP_NONE: return 1;
        case B200_OP_MUL_MAT: return supports_mul_mat(op) ? 1 : 0;
        case B200_OP_MUL_MAT_ID: return supports_mul_mat_id(op) ? 1 : 0;
        case B200_OP_FLASH_ATTN_EXT: return supports_flash_attn_ext(op) ? 1 : 0;
        case B200_OP_ALLREDUCE: return supports_allreduce(op) ? 1 : 0;
        default: return supports_glue(op) ? 1 : 0;
    }
}

extern "C" int b200_op_compute(b200_ctx *ctx, const b200_op *op) {
    if (!ctx || !op) return B200_ERR_FAILED;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (!b200_supports_op(ctx->device, op)) { b200_set_error("op %d not supported for these operands", op->op); return B200_ERR_UNSUPPORTED; }
    ctx->fa_map_valid = false;
    return dispatch(ctx, op);
}

// ---------------------------------------------------------------------------------------------- fusion
// graph_compute turns the op list into an EXEC list.  Besides plain ops it knows three fused launches, all of them only
// for decode-sized ubatches (<= 4 tokens), where kernel boundaries -- not bytes -- dominate (SURVEY.md 8f rank 1):
//   EX_GEMV        one streaming GEMV over 1-3 weight matrices with the producer ops folded into its prologue
//                  (rms_norm*weight or silu(gate)*up, activation quantisation) and the residual ADD into its epilogue
//   EX_ROPE_STORE  ROPE(q) + ROPE(k) + KV-store of k and v
// A llama layer becomes: [norm+QKV] [rope+store] [flash_attn (+combine)] [wo+residual] [norm+gate|up] [swiglu+down+residual].
// Intermediates that only lived between the fused ops are never materialised; the matcher proves with a liveness scan
// over the op list (address ranges, first access after the pattern) that nobody else reads them.
enum { EX_OP = 0, EX_GEMV = 1, EX_ROPE_STORE = 2 };
static const int g_fuse_debug = getenv("GGML_B200_FUSE_DEBUG") ? atoi(getenv("GGML_B200_FUSE_DEBUG")) : 0;
struct ExecNode {
    int kind = EX_OP;
    b200_op op;                                  // EX_OP
    GemvSegDesc seg[GEMV_MAX_SEG]; int nseg = 0; // EX_GEMV
    int64_t K = 0; GemvActDesc act; int ncols = 0; bool w_const = false;
    GemvPf pf[GEMV_MAX_PF] = {}; int npf = 0;    // L2 look-ahead ranges (weights of the launches that follow)
    int pair = 0;                                // FFN: 1 = gate|up launch (may write silu(gate)*up itself), 2 = the down launch that follows it
    RopeStoreDesc rs;                            // EX_ROPE_STORE
    int kv_slot = -1;                            // index of this node's K destination in the KV pointer table (V = +1)
};

static bool same_tensor(const b200_tensor &a, const b200_tensor &b) {
    return a.data == b.data && a.type == b.type && !memcmp(a.ne, b.ne, sizeof(a.ne)) && !memcmp(a.nb, b.nb, sizeof(a.nb));
}
static void tensor_range(const b200_tensor &t, uintptr_t &lo, uintptr_t &hi) {
    lo = (uintptr_t)t.data;
    uint64_t span = (uint64_t)b200_type_block_bytes(t.type);
    const int be = b200_type_block_elems(t.type);
    span += (uint64_t)(t.ne[0] / be - 1) * t.nb[0];
    for (int i = 1; i < 4; i++) if (t.ne[i] > 1) span += (uint64_t)(t.ne[i] - 1) * t.nb[i];
    hi = lo + span;
}
static bool overlaps(const b200_tensor &a, const b200_tensor &b) {
    if (!a.data || !b.data) return false;
    uintptr_t al, ah, bl, bh;
    tensor_range(a, al, ah); tensor_range(b, bl, bh);
    return al < bh && bl < ah;
}
// does tensor a span every byte of tensor t?  (a write of a dense a then replaces t's whole value; a mere overlap leaves some of it)
static bool covers(const b200_tensor &a, const b200_tensor &t) {
    if (!a.data || !t.data) return false;
    uintptr_t al, ah, tl, th;
    tensor_range(a, al, ah); tensor_range(t, tl, th);
    return al <= tl && th <= ah;
}
// is the VALUE currently held by tensor t still needed by ops[from..n)?  (first touch of its bytes: a read => yes, a write => no)
static bool live_after(const b200_op *ops, int n, int from, const b200_tensor &t) {
    for (int i = from; i < n; i++) {
        for (int s = 0; s < ops[i].n_src && s < B200_MAX_SRC; s++) if (overlaps(ops[i].src[s], t)) return true;
        if (overlaps(ops[i].dst, t)) return false;
    }
    return false;
}

constexpr int FUSE_MAX_T = 32;        // layer fusions cover batch-1 decode (<= 4 columns: GEMV) and continuous-batching steps (<= 32: gemv_mma)
static bool is_vec_f32(const b200_tensor &t, int64_t rows) {   // dense f32 [rows, T<=32]
    return t.type == B200_TYPE_F32 && t.ne[0] == rows && t.ne[1] >= 1 && t.ne[1] <= FUSE_MAX_T && t.ne[2] == 1 && t.ne[3] == 1 && t.nb[0] == 4 &&
           t.nb[1] == (uint64_t)rows * 4 && !((uintptr_t)t.data & 15);
}
// a decode-sized quantised matmul the GEMV can take as a segment: W quant rows back to back, x dense [K, T], dst dense [N, T]
static bool is_decode_mm(const b200_op &o) {
    if (o.op != B200_OP_MUL_MAT || (o.src[0].flags & B200_TENSOR_FLAG_SPLIT) || !supports_mul_mat(&o)) return false;
    const b200_tensor &w = o.src[0], &x = o.src[1], &d = o.dst;
    if (!b200_type_is_quant(w.type) || w.ne[2] != 1 || w.ne[3] != 1) return false;
    return is_vec_f32(x, w.ne[0]) && is_vec_f32(d, w.ne[1]) && x.ne[1] == d.ne[1];
}
static GemvSegDesc seg_of(const b200_op &mm, float *dst, size_t dst_stride, const float *residual) {
    GemvSegDesc g = {};
    g.type = mm.src[0].type; g.W = (const uint8_t *)mm.src[0].data; g.rb = b200_row_bytes(g.type, mm.src[0].ne[0]); g.N = mm.src[0].ne[1];
    g.dst = dst; g.dst_stride = dst_stride; g.residual = residual;
    return g;
}
static bool all_weights(const b200_op *const *mms, int n) {
    for (int i = 0; i < n; i++) if (!(mms[i]->src[0].flags & B200_TENSOR_FLAG_WEIGHT)) return false;
    return true;
}

// RMS_NORM(x) -> MUL(norm, w): returns true and the norm weight when ops[i], ops[i+1] form that pair over a dense [E, T<=4] x
static bool match_norm_mul(const b200_op *ops, int n, int i, const b200_tensor *&xin, const float *&w, float &eps) {
    if (i + 1 >= n || ops[i].op != B200_OP_RMS_NORM || ops[i + 1].op != B200_OP_MUL) return false;
    const b200_op &a = ops[i], &b = ops[i + 1];
    if (!is_vec_f32(a.src[0], a.src[0].ne[0]) || !same_tensor(b.src[0], a.dst) || !is_vec_f32(b.dst, a.src[0].ne[0])) return false;
    const b200_tensor &nw = b.src[1];
    if (nw.type != B200_TYPE_F32 || nw.nb[0] != 4 || nw.ne[0] != a.src[0].ne[0] || nw.ne[1] != 1 || nw.ne[2] != 1 || nw.ne[3] != 1 || ((uintptr_t)nw.data & 15)) return false;
    xin = &a.src[0]; w = (const float *)nw.data;
    memcpy(&eps, &a.params[0], 4);
    return true;
}

struct FuseScratch { float *q, *k, *v, *g, *u; };

// attention block: NORM MUL {MMq MMk MMv ROPEq ROPEk CPYk CPYv in any dependency-respecting order} FA
#define MA_FAIL(code) do { if (g_fuse_debug) fprintf(stderr, "[b200 fuse] attention pattern at op %d rejected: check %d\n", i, code); return 0; } while (0)
static int match_attention(b200_ctx *ctx, const b200_op *ops, int n, int i, const FuseScratch &fs, std::vector<ExecNode> &out) {
    const b200_tensor *xin; const float *nw; float eps;
    if (i + 9 >= n || !match_norm_mul(ops, n, i, xin, nw, eps)) MA_FAIL(1);
    // the FLASH_ATTN_EXT that closes the block: 7 ops after NORM MUL, plus (first layer of a llama.cpp graph) the f32 -> f16
    // conversion of the KQ mask, which llama.cpp schedules right before its first consumer
    int fa_idx = -1;
    for (int j = i + 9; j < n && j <= i + 11; j++) if (ops[j].op == B200_OP_FLASH_ATTN_EXT) { fa_idx = j; break; }
    if (fa_idx < 0) MA_FAIL(2);
    const b200_op &fa = ops[fa_idx];
    const b200_op *mm[3], *rope[2], *cpy[2], *extra[2];
    int nmm = 0, nrope = 0, ncpy = 0, nextra = 0;
    for (int j = i + 2; j < fa_idx; j++) {
        const b200_op &o = ops[j];
        if (o.op == B200_OP_MUL_MAT && nmm < 3) mm[nmm++] = &o;
        else if (o.op == B200_OP_ROPE && nrope < 2) rope[nrope++] = &o;
        else if (o.op == B200_OP_CPY && fa.n_src > 3 && o.dst.data == fa.src[3].data && nextra < 2) extra[nextra++] = &o;     // mask conversion
        else if (o.op == B200_OP_CPY && ncpy < 2) cpy[ncpy++] = &o;
        else MA_FAIL(3);
    }
    if (nmm != 3 || nrope != 2 || ncpy != 2) MA_FAIL(4);
    const b200_tensor &B = ops[i + 1].dst;
    for (int j = 0; j < 3; j++) if (!is_decode_mm(*mm[j]) || !same_tensor(mm[j]->src[1], B)) MA_FAIL(5);
    if (!all_weights(mm, 3)) MA_FAIL(6);
    for (int x = 0; x < nextra; x++) if (overlaps(extra[x]->src[0], ops[i].dst) || overlaps(extra[x]->src[0], B)) MA_FAIL(17);
    // roles: q = the matmul whose rope feeds FA; k = the matmul whose rope feeds a CPY; v = the matmul feeding a CPY directly.
    // ggml-alloc hands the SAME buffer to the three matmul outputs one after the other (each dies at its rope / store), so a
    // consumer is paired with the LATEST matmul before it that wrote its source address, not with "the" matmul at that address
    const b200_op *mq = nullptr, *mk = nullptr, *mv = nullptr, *rq = nullptr, *rk = nullptr, *ck = nullptr, *cv = nullptr;
    for (int r = 0; r < 2; r++) {
        if (rope[r]->dst.data == fa.src[0].data) rq = rope[r];
        else for (int c = 0; c < 2; c++) if (cpy[c]->src[0].data == rope[r]->dst.data && cpy[c] > rope[r]) { rk = rope[r]; ck = cpy[c]; }
    }
    if (!rq || !rk || rq == rk) MA_FAIL(7);
    cv = ck == cpy[0] ? cpy[1] : cpy[0];
    auto producer = [&](const b200_op *consumer) -> const b200_op * {
        const b200_op *best = nullptr;
        for (int j = 0; j < 3; j++) if (mm[j] < consumer && mm[j]->dst.data == consumer->src[0].data && (!best || mm[j] > best)) best = mm[j];
        return best;
    };
    mq = producer(rq); mk = producer(rk); mv = producer(cv);
    if (!mq || !mk || !mv || mq == mk || mq == mv || mk == mv) MA_FAIL(8);
    // a matmul output that shares its buffer with a later one must be consumed before that one is produced
    const b200_op *cons[3] = {rq, rk, cv}, *prod[3] = {mq, mk, mv};
    for (int a_ = 0; a_ < 3; a_++) for (int b_ = 0; b_ < 3; b_++)
        if (a_ != b_ && prod[a_]->dst.data == prod[b_]->dst.data && prod[a_] < prod[b_] && cons[a_] > prod[b_]) MA_FAIL(18);
    // shapes: rope over [D, heads, T] f32 dense views of the matmul outputs, identical rope parameters and positions
    const int64_t T = B.ne[1], D = rq->src[0].ne[0], H = rq->src[0].ne[1], Hkv = rk->src[0].ne[1];
    auto rope_ok = [&](const b200_op *r, int64_t heads) {
        const b200_tensor &a = r->src[0];
        return a.type == B200_TYPE_F32 && r->dst.type == B200_TYPE_F32 && a.ne[0] == D && a.ne[1] == heads && a.ne[2] == T && a.ne[3] == 1 &&
               a.nb[0] == 4 && a.nb[1] == (uint64_t)D * 4 && a.nb[2] == (uint64_t)D * heads * 4 && r->src[1].type == B200_TYPE_I32 &&
               r->src[1].ne[0] == T && supports_glue(r);
    };
    if (D > 512 || D % 32 || !rope_ok(rq, H) || !rope_ok(rk, Hkv)) MA_FAIL(9);
    if (memcmp(rq->params, rk->params, sizeof(rq->params)) || rq->src[1].data != rk->src[1].data || rq->src[2].data != rk->src[2].data) MA_FAIL(10);
    if (mq->src[0].ne[1] != H * D || mk->src[0].ne[1] != Hkv * D || mv->src[0].ne[1] != Hkv * D) MA_FAIL(11);
    const b200_tensor &qd = rq->dst;
    if (qd.nb[0] != 4 || qd.ne[0] != D || qd.ne[1] != H || qd.ne[2] != T) MA_FAIL(12);
    // KV store destinations: contiguous runs of T rows of Hkv*D elements in the cache type
    const int kvt = ck->dst.type;
    if (kvt != cv->dst.type || (kvt != B200_TYPE_F16 && kvt != B200_TYPE_Q8_0 && kvt != B200_TYPE_Q4_0)) MA_FAIL(13);
    if (!tensor_is_contiguous(ck->dst) || !tensor_is_contiguous(cv->dst) || tensor_nelements(ck->dst) != Hkv * D * T ||
        tensor_nelements(cv->dst) != Hkv * D * T) MA_FAIL(14);
    if (ck->src[0].type != B200_TYPE_F32 || cv->src[0].type != B200_TYPE_F32 || !tensor_is_contiguous(ck->src[0]) || !tensor_is_contiguous(cv->src[0])) MA_FAIL(15);
    // nobody else may need the intermediates we never write
    const b200_tensor *dead[] = {&ops[i].dst, &B, &mq->dst, &mk->dst, &mv->dst, &rk->dst};
    // (memory of a dead intermediate that ggml-alloc re-used for the mask conversion inside the block is read later as the MASK,
    //  which we do write: not a use of the intermediate)
    for (const b200_tensor *t : dead) if (live_after(ops, n, fa_idx, *t)) {
        bool reused = false;
        for (int x = 0; x < nextra; x++) reused |= covers(extra[x]->dst, *t);
        if (!reused) MA_FAIL(16);
    }
    (void)ctx;
    for (int x = 0; x < nextra; x++) { ExecNode m; m.kind = EX_OP; m.op = *extra[x]; out.push_back(m); }
    ExecNode g;
    g.kind = EX_GEMV; g.nseg = 3; g.K = xin->ne[0]; g.ncols = (int)T; g.w_const = true;
    g.seg[0] = seg_of(*mq, fs.q, (size_t)(H * D), nullptr);
    g.seg[1] = seg_of(*mk, fs.k, (size_t)(Hkv * D), nullptr);
    g.seg[2] = seg_of(*mv, fs.v, (size_t)(Hkv * D), nullptr);
    g.act = GemvActDesc{};
    g.act.mode = ACT_F32_NORM; g.act.x = (const float *)xin->data; g.act.x_stride = xin->nb[1]; g.act.x2 = nw; g.act.eps = eps;
    if (b200_act_mode_q8k(g.seg[0].type) != b200_act_mode_q8k(g.seg[1].type) || b200_act_mode_q8k(g.seg[0].type) != b200_act_mode_q8k(g.seg[2].type)) return 0;
    out.push_back(g);
    ExecNode r;
    r.kind = EX_ROPE_STORE;
    RopeStoreDesc &d = r.rs;
    memset(&d, 0, sizeof(d));
    d.q = fs.q; d.k = fs.k; d.v = fs.v;
    d.pos = (const int32_t *)rq->src[1].data;
    d.freq_factors = rq->n_src > 2 ? (const float *)rq->src[2].data : nullptr;
    d.q_out = (float *)qd.data; d.q_out_nb1 = qd.nb[1]; d.q_out_nb2 = qd.nb[2];
    d.k_dst = ck->dst.data; d.v_dst = cv->dst.data;
    d.D = (int)D; d.H = (int)H; d.Hkv = (int)Hkv; d.T = (int)T; d.kv_type = kvt;
    memcpy(d.rope_params, rq->params, sizeof(d.rope_params));
    out.push_back(r);
    ExecNode f;
    f.kind = EX_OP; f.op = fa;
    out.push_back(f);
    return fa_idx - i + 1;
}

// FFN block: NORM MUL {MMgate SILU MMup MUL MMdown} ADD
static int match_ffn(const b200_op *ops, int n, int i, const FuseScratch &fs, std::vector<ExecNode> &out) {
    const b200_tensor *xin; const float *nw; float eps;
    if (i + 7 >= n || !match_norm_mul(ops, n, i, xin, nw, eps)) return 0;
    const b200_op &add = ops[i + 7];
    const bool tp = add.op == B200_OP_ALLREDUCE;       // tensor parallel: down's partial sums go to the all-reduce (which adds the residual)
    if (add.op != B200_OP_ADD && !tp) return 0;
    const b200_op *mm[3], *silu = nullptr, *mul = nullptr;
    int nmm = 0;
    for (int j = i + 2; j < i + 7; j++) {
        const b200_op &o = ops[j];
        if (o.op == B200_OP_MUL_MAT && nmm < 3) mm[nmm++] = &o;
        else if (o.op == B200_OP_SILU && !silu) silu = &o;
        else if (o.op == B200_OP_MUL && !mul) mul = &o;
        else return 0;
    }
    if (nmm != 3 || !silu || !mul) return 0;
    const b200_tensor &B = ops[i + 1].dst;
    const b200_op *gate = nullptr, *up = nullptr, *down = nullptr;
    for (int j = 0; j < 3; j++) {
        if (!is_decode_mm(*mm[j])) return 0;
        if (same_tensor(mm[j]->src[1], B)) { if (mm[j]->dst.data == silu->src[0].data) gate = mm[j]; else up = mm[j]; }
        else down = mm[j];
    }
    if (!gate || !up || !down || !all_weights(mm, 3)) return 0;
    if (!((mul->src[0].data == silu->dst.data && mul->src[1].data == up->dst.data) || (mul->src[1].data == silu->dst.data && mul->src[0].data == up->dst.data))) return 0;
    if (!same_tensor(down->src[1], mul->dst)) return 0;
    const int64_t T = B.ne[1], FF = gate->src[0].ne[1], E = down->src[0].ne[1];
    if (b200_act_mode_q8k(gate->src[0].type) != b200_act_mode_q8k(up->src[0].type)) return 0;
    const b200_tensor *resid = nullptr;
    if (tp) {
        if (add.src[0].data != down->dst.data || !is_vec_f32(down->dst, E) || up->src[0].ne[1] != FF || down->src[0].ne[0] != FF) return 0;
        const b200_tensor *dead[] = {&ops[i].dst, &B, &gate->dst, &silu->dst, &up->dst, &mul->dst};
        for (const b200_tensor *t : dead) if (!covers(down->dst, *t) && live_after(ops, n, i + 7, *t)) return 0;
    } else {
        resid = add.src[0].data == down->dst.data ? &add.src[1] : (add.src[1].data == down->dst.data ? &add.src[0] : nullptr);
        if (!resid) return 0;
        if (up->src[0].ne[1] != FF || down->src[0].ne[0] != FF || !is_vec_f32(*resid, E) || !is_vec_f32(add.dst, E) || resid->ne[1] != T || add.dst.ne[1] != T) return 0;
        const b200_tensor *dead[] = {&ops[i].dst, &B, &gate->dst, &silu->dst, &up->dst, &mul->dst, &down->dst};
        for (const b200_tensor *t : dead) if (!covers(add.dst, *t) && live_after(ops, n, i + 8, *t)) return 0;
    }
    ExecNode g;
    g.kind = EX_GEMV; g.nseg = 2; g.K = xin->ne[0]; g.ncols = (int)T; g.w_const = true;
    g.seg[0] = seg_of(*gate, fs.g, (size_t)FF, nullptr);
    g.seg[1] = seg_of(*up, fs.u, (size_t)FF, nullptr);
    g.act = GemvActDesc{};
    g.act.mode = ACT_F32_NORM; g.act.x = (const float *)xin->data; g.act.x_stride = xin->nb[1]; g.act.x2 = nw; g.act.eps = eps;
    g.pair = 1;
    out.push_back(g);
    ExecNode d;
    d.pair = 2;
    d.kind = EX_GEMV; d.nseg = 1; d.K = FF; d.ncols = (int)T; d.w_const = true;
    d.seg[0] = tp ? seg_of(*down, (float *)down->dst.data, (size_t)E, nullptr) : seg_of(*down, (float *)add.dst.data, (size_t)E, (const float *)resid->data);
    d.act = GemvActDesc{};
    d.act.mode = ACT_F32_SWIGLU; d.act.x = fs.g; d.act.x_stride = (size_t)FF * 4; d.act.x2 = fs.u;
    out.push_back(d);
    return tp ? 7 : 8;
}

// MUL_MAT -> ADD(mm, residual)
static int match_mm_add(const b200_op *ops, int n, int i, std::vector<ExecNode> &out) {
    if (i + 1 >= n || !is_decode_mm(ops[i]) || ops[i + 1].op != B200_OP_ADD) return 0;
    const b200_op &mm = ops[i], &add = ops[i + 1];
    if (!(mm.src[0].flags & B200_TENSOR_FLAG_WEIGHT)) return 0;
    const b200_tensor *resid = add.src[0].data == mm.dst.data ? &add.src[1] : (add.src[1].data == mm.dst.data ? &add.src[0] : nullptr);
    const int64_t N = mm.src[0].ne[1], T = mm.dst.ne[1];
    if (!resid || !is_vec_f32(*resid, N) || !is_vec_f32(add.dst, N) || resid->ne[1] != T || add.dst.ne[1] != T) return 0;
    if (overlaps(add.dst, mm.src[1])) return 0;
    if (!covers(add.dst, mm.dst) && live_after(ops, n, i + 2, mm.dst)) return 0;
    ExecNode g;
    g.kind = EX_GEMV; g.nseg = 1; g.K = mm.src[0].ne[0]; g.ncols = (int)T; g.w_const = true;
    g.seg[0] = seg_of(mm, (float *)add.dst.data, (size_t)N, (const float *)resid->data);
    g.act = GemvActDesc{};
    g.act.mode = ACT_F32; g.act.x = (const float *)mm.src[1].data; g.act.x_stride = mm.src[1].nb[1];
    out.push_back(g);
    return 2;
}

// NORM MUL MUL_MAT (final norm + output projection, or any single consumer)
static int match_norm_mm(const b200_op *ops, int n, int i, std::vector<ExecNode> &out) {
    const b200_tensor *xin; const float *nw; float eps;
    if (i + 2 >= n || !match_norm_mul(ops, n, i, xin, nw, eps) || !is_decode_mm(ops[i + 2])) return 0;
    const b200_op &mm = ops[i + 2];
    if (!same_tensor(mm.src[1], ops[i + 1].dst) || !(mm.src[0].flags & B200_TENSOR_FLAG_WEIGHT)) return 0;
    if (live_after(ops, n, i + 3, ops[i].dst) || live_after(ops, n, i + 3, ops[i + 1].dst)) return 0;
    if (overlaps(mm.dst, *xin)) return 0;
    ExecNode g;
    g.kind = EX_GEMV; g.nseg = 1; g.K = xin->ne[0]; g.ncols = (int)mm.dst.ne[1]; g.w_const = true;
    g.seg[0] = seg_of(mm, (float *)mm.dst.data, (size_t)mm.src[0].ne[1], nullptr);
    g.act = GemvActDesc{};
    g.act.mode = ACT_F32_NORM; g.act.x = (const float *)xin->data; g.act.x_stride = xin->nb[1]; g.act.x2 = nw; g.act.eps = eps;
    out.push_back(g);
    return 3;
}

// returns the list actually executed
static int fuse(b200_ctx *ctx, const b200_op *ops, int n, std::vector<ExecNode> &out) {
    out.clear();
    out.reserve(n);
    // scratch for the intermediates of the layer fusions (q,k,v and gate,up): sized from the largest matmuls in the list
    FuseScratch fs = {};
    bool layer_fusion = ctx->opt_fusion >= 2 && !ctx->opt_cpu_exact;     // parity mode: matmuls go through exact.cu one by one
    if (layer_fusion) {
        int64_t maxN = 0;
        for (int i = 0; i < n; i++) if (ops[i].op == B200_OP_MUL_MAT && is_decode_mm(ops[i]) && ops[i].src[0].ne[1] < (1 << 16)) maxN = std::max(maxN, ops[i].src[0].ne[1]);
        if (maxN == 0) layer_fusion = false;
        else {
            int64_t maxT = 1;
            for (int i = 0; i < n; i++) if (ops[i].op == B200_OP_MUL_MAT && is_decode_mm(ops[i])) maxT = std::max(maxT, ops[i].dst.ne[1]);
            const size_t per = (size_t)maxN * 4 * (size_t)(maxT <= 4 ? 4 : FUSE_MAX_T);
            float *base = (float *)ctx->get_scratch(SCRATCH_FUSE, per * 5);
            if (!base) return B200_ERR_ALLOC;
            fs.q = base; fs.k = base + per / 4; fs.v = base + 2 * (per / 4); fs.g = base + 3 * (per / 4); fs.u = base + 4 * (per / 4);
        }
    }
    for (int i = 0; i < n;) {
        const b200_op &a = ops[i];
        if (layer_fusion) {
            int used = 0;
            if (a.op == B200_OP_RMS_NORM) {
                used = match_attention(ctx, ops, n, i, fs, out);
                if (!used) used = match_ffn(ops, n, i, fs, out);
                if (!used) used = match_norm_mm(ops, n, i, out);
            } else if (a.op == B200_OP_MUL_MAT) {
                used = match_mm_add(ops, n, i, out);
            }
            if (used) { i += used; continue; }
        }
        if (i + 1 < n) {
            const b200_op &b = ops[i + 1];
            // RMS_NORM -> MUL(norm, weight): y = rms_norm(x) * w
            if (a.op == B200_OP_RMS_NORM && b.op == B200_OP_MUL && same_tensor(b.src[0], a.dst) && b.src[1].type == B200_TYPE_F32 &&
                b.src[1].nb[0] == 4 && b.src[1].ne[0] == a.dst.ne[0] &&
                (b.dst.data == a.dst.data || !live_after(ops, n, i + 2, a.dst))) {
                b200_op f = a;
                f.op = B200_OP_RMS_NORM_MUL;
                f.n_src = 2;
                f.src[1] = b.src[1];
                f.dst = b.dst;
                if (supports_glue(&f)) { ExecNode e; e.op = f; out.push_back(e); i += 2; continue; }
            }
            // SILU(gate) -> MUL(silu, up)
            if (a.op == B200_OP_SILU && b.op == B200_OP_MUL && same_tensor(b.src[0], a.dst) &&
                (b.dst.data == a.dst.data || !live_after(ops, n, i + 2, a.dst))) {
                b200_op f = a;
                f.op = B200_OP_SWIGLU_FUSED;
                f.n_src = 2;
                f.src[1] = b.src[1];
                f.dst = b.dst;
                if (supports_glue(&f)) { ExecNode e; e.op = f; out.push_back(e); i += 2; continue; }
            }
        }
        ExecNode e;
        e.op = a;
        out.push_back(e);
        i++;
    }
    // weight look-ahead: a fused GEMV asks the L2 to start fetching the constant weights of the GEMV-like nodes that follow.
    // Adjacent successor: its matrices.  When attention sits in between (rope+store, flash_attn, combine move ~3 MB per layer and
    // leave HBM idle for ~15 us), the matrices of the next TWO nodes (wo, then gate|up): they stream into the L2 under the
    // attention kernels; the node in between then skips its own look-ahead (already on its way).
    auto gemv_like = [](const ExecNode &e) {
        return e.kind == EX_GEMV || (e.kind == EX_OP && e.op.op == B200_OP_MUL_MAT && b200_type_is_quant(e.op.src[0].type) && (e.op.src[0].flags & B200_TENSOR_FLAG_WEIGHT));
    };
    auto add_ranges = [](ExecNode &e, const ExecNode &nx) {
        if (nx.kind == EX_GEMV) {
            if (!nx.w_const) return;
            for (int s = 0; s < nx.nseg && e.npf < GEMV_MAX_PF; s++) {
                if (nx.seg[s].expert_id) continue;           // the expert is only known on the device
                e.pf[e.npf].ptr = nx.seg[s].W; e.pf[e.npf].bytes = (size_t)nx.seg[s].N * nx.seg[s].rb; e.npf++;
            }
        } else if (e.npf < GEMV_MAX_PF) {
            e.pf[e.npf].ptr = nx.op.src[0].data; e.pf[e.npf].bytes = (size_t)nx.op.src[0].ne[1] * b200_row_bytes(nx.op.src[0].type, nx.op.src[0].ne[0]); e.npf++;
        }
    };
    std::vector<char> covered(out.size(), 0);
    for (size_t i = 0; i < out.size(); i++) {
        ExecNode &e = out[i];
        if (e.kind != EX_GEMV) continue;
        size_t j = i + 1;
        while (j < out.size() && !gemv_like(out[j])) j++;
        if (j >= out.size()) continue;
        if (j == i + 1) { if (!covered[j]) add_ranges(e, out[j]); continue; }
        add_ranges(e, out[j]); covered[j] = 1;
        size_t k = j + 1;
        if (k < out.size() && gemv_like(out[k])) { add_ranges(e, out[k]); covered[k] = 1; }
    }
    return B200_OK;
}

static int run_list(b200_ctx *ctx, const std::vector<ExecNode> &list) {
    // timing experiments only (results are then wrong): option "debug_skip" / GGML_B200_DEBUG_SKIP bit 0 flash_attn, 1 rope+store, 2 GEMV, 3 all-reduce
    static const int env_skip = getenv("GGML_B200_DEBUG_SKIP") ? atoi(getenv("GGML_B200_DEBUG_SKIP")) : 0;
    const int dbg_skip = env_skip | ctx->opt_debug_skip;
    bool pair_done = false;
    for (const ExecNode &e : list) {
        int rc;
        if (dbg_skip) {
            if ((dbg_skip & 1) && e.kind == EX_OP && e.op.op == B200_OP_FLASH_ATTN_EXT) continue;
            if ((dbg_skip & 2) && e.kind == EX_ROPE_STORE) continue;
            if ((dbg_skip & 4) && e.kind == EX_GEMV) continue;
            if ((dbg_skip & 8) && e.kind == EX_OP && e.op.op == B200_OP_ALLREDUCE) continue;
        }
        if (e.kind == EX_GEMV) {
            if (e.pair == 1 && ctx->opt_ffn_pair) rc = gemv_launch(ctx, e.seg, e.nseg, e.K, e.act, e.ncols, e.w_const, e.pf, e.npf, &pair_done);
            else if (e.pair == 2 && pair_done) {          // the gate|up launch left h = silu(gate) * up in the gate scratch: plain f32 activations
                GemvActDesc a = e.act; a.mode = ACT_F32; a.x2 = nullptr;
                rc = gemv_launch(ctx, e.seg, e.nseg, e.K, a, e.ncols, e.w_const, e.pf, e.npf);
                pair_done = false;
            }
            else rc = gemv_launch(ctx, e.seg, e.nseg, e.K, e.act, e.ncols, e.w_const, e.pf, e.npf);
        }
        else if (e.kind == EX_ROPE_STORE) rc = launch_rope_store(ctx, e.rs);
        else rc = dispatch(ctx, &e.op);
        if (rc) return rc;
    }
    return B200_OK;
}

static bool is_kv_store(const b200_op &o) {
    if (o.op != B200_OP_CPY || o.src[0].type != B200_TYPE_F32) return false;
    const b200_tensor &d = o.dst;
    if (d.type != B200_TYPE_F16 && d.type != B200_TYPE_Q8_0 && d.type != B200_TYPE_Q4_0) return false;
    return d.ne[1] == 1 && d.ne[2] == 1 && d.ne[3] == 1 && !(d.flags & B200_TENSOR_FLAG_WEIGHT);
}

// every rope+store descriptor of a list
static void collect_rope_stores(std::vector<ExecNode> &list, std::vector<RopeStoreDesc *> &out) {
    out.clear();
    for (ExecNode &x : list) if (x.kind == EX_ROPE_STORE) out.push_back(&x.rs);
}
// point every fused rope+store node at its slots of the entry's device table; false if a KV store is not inside such a node
static bool bind_kv_table(GraphCacheEntry &e, const b200_op *ops, std::vector<ExecNode> &list, bool assign) {
    e.node_kv.clear();
    size_t covered = 0;
    int j = 0;
    std::vector<RopeStoreDesc *> rss;
    collect_rope_stores(list, rss);
    for (RopeStoreDesc *rs : rss) {
        int ki = -1, vi = -1;
        for (int idx : e.kv_idx) {
            if (ops[idx].dst.data == rs->k_dst && ki < 0) ki = idx;
            else if (ops[idx].dst.data == rs->v_dst && vi < 0) vi = idx;
        }
        if (ki < 0 || vi < 0) return false;
        e.node_kv.push_back({ki, vi});
        covered += 2;
        if (assign) { rs->k_dst_ind = (void *const *)(e.dev_table + 2 * j); rs->v_dst_ind = (void *const *)(e.dev_table + 2 * j + 1); }
        j++;
    }
    return covered == e.kv_idx.size();
}
static void unbind_kv_table(std::vector<ExecNode> &list) {
    std::vector<RopeStoreDesc *> rss;
    collect_rope_stores(list, rss);
    for (RopeStoreDesc *rs : rss) rs->k_dst_ind = rs->v_dst_ind = nullptr;
}
static int upload_kv_table(b200_ctx *ctx, const GraphCacheEntry &e, const b200_op *ops) {
    if (e.node_kv.empty()) return B200_OK;
    void *host[2 * 512];
    const size_t n = e.node_kv.size() > 512 ? 512 : e.node_kv.size();
    for (size_t j = 0; j < n; j++) { host[2 * j] = ops[e.node_kv[j].first].dst.data; host[2 * j + 1] = ops[e.node_kv[j].second].dst.data; }
    // pageable source: the driver stages it before returning, so `host` may die right away; ordered before the replay on the stream
    CUDA_TRY(cudaMemcpyAsync(e.dev_table, host, 2 * n * sizeof(void *), cudaMemcpyHostToDevice, ctx->stream));
    return B200_OK;
}

// the replay test shared by the fast path and the capture path: entry whose key equals `key` (and, without the indirection table, whose
// KV-store destinations are the same pointers)
static GraphCacheEntry *find_entry(GraphCache &gc, const b200_op *ops, int n_ops, const std::vector<b200_op> &key, const std::vector<int> &kv_idx) {
    for (auto &e : gc.entries) {
        if ((int)e.key.size() != n_ops || memcmp(e.key.data(), key.data(), sizeof(b200_op) * (size_t)n_ops) != 0) continue;
        if (!e.indirect) {                           // exact pointers required
            bool same = e.kv_ptrs.size() == kv_idx.size();
            for (size_t j = 0; same && j < kv_idx.size(); j++) same = e.kv_ptrs[j] == ops[kv_idx[j]].dst.data;
            if (!same) continue;
        }
        return &e;
    }
    return nullptr;
}

extern "C" int b200_graph_compute(b200_ctx *ctx, const b200_op *ops, int n_ops) {
    if (!ctx || (!ops && n_ops)) return B200_ERR_FAILED;
    CUDA_TRY(cudaSetDevice(ctx->device));
    ctx->fa_map_valid = false;            // the mask may have been rewritten between calls
    // ---- fast path: a decode step whose op list (modulo the KV-store destinations) has a captured graph is replayed before any
    //      per-op work (support checks, pattern matching): ~1000 ops per token are otherwise re-validated for nothing ----
    if (ctx->opt_cuda_graphs && n_ops >= 8 && ctx->graph_cache && !ctx->graph_cache->entries.empty()) {
        GraphCache &gc = *ctx->graph_cache;
        std::vector<b200_op> &key = gc.scratch_key;
        key.assign(ops, ops + n_ops);
        std::vector<int> &kv_idx = gc.scratch_idx;
        kv_idx.clear();
        for (int i = 0; i < n_ops; i++) if (is_kv_store(ops[i])) { kv_idx.push_back(i); key[i].dst.data = nullptr; }
        GraphCacheEntry *e = find_entry(gc, ops, n_ops, key, kv_idx);
        if (e && e->exec) {
            if (e->indirect) { int rc = upload_kv_table(ctx, *e, ops); if (rc) return rc; }
            CUDA_TRY(cudaGraphLaunch(e->exec, ctx->stream));
            ctx->launches += 1;
            e->hits++;
            return B200_OK;
        }
    }
    for (int i = 0; i < n_ops; i++)
        if (!b200_supports_op(ctx->device, &ops[i])) {
            b200_set_error("graph op %d (id %d) not supported", i, ops[i].op);
            return B200_ERR_UNSUPPORTED;
        }
    if (g_fuse_debug >= 2) {                 // op list as the backend received it (one line per op: id, dst shape, src0 shape)
        static int dumped = 0;
        if (dumped++ < 3)
            for (int i = 0; i < n_ops && i < 64; i++)
                fprintf(stderr, "[b200 ops] %3d op=%2d dst=[%lld,%lld,%lld] t%d src0=[%lld,%lld,%lld] t%d src1=[%lld,%lld,%lld] t%d\n", i, ops[i].op,
                        (long long)ops[i].dst.ne[0], (long long)ops[i].dst.ne[1], (long long)ops[i].dst.ne[2], ops[i].dst.type,
                        (long long)ops[i].src[0].ne[0], (long long)ops[i].src[0].ne[1], (long long)ops[i].src[0].ne[2], ops[i].src[0].type,
                        (long long)ops[i].src[1].ne[0], (long long)ops[i].src[1].ne[1], (long long)ops[i].src[1].ne[2], ops[i].src[1].type);
    }
    std::vector<ExecNode> list;
    if (ctx->opt_fusion) { int frc = fuse(ctx, ops, n_ops, list); if (frc) return frc; }
    else { list.resize(n_ops); for (int i = 0; i < n_ops; i++) list[i].op = ops[i]; }

    if (!ctx->opt_cuda_graphs || n_ops < 8) return run_list(ctx, list);
    for (int i = 0; i < n_ops; i++)            // row-split matmuls fork to other devices' streams: launched eagerly
        if (ops[i].op == B200_OP_MUL_MAT && (ops[i].src[0].flags & B200_TENSOR_FLAG_SPLIT)) return run_list(ctx, list);

    // only decode-sized steps repeat (a prompt ubatch is seen once, and capturing its ~1000 big launches costs more than it saves)
    {
        bool decode_like = false;
        for (const ExecNode &x : list) {
            decode_like |= x.kind == EX_GEMV;
            // a continuous-batching step (<= 32 token columns) repeats like a decode step; F16/BF16 weights (unfused) included
            const int wt = x.op.src[0].type;
            decode_like |= x.kind == EX_OP && x.op.op == B200_OP_MUL_MAT && x.op.src[1].ne[1] <= 32 && (x.op.src[0].flags & B200_TENSOR_FLAG_WEIGHT) &&
                           (b200_type_is_quant(wt) || wt == B200_TYPE_F16 || wt == B200_TYPE_BF16);
        }
        if (!decode_like && ctx->opt_fusion >= 2) return run_list(ctx, list);
    }
    // ---- CUDA graph replay keyed on the op list modulo the KV-store destinations ----
    if (!ctx->graph_cache) ctx->graph_cache = new GraphCache();
    GraphCache &gc = *ctx->graph_cache;
    std::vector<b200_op> &key = gc.scratch_key;
    key.assign(ops, ops + n_ops);
    std::vector<int> &kv_idx = gc.scratch_idx;
    kv_idx.clear();
    for (int i = 0; i < n_ops; i++) if (is_kv_store(ops[i])) { kv_idx.push_back(i); key[i].dst.data = nullptr; }
    for (auto &e : gc.entries) {
        if ((int)e.key.size() != n_ops || memcmp(e.key.data(), key.data(), sizeof(b200_op) * (size_t)n_ops) != 0) continue;
        if (!e.indirect) {                           // exact pointers required
            bool same = e.kv_ptrs.size() == kv_idx.size();
            for (size_t j = 0; same && j < kv_idx.size(); j++) same = e.kv_ptrs[j] == ops[kv_idx[j]].dst.data;
            if (!same) continue;
        }
        if (e.exec) {
            if (e.indirect) { int rc = upload_kv_table(ctx, e, ops); if (rc) return rc; }
            CUDA_TRY(cudaGraphLaunch(e.exec, ctx->stream));
            ctx->launches += 1;
            e.hits++;
            if (getenv("GGML_B200_GRAPH_DEBUG") && (e.hits & 15) == 1) fprintf(stderr, "[b200 graph] replay hit %d (indirect %d, %zu kv nodes)\n", e.hits, (int)e.indirect, e.node_kv.size());
            return B200_OK;
        }
        // second sighting: capture now.  Scratch must already be large enough (first run grew it).
        if (e.indirect) {
            if (!e.dev_table && cudaMalloc((void **)&e.dev_table, 2 * 512 * sizeof(void *)) != cudaSuccess) { cudaGetLastError(); e.dev_table = nullptr; e.indirect = false; }
            if (e.indirect && (e.node_kv.size() > 512 || !bind_kv_table(e, ops, list, true))) e.indirect = false;
            if (e.indirect) { int rc = upload_kv_table(ctx, e, ops); if (rc) return rc; }
            else { e.kv_ptrs.clear(); for (int idx : kv_idx) e.kv_ptrs.push_back(ops[idx].dst.data); unbind_kv_table(list); }
        }
        cudaGraph_t g = nullptr;
        ctx->capturing = true;
        CUDA_TRY(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
        int rc = run_list(ctx, list);
        cudaError_t ce = cudaStreamEndCapture(ctx->stream, &g);
        ctx->capturing = false;
        if (rc || ce != cudaSuccess || !g) {
            cudaGetLastError();
            if (g) cudaGraphDestroy(g);
            unbind_kv_table(list);
            return run_list(ctx, list);          // fall back to eager launches
        }
        if (cudaGraphInstantiate(&e.exec, g, 0) != cudaSuccess) {
            cudaGetLastError(); e.exec = nullptr; cudaGraphDestroy(g);
            unbind_kv_table(list);
            return run_list(ctx, list);
        }
        cudaGraphDestroy(g);
        CUDA_TRY(cudaGraphLaunch(e.exec, ctx->stream));
        ctx->launches += 1;
        return B200_OK;
    }
    if (gc.entries.size() >= 64) {           // bounded cache: drop the oldest
        if (gc.entries.front().exec) cudaGraphExecDestroy(gc.entries.front().exec);
        if (gc.entries.front().dev_table) cudaFree(gc.entries.front().dev_table);
        gc.entries.erase(gc.entries.begin());
    }
    static const int gdebug = getenv("GGML_B200_GRAPH_DEBUG") ? atoi(getenv("GGML_B200_GRAPH_DEBUG")) : 0;
    if (gdebug && !gc.entries.empty()) {          // why did this list miss?  first difference against the newest entry
        const GraphCacheEntry &le = gc.entries.back();
        if ((int)le.key.size() != n_ops) fprintf(stderr, "[b200 graph] miss: %d ops vs %zu\n", n_ops, le.key.size());
        else for (int i = 0; i < n_ops; i++) if (memcmp(&le.key[i], &key[i], sizeof(b200_op))) {
            const b200_op &a = le.key[i], &b = key[i];
            fprintf(stderr, "[b200 graph] miss at op %d/%d (id %d): dst %p/%p ne %lld,%lld/%lld,%lld src0 %p/%p ne1 %lld/%lld src1 %p/%p src3 %p/%p params0 %d/%d\n", i, n_ops, b.op,
                    a.dst.data, b.dst.data, (long long)a.dst.ne[0], (long long)a.dst.ne[1], (long long)b.dst.ne[0], (long long)b.dst.ne[1], a.src[0].data, b.src[0].data,
                    (long long)a.src[0].ne[1], (long long)b.src[0].ne[1], a.src[1].data, b.src[1].data, a.src[3].data, b.src[3].data, a.params[0], b.params[0]);
            break;
        }
    }
    if (gdebug) {
        int ng = 0, nr = 0;
        for (const ExecNode &x : list) { ng += x.kind == EX_GEMV; nr += x.kind == EX_ROPE_STORE; }
        fprintf(stderr, "[b200 graph] new list: %d ops -> %zu nodes (%d fused gemv, %d rope+store), %zu kv stores; op ids:", n_ops, list.size(), ng, nr, kv_idx.size());
        for (int i = 0; i < n_ops && i < 64; i++) fprintf(stderr, " %d", ops[i].op);
        fprintf(stderr, "\n");
    }
    GraphCacheEntry ne;
    ne.key = key;
    ne.kv_idx = kv_idx;
    for (int idx : kv_idx) ne.kv_ptrs.push_back(ops[idx].dst.data);
    ne.indirect = !kv_idx.empty() && bind_kv_table(ne, ops, list, false);
    gc.entries.push_back(std::move(ne));
    return run_list(ctx, list);
}
