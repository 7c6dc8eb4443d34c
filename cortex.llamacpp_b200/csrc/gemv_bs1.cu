// gemv_bs1.cu -- the batch-1 decode GEMV for K-quant weights (Q4_K / Q5_K / Q6_K): the kernel a decoded token spends
// most of its time in.  Same contract as gemv.cu (it is dispatched from gemv_launch for ncols == 1), different shape:
//
//   * gemv.cu's general kernel is ~100 KB of SASS (1-4 columns x 1/2/4 rows per stage x five formats) and owns a whole
//     SM (227 KB ring, 96 registers x 640 threads).  At batch 1 a CTA of a Llama-3-8B matmul only sees 64-450 KB of
//     weights, so a launch lives for a few microseconds and its cost is start-up, instruction fetch and tail, not
//     streaming (ncu: stall_no_instruction was the top stall, profiles/r1_gemv_v5_diag.txt).  This kernel is built
//     for that regime:
//   * HALF an SM per CTA (<= 113 KB shared memory, 512 threads, <= 64 registers): under programmatic dependent launch
//     the NEXT matmul's CTA becomes resident next to the current one and streams its (constant) weights into its own
//     ring while the current one is still computing -- HBM keeps streaming across the kernel boundary;
//   * tiny code: one row at a time, one item-loop per format, nothing unrolled over rows or columns;
//   * lean block decoders: Q4_K needs ~80 instructions per 64 weights (packed 6-bit scale unpack with PRMT, high
//     nibbles multiplied in place (x16, exact) instead of shifted, mins through dp2a on per-32 activation sums);
//     Q6_K walks its 2-byte aligned blocks with aligned 32-bit loads + a run-time PRMT selector (no divergent paths);
//   * the producer warp never blocks: every lane owns one ring stage and polls its `empty` barrier, so stages are
//     re-armed as soon as they are released (no round-synchronous bursts); consumer warp w owns stages w, w+ncw, ...
//     for the whole launch, so the 1-bit mbarrier phase can never alias;
//   * rows are split evenly per segment (CTA c takes rows [N*c/G, N*(c+1)/G) of every segment): no search, no
//     thread-0 prologue, and the producer issues its first copies before the CTA-wide barrier.
// Integer arithmetic is the CPU oracle's (ggml_vec_dot_q{4,5,6}_K_q8_K) bit for bit; activations are quantised in the
// prologue exactly like quantize_row_q8_K_ref (quant_warp.cuh).
// Algorithmic bytes per launch: sum N*K*bpw (weights) + 4K (f32 activations, x2 for swiglu) + 4N (output).
#include "common.cuh"
#include "quant_warp.cuh"
#include "gemv.h"
#include "gemv_bs1_items.cuh"

namespace {

constexpr int BS1_MAX_STAGES = 32;      // one producer lane per stage
constexpr int BS1_MAX_THREADS = 1024;   // consumer warps + 1 producer warp; the launch picks 512 or 1024 (GGML_B200_BS1_WARPS)

struct Bs1Seg {
    const uint8_t *W;
    float *        dst;
    const float *  residual;
    const int32_t *expert_id;
    size_t         expert_stride;
    uint32_t       rb;                  // bytes per row
    int            type, N, R;          // rows per ring stage (power of two)
    int            q, rem, lgR;         // N = q * grid + rem: CTA c owns rows [c*q + min(c, rem), (c+1)*q + min(c+1, rem))
};

struct Bs1Params {
    Bs1Seg         seg[GEMV_MAX_SEG];
    int            nseg, K, act_mode;
    const float *  x, *x2;
    float          eps;
    double         inv_K;                      // 1 / K when K is a power of two (exact), else 0
    int            nstages;
    uint32_t       stage_bytes;
    int            w_const, use_pdl, ncw;      // ncw: consumer warps (blockDim / 32 - 1)
    int            cs;                         // thread-block cluster size sharing the activation prologue (1 = none)
    uint32_t       off_aq64, off_aq128, off_ad, off_s32, off_s16, off_ring;   // 0 = layout not needed (aq*, s*)
    const uint8_t *pf_ptr[GEMV_MAX_PF];     // L2 look-ahead: weight ranges of the launches that follow (gemv.h)
    unsigned long long pf_bytes[GEMV_MAX_PF];
    int            window;                     // first-fill window in stages (0 = the whole ring at once)
    int            pair;                       // 1: seg 0 = gate, seg 1 = up (same rows): the epilogue writes silu(gate) * up into seg[0].dst, nothing else
    uint32_t       off_gval, off_gflag;        // pair mode: this CTA's gate row results + "ready" words
    int            npf, pf_late;               // pf_late: issue after this launch's own copies (HBM idles through tail, boundary and prologue)
    unsigned long long *prof;           // optional [grid][32] globaltimer stamps (tools/bs1_prof.py)
};

constexpr int TB_Q4_K = 1, TB_Q5_K = 2, TB_Q6_K = 4;

__device__ __forceinline__ bool mbar_test_wait(uint64_t *bar, uint32_t parity) {      // non-blocking poll
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
using namespace bs1;        // the block decoders live in gemv_bs1_items.cuh (host/device portable: tests/host_emul runs them on the CPU)

// ---------------------------------------------------------------------------------------------- prologue
// f32 activations (optionally rms_norm(x)*w or silu(g)*u) -> q8_K in shared memory, bit-exact vs quantize_row_q8_K_ref
#define PROFQ(slot) do { if (p.prof && lane == 0 && warp == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); p.prof[(size_t)blockIdx.x * 32 + (slot)] = t_; } } while (0)
// ---- thread-block cluster helpers: the CTAs of a cluster split the activation prologue and write each quantised block into
//      every member's shared memory (distributed shared memory), so a long activation vector is read and quantised once per
//      cluster instead of once per CTA ----
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank)); return r;
}
__device__ __forceinline__ void st_cluster_v2(uint32_t addr, uint2 v) { asm volatile("st.shared::cluster.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(v.x), "r"(v.y) : "memory"); }
__device__ __forceinline__ void st_cluster_u32(uint32_t addr, uint32_t v) { asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void st_cluster_u16(uint32_t addr, uint16_t v) { asm volatile("st.shared::cluster.u16 [%0], %1;" ::"r"(addr), "h"(v) : "memory"); }
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }

// one warp: 256 activations (lane owns v[0..7]) -> q8_K block b in the shared-memory layouts (of every CTA of the cluster)
__device__ __forceinline__ void bs1_quant_chunk(const Bs1Params &p, uint8_t *smem, int b, int lane, const float (&v)[8]) {
    const int e0 = b * 256 + lane * 8;
    uint2 qp; float d; int pair;
    warp_quant_q8k(v, lane, qp, d, pair);                // pair: 16-element sum, valid in even lanes
    const int quad = pair + __shfl_xor_sync(0xffffffffu, pair, 2);
    const uint32_t o_s16 = p.off_s16 + (uint32_t)(b * 16 + (lane >> 1)) * 2, o_s32 = p.off_s32 + (uint32_t)(b * 8 + (lane >> 2)) * 2;
    const uint32_t o_d = p.off_ad + (uint32_t)b * 4;
    const uint32_t o_q64 = p.off_aq64 + (uint32_t)((e0 >> 8) * 272 + (e0 & 255)), o_q128 = p.off_aq128 + (uint32_t)((e0 >> 7) * 144 + (e0 & 127));
    if (p.cs <= 1) {
        if (p.off_s16 && (lane & 1) == 0) *(int16_t *)(smem + o_s16) = (int16_t)pair;
        if (p.off_s32 && (lane & 3) == 0) *(int16_t *)(smem + o_s32) = (int16_t)quad;
        if (lane == 0) *(float *)(smem + o_d) = d;
        if (p.off_aq64)  *(uint2 *)(smem + o_q64) = qp;
        if (p.off_aq128) *(uint2 *)(smem + o_q128) = qp;
    } else {
        const uint32_t base = smem_u32(smem);
        for (int r = 0; r < p.cs; r++) {
            const uint32_t rb = mapa_shared(base, (uint32_t)r);
            if (p.off_s16 && (lane & 1) == 0) st_cluster_u16(rb + o_s16, (uint16_t)(int16_t)pair);
            if (p.off_s32 && (lane & 3) == 0) st_cluster_u16(rb + o_s32, (uint16_t)(int16_t)quad);
            if (lane == 0) st_cluster_u32(rb + o_d, __float_as_uint(d));
            if (p.off_aq64)  st_cluster_v2(rb + o_q64, qp);
            if (p.off_aq128) st_cluster_v2(rb + o_q128, qp);
        }
    }
}
__device__ __forceinline__ void bs1_apply_mode(const Bs1Params &p, float (&v)[8], const float4 &w0, const float4 &w1, float norm_scale) {
    const float w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
    if (p.act_mode == ACT_F32_NORM) {
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = __fmul_rn(__fmul_rn(v[j], norm_scale), w[j]);
    } else if (p.act_mode == ACT_F32_SWIGLU) {
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = __fmul_rn(ggml_silu_lane(v[j]), w[j]);
    }
}
// sum over the consumer warps of per-warp partial sums of squares -> 1/rms (rms_norm like glue.cu / the CPU oracle: sum in double)
// `nact` warps (0 .. nact - 1) hold blocks of the vector: only they meet at the barrier and need the result (the others would add exact zeros)
__device__ __forceinline__ float bs1_norm_scale(const Bs1Params &p, double *s_red, double s, int warp, int lane, int nact) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) s_red[warp] = s;
    named_bar_sync(2, nact * 32);
    // every warp adds the <= 31 partial sums with the same shuffle tree (fixed order => identical on all warps and CTAs)
    double t = lane < nact ? s_red[lane] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    // K a power of two (4096, 8192 ...): the division is an exact scaling, done as one multiply
    const double mean = p.inv_K != 0.0 ? t * p.inv_K : t / (double)p.K;
    return __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn((float)mean, p.eps)));
}
// f32 activations (optionally rms_norm(x)*w or silu(g)*u) -> q8_K in shared memory, bit-exact vs quantize_row_q8_K_ref.
// K <= 2 * 256 * ncw (every llama shape at batch 1): each warp holds its <= 2 blocks in registers, so x is read ONCE even
// when the rms_norm needs the sum of squares of the whole vector first.
__device__ __forceinline__ void bs1_prologue(const Bs1Params &p, uint8_t *smem, double *s_red, int warp, int lane) {
    const int nchunk = p.K >> 8, ncw = p.ncw;
    const int cs = p.cs, crank = cs > 1 ? (int)cluster_ctarank() : 0;        // cluster mode: CTA `crank` takes blocks b = cs * j + crank
    if (nchunk <= 2 * ncw * cs) {
        float4 xa[2][2], xb[2][2];
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int b = (warp + u * ncw) * cs + crank;
            xa[u][0] = xa[u][1] = xb[u][0] = xb[u][1] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (b < nchunk) {
                const int e0 = b * 256 + lane * 8;
                xa[u][0] = *(const float4 *)(p.x + e0); xa[u][1] = *(const float4 *)(p.x + e0 + 4);
                if (p.act_mode != ACT_F32) { xb[u][0] = *(const float4 *)(p.x2 + e0); xb[u][1] = *(const float4 *)(p.x2 + e0 + 4); }
            }
        }
        float norm_scale = 1.0f;
        if (p.prof) { asm volatile("" : "+f"(xa[0][0].x)); PROFQ(26); }
        const int nact = min(ncw, nchunk);           // norm mode never runs in clusters: warp w holds blocks w and w + ncw
        if (p.act_mode == ACT_F32_NORM && warp < nact) {
            double s = 0.0;
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const float v[8] = {xa[u][0].x, xa[u][0].y, xa[u][0].z, xa[u][0].w, xa[u][1].x, xa[u][1].y, xa[u][1].z, xa[u][1].w};
#pragma unroll
                for (int j = 0; j < 8; j++) s += (double)__fmul_rn(v[j], v[j]);
            }
            if (p.prof) { asm volatile("" : "+d"(s)); PROFQ(27); }
            norm_scale = bs1_norm_scale(p, s_red, s, warp, lane, nact);
            if (p.prof) { asm volatile("" : "+f"(norm_scale)); PROFQ(28); }
        }
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int b = (warp + u * ncw) * cs + crank;
            if (b < nchunk) {
                float v[8] = {xa[u][0].x, xa[u][0].y, xa[u][0].z, xa[u][0].w, xa[u][1].x, xa[u][1].y, xa[u][1].z, xa[u][1].w};
                if (p.prof) { asm volatile("" : "+f"(v[0])); if (u == 0) PROFQ(24); }
                bs1_apply_mode(p, v, xb[u][0], xb[u][1], norm_scale);
                bs1_quant_chunk(p, smem, b, lane, v);
                if (p.prof && u == 0) PROFQ(25);
            }
        }
        return;
    }
    // long rows: stream the blocks (x is read twice in rms_norm mode)
    float norm_scale = 1.0f;
    if (p.act_mode == ACT_F32_NORM) {
        double s = 0.0;
        for (int i = threadIdx.x; i < p.K; i += ncw * 32) { const float v = p.x[i]; s += (double)__fmul_rn(v, v); }
        norm_scale = bs1_norm_scale(p, s_red, s, warp, lane, ncw);
    }
#pragma unroll 1
    for (int b = warp; b < nchunk; b += ncw) {
        const int e0 = b * 256 + lane * 8;
        const float4 a0 = *(const float4 *)(p.x + e0), a1 = *(const float4 *)(p.x + e0 + 4);
        float4 w0 = a0, w1 = a1;
        if (p.act_mode != ACT_F32) { w0 = *(const float4 *)(p.x2 + e0); w1 = *(const float4 *)(p.x2 + e0 + 4); }
        float v[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        bs1_apply_mode(p, v, w0, w1, norm_scale);
        bs1_quant_chunk(p, smem, b, lane, v);
    }
}

// Row result -> destination.  Pair mode (the FFN's gate|up launch): the gate row's value is parked in shared memory; the warp that
// finishes the UP row of the same index (chunks of seg 1 follow all chunks of seg 0: ~3 ring passes later, usually another warp)
// picks it up and stores h = silu(gate) * up, computed exactly like the swiglu activation prologue does (ggml_silu_lane, then one
// rounded multiply).  The down projection then reads ONE f32 vector and needs no expf in its prologue.  A warp never waits while it
// holds a ring stage (the stage is released before the row reduction), so the gate rows always make progress.
__device__ __forceinline__ void bs1_store_row(const Bs1Params &p, const Bs1Seg &sg, int s, int o, int ol, float acc, float *gval, volatile uint32_t *gflag) {
    if (p.pair) {
        if (s == 0) {
            gval[ol] = acc;
            __threadfence_block();
            gflag[ol] = 1u;
        } else {
            while (gflag[ol] == 0u) { }
            __threadfence_block();
            const float g = ((volatile float *)gval)[ol];
            p.seg[0].dst[o] = __fmul_rn(ggml_silu_lane(g), acc);
        }
        return;
    }
    if (sg.residual) acc = __fadd_rn(acc, sg.residual[o]);
    sg.dst[o] = acc;
}

// the weights of the launches that follow: ask the L2 to start fetching this CTA's 1/G of every range (fire and forget)
__device__ __forceinline__ void bs1_l2_lookahead(const Bs1Params &p, int G, int c, int lane) {
    constexpr unsigned long long PIECE = 8192;
    for (int r = 0; r < p.npf; r++) {
        const unsigned long long per = ((p.pf_bytes[r] / G) + 15ull) & ~15ull;
        const unsigned long long b0 = per * c, lim = p.pf_bytes[r] & ~15ull;
        const unsigned long long b1 = b0 + per < lim ? b0 + per : lim;
        for (unsigned long long o = b0 + (unsigned long long)lane * PIECE; o < b1; o += 32 * PIECE) {
            const uint32_t n = (uint32_t)(b1 - o < PIECE ? b1 - o : PIECE);
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p.pf_ptr[r] + o), "r"(n) : "memory");
        }
    }
}

template <int TYPES>
__global__ void __launch_bounds__(BS1_MAX_THREADS, 1) b200_gemv_bs1_kernel(const Bs1Params p) {
    const int BS1_NCW = p.ncw, BS1_THREADS = (p.ncw + 1) * 32;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *full  = (uint64_t *)smem;                  // [32]
    uint64_t *empty = full + BS1_MAX_STAGES;             // [32]
    double *  s_red = (double *)(empty + BS1_MAX_STAGES);    // [32]
    uint8_t * ring  = smem + p.off_ring;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int G = gridDim.x, c = blockIdx.x;
    const int ns = p.nstages;
#define PROF(slot) do { if (p.prof && lane == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); p.prof[(size_t)blockIdx.x * 32 + (slot)] = t_; } } while (0)
    if (warp == 0) PROF(0);
    // programmatic dependent launch: the next kernel's CTAs may become resident right away (half an SM is left for them);
    // everything of theirs that depends on our output blocks in griddepcontrol.wait until this grid has completed
    if (p.use_pdl) pdl_trigger();

    // ---- this CTA's rows: an even share of every segment; chunk = R rows of one segment ----
    int lo[GEMV_MAX_SEG], hi[GEMV_MAX_SEG], ch0[GEMV_MAX_SEG + 1];
    ch0[0] = 0;
#pragma unroll
    for (int s = 0; s < GEMV_MAX_SEG; s++) {
        lo[s] = hi[s] = 0;
        if (s < p.nseg) {
            lo[s] = c * p.seg[s].q + min(c, p.seg[s].rem);
            hi[s] = (c + 1) * p.seg[s].q + min(c + 1, p.seg[s].rem);
        }
        ch0[s + 1] = ch0[s] + (s < p.nseg ? (hi[s] - lo[s] + p.seg[s].R - 1) >> p.seg[s].lgR : 0);
    }
    const int nchunks = ch0[GEMV_MAX_SEG];

    if (warp == BS1_NCW) {
        // ------------------------------------------------------------------ producer: lane l owns ring stage l
        if (lane < ns) { mbar_init(&full[lane], 1); mbar_init(&empty[lane], 1); }
        mbar_fence_init();
        __syncwarp();
        if (p.cs > 1) cluster_arrive();      // cluster mode: one cluster-wide barrier covers the mbarrier init and every member's activation stores
        else asm volatile("bar.arrive 1, %0;" ::"r"(BS1_THREADS) : "memory");       // consumers learn about the barriers at the end of their prologue
        bool any_expert = false;
#pragma unroll
        for (int s = 0; s < GEMV_MAX_SEG; s++) any_expert |= s < p.nseg && p.seg[s].expert_id != nullptr;
        bool waited = false;
        if (p.use_pdl && (!p.w_const || any_expert)) { pdl_wait(); waited = true; }
        const uint64_t pol = l2_policy_evict_first();
        int i = lane, use = 0;
        bool first_pass = true;
        const int win = p.window > 0 ? p.window : BS1_MAX_STAGES;
        PROF(1);
        while (__any_sync(0xffffffffu, lane < ns && i < nchunks)) {
            // first fill: a sliding window of `win` stages in flight per SM (stage l is issued when stage l - win has landed) instead of the
            // whole ring at once -- 32 MB queued chip-wide would put 3-5 us of DRAM queueing in front of the first stage AND of the
            // activation loads; 8-12 stages cover the bandwidth-delay product.  Afterwards a stage is re-armed the moment it is released.
            // "stage l - win has landed" = its `full` barrier is past phase 0, OR its lane has already re-armed it (use >= 2: a re-arm needs
            // the consumer's release, which needs the landing).  The second clause is monotonic: the 1-bit phase test alone would read
            // false again after an even number of landings, should this warp ever be held off for a whole consume + refill period.
            const int use_behind = __shfl_sync(0xffffffffu, use, lane >= win ? lane - win : lane);
            bool go = lane < ns && i < nchunks;
            if (go) go = use == 0 ? (lane < win || use_behind >= 2 || mbar_test_wait(&full[lane - win], 0)) : mbar_test_wait(&empty[lane], (use - 1) & 1);
            if (go) {
                int s = 0, lo_s = lo[0], hi_s = hi[0], c0 = 0;
#pragma unroll
                for (int t = 1; t < GEMV_MAX_SEG; t++) if (t < p.nseg && i >= ch0[t]) { s = t; lo_s = lo[t]; hi_s = hi[t]; c0 = ch0[t]; }
                const Bs1Seg &sg = p.seg[s];
                const int row = lo_s + (i - c0) * sg.R;
                const int nr = min(sg.R, hi_s - row);
                const uint8_t *Wb = sg.expert_id ? sg.W + (size_t)(*sg.expert_id) * sg.expert_stride : sg.W;
                const uint8_t *src = Wb + (size_t)row * sg.rb;
                const uint32_t extra = (uint32_t)((uintptr_t)src & 15);
                const uint32_t bytes = (extra + (uint32_t)nr * sg.rb + 15u) & ~15u;
                mbar_arrive_expect_tx(&full[lane], bytes);
                bulk_g2s_hint(ring + (size_t)lane * p.stage_bytes, src - extra, bytes, &full[lane], pol);
                i += ns; use++;
            }
            if (first_pass) {
                first_pass = false;
                PROF(2);
                if (p.npf && !p.pf_late) bs1_l2_lookahead(p, G, c, lane);
            }
        }
        PROF(3);
        if (p.npf && p.pf_late) bs1_l2_lookahead(p, G, c, lane);
        if (p.use_pdl && !waited) pdl_wait();
        return;
    }

    // ---------------------------------------------------------------------- consumers: prologue
    float *gval = (float *)(smem + p.off_gval);
    volatile uint32_t *gflag = (volatile uint32_t *)(smem + p.off_gflag);
    if (p.pair) for (int i = threadIdx.x; i < hi[0] - lo[0]; i += BS1_NCW * 32) gflag[i] = 0u;      // published by the prologue's CTA barrier
    if (p.use_pdl) pdl_wait();          // the activations belong to the previous kernels
    if (warp == 0) PROF(4);
    bs1_prologue(p, smem, s_red, warp, lane);
    if (p.cs > 1) { cluster_arrive(); cluster_wait(); }       // every member's blocks have landed in this CTA's shared memory
    else named_bar_sync(1, BS1_THREADS);     // activations complete + mbarriers initialised (producer arrived long ago)
    if (warp == 0) PROF(5);
    if (nchunks == 0) return;

    // ---------------------------------------------------------------------- consumers: main loop
    const uint8_t *aq64 = smem + p.off_aq64, *aq128 = smem + p.off_aq128;
    const uint32_t *s32 = (const uint32_t *)(smem + p.off_s32);
    const U4 *s16 = (const U4 *)(smem + p.off_s16);
    const float *ad = (const float *)(smem + p.off_ad);
    const int nblk = p.K >> 8, nit128 = p.K >> 7;
#pragma unroll 1
    for (int use = 0; use * ns < nchunks; use++) {
#pragma unroll 1
        for (int st = warp; st < ns; st += BS1_NCW) {
            const int i = use * ns + st;
            if (i >= nchunks) break;
            int s = 0, lo_s = lo[0], hi_s = hi[0], c0 = 0;
#pragma unroll
            for (int t = 1; t < GEMV_MAX_SEG; t++) if (t < p.nseg && i >= ch0[t]) { s = t; lo_s = lo[t]; hi_s = hi[t]; c0 = ch0[t]; }
            const Bs1Seg &sg = p.seg[s];
            const int row0 = lo_s + (i - c0) * sg.R;
            const int nr = min(sg.R, hi_s - row0);
            const uint8_t *Wb = sg.expert_id ? sg.W + (size_t)(*sg.expert_id) * sg.expert_stride : sg.W;
            const uint32_t extra = (uint32_t)((uintptr_t)(Wb + (size_t)row0 * sg.rb) & 15);
            const uint8_t *rowp = ring + (size_t)st * p.stage_bytes + extra;
            const int ty = sg.type;
            mbar_wait(&full[st], use & 1);
            if (i == 0) PROF(6);
            if ((TYPES & (TB_Q4_K | TB_Q5_K)) && ((TYPES & TB_Q6_K) == 0 || ty != B200_TYPE_Q6_K)) {
                // Q4_K / Q5_K: a whole block per lane.  Short rows (< 32 blocks): two rows per pass, one per half-warp;
                // long rows (K >= 8192): all 32 lanes on one row, so a row costs ceil(nblk / 32) block decodes of latency
                const bool q5 = (TYPES & TB_Q5_K) && (TYPES == TB_Q5_K || ty == B200_TYPE_Q5_K);
                const int lpr = (nblk >= 32 && sg.R == 1) ? 32 : 16, rpp = 32 / lpr;          // lanes per row, rows per pass
                const int sub = lane / lpr, bl = lane % lpr;
                const U4 *sums4 = (const U4 *)s32;
                const uint32_t bbytes = q5 ? 176u : 144u;
#pragma unroll 1
                for (int r = 0; r < nr; r += rpp) {
                    const bool mine = r + sub < nr;
                    const uint8_t *rp = rowp + (size_t)(r + (mine ? sub : 0)) * sg.rb;
                    float acc = 0.0f;
#pragma unroll 1
                    for (int blk = bl; blk < nblk; blk += lpr) {
                        const uint8_t *b = rp + blk * bbytes;
                        const uint8_t *ap = aq64 + blk * 272;
                        if ((TYPES & TB_Q5_K) && q5) acc += block_q45k<true>(b, ap, sums4[blk], ad[blk]);
                        else if (TYPES & TB_Q4_K) acc += block_q45k<false>(b, ap, sums4[blk], ad[blk]);
                    }
                    if (r + rpp >= nr) {                 // stage bytes consumed: hand it back before the reduction
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&empty[st]);
                    }
                    if (lpr == 32) acc += __shfl_xor_sync(0xffffffffu, acc, 16);
#pragma unroll
                    for (int o = 8; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
                    if (bl == 0 && mine) bs1_store_row(p, sg, s, row0 + r + sub, row0 + r + sub - lo_s, acc, gval, gflag);
                }
            } else if (TYPES & TB_Q6_K) {
#pragma unroll 1
                for (int r = 0; r < nr; r++, rowp += sg.rb) {
                    float acc = 0.0f;
#pragma unroll 1
                    for (int it = lane; it < nit128; it += 32) acc += item_q6k(rowp, it, aq128, s16, ad);
                    if (r == nr - 1) {
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&empty[st]);
                    }
                    acc = warp_reduce_sum(acc);
                    if (lane == 0) bs1_store_row(p, sg, s, row0 + r, row0 + r - lo_s, acc, gval, gflag);
                }
            }
            if (i == 0) PROF(7);
        }
    }
    PROF(8 + (warp & 15));               // consumer warps' finish times (two warps share a slot: the later one wins)
#undef PROF
}

int g_bs1_ctas = 0, g_bs1_smem_kb = 0, g_bs1_off = 0, g_bs1_warps = 0, g_bs1_cluster = 4, g_bs1_lpr32 = 1, g_bs1_window = 64;     // window: measured best at 48-64 KB per SM (+1.5 % on the decode step)
bool g_bs1_env = false;

template <int TYPES>
int bs1_launch_t(b200_ctx *ctx, const Bs1Params &p, int grid, size_t smem_bytes) {
    auto kern = b200_gemv_bs1_kernel<TYPES>;
    static bool attr_set[16] = {false};
    if (!attr_set[ctx->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->smem_optin));
        attr_set[ctx->device & 15] = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)(p.ncw + 1) * 32);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[2];
    int nattr = 0;
    if (p.use_pdl) {
        attr[nattr].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[nattr].val.programmaticStreamSerializationAllowed = 1;
        nattr++;
    }
    if (p.cs > 1) {
        attr[nattr].id = cudaLaunchAttributeClusterDimension;
        attr[nattr].val.clusterDim.x = (unsigned)p.cs; attr[nattr].val.clusterDim.y = 1; attr[nattr].val.clusterDim.z = 1;
        nattr++;
    }
    cfg.attrs = attr;
    cfg.numAttrs = nattr;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, p));
    ctx->launches++;
    return B200_OK;
}

// how many clusters of `cs` CTAs with this shared-memory size can be resident at once (GPC packing decides); cached per size
template <int TYPES>
int bs1_max_clusters(b200_ctx *ctx, int cs, int threads, size_t smem_bytes) {
    auto kern = b200_gemv_bs1_kernel<TYPES>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->smem_optin);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(ctx->sm_count / cs * cs)); cfg.blockDim = dim3((unsigned)threads); cfg.dynamicSmemBytes = smem_bytes;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cs; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

}  // namespace

// 1 = launched, 0 = not eligible (caller falls through to the general kernel), < 0 = error
int gemv_bs1_try_launch(b200_ctx *ctx, const GemvSegDesc *segs, int nseg, int64_t K, const GemvActDesc &ga, bool w_const,
                        const GemvPf *pf, int npf, int l2pf, bool *pair) {
    const bool want_pair = pair != nullptr;
    if (pair) *pair = false;
    if (!g_bs1_env) {
        if (const char *e = getenv("GGML_B200_BS1_CTAS")) g_bs1_ctas = atoi(e);          // CTAs per SM (1 or 2; default 2)
        if (const char *e = getenv("GGML_B200_BS1_SMEM_KB")) g_bs1_smem_kb = atoi(e);    // shared memory per CTA
        if (const char *e = getenv("GGML_B200_BS1_OFF")) g_bs1_off = atoi(e);
        if (const char *e = getenv("GGML_B200_BS1_CLUSTER")) g_bs1_cluster = atoi(e);   // 1 = off, 2 or 4 CTAs share the prologue of long vectors
        if (const char *e = getenv("GGML_B200_BS1_LPR32")) g_bs1_lpr32 = atoi(e);
        if (const char *e = getenv("GGML_B200_BS1_WARPS")) g_bs1_warps = atoi(e);       // 16 or 32 warps per CTA (default 32)
        if (const char *e = getenv("GGML_B200_BS1_WINDOW")) g_bs1_window = atoi(e);     // first-fill window in KB per SM (0 = whole ring at once)
        g_bs1_env = true;
    }
    if (g_bs1_off || nseg < 1 || nseg > GEMV_MAX_SEG || K <= 0 || (K & 255) || K > 65536) return 0;
    if (ga.mode != ACT_F32 && ga.mode != ACT_F32_NORM && ga.mode != ACT_F32_SWIGLU) return 0;
    if (((uintptr_t)ga.x & 15) || (ga.mode != ACT_F32 && ((uintptr_t)ga.x2 & 15))) return 0;
    int mask = 0;
    for (int s = 0; s < nseg; s++) {
        const int t = segs[s].type;
        if (t == B200_TYPE_Q4_K) mask |= TB_Q4_K; else if (t == B200_TYPE_Q5_K) mask |= TB_Q5_K; else if (t == B200_TYPE_Q6_K) mask |= TB_Q6_K; else return 0;
        if (segs[s].dbgP || segs[s].N <= 0 || segs[s].N > (1 << 22)) return 0;
        if (t != B200_TYPE_Q6_K && (((uintptr_t)segs[s].W & 15) || (segs[s].rb & 15) || (segs[s].expert_stride & 15))) return 0;
        if (t == B200_TYPE_Q6_K && (((uintptr_t)segs[s].W & 1) || (segs[s].expert_stride & 1))) return 0;
    }
    Bs1Params p = {};
    p.nseg = nseg; p.K = (int)K; p.act_mode = ga.mode; p.x = ga.x; p.x2 = ga.x2; p.eps = ga.eps;
    p.inv_K = (K & (K - 1)) == 0 ? 1.0 / (double)K : 0.0;
    p.w_const = w_const ? 1 : 0; p.use_pdl = ctx->opt_pdl;
    // shared memory: barriers | s_red | aq64 | aq128 | d | s32 | s16 | ring
    uint32_t off = 2 * BS1_MAX_STAGES * 8 + 32 * 8;
    const bool need64 = (mask & (TB_Q4_K | TB_Q5_K)) != 0, need128 = (mask & TB_Q6_K) != 0;
    if (need64)  { p.off_aq64 = off;  off += (uint32_t)(K / 256) * 272; off = (off + 15) & ~15u; }
    if (need128) { p.off_aq128 = off; off += (uint32_t)(K / 128) * 144; off = (off + 15) & ~15u; }
    p.off_ad = off; off += (uint32_t)(K / 256) * 4; off = (off + 15) & ~15u;
    if (need64)  { p.off_s32 = off; off += (uint32_t)(K / 32) * 2; off = (off + 15) & ~15u; }
    if (need128) { p.off_s16 = off; off += (uint32_t)(K / 16) * 2; off = (off + 15) & ~15u; }
    static const int pair_off = getenv("GGML_B200_BS1_PAIR") ? !atoi(getenv("GGML_B200_BS1_PAIR")) : 0;
    if (want_pair && !pair_off && nseg == 2 && segs[0].N == segs[1].N && segs[0].N / ctx->sm_count + 1 <= 2048 && !segs[0].residual && !segs[1].residual &&
        !segs[0].expert_id && !segs[1].expert_id) {
        const uint32_t rows = (uint32_t)(segs[0].N / ctx->sm_count + 1);
        p.pair = 1;
        p.off_gval = off; off += rows * 4; off = (off + 15) & ~15u;
        p.off_gflag = off; off += rows * 4; off = (off + 15) & ~15u;
    }
    off = (off + 127) & ~127u;
    p.off_ring = off;
    const int cps = g_bs1_ctas == 2 ? 2 : 1;
    size_t budget = g_bs1_smem_kb > 0 ? (size_t)g_bs1_smem_kb * 1024 : (size_t)220 * 1024;     // measured best: one CTA per SM with a deep ring (profiles/r1_bs1_ab.txt)
    if (budget > ctx->smem_optin) budget = ctx->smem_optin;
    uint32_t max_rb = 0;
    for (int s = 0; s < nseg; s++) max_rb = segs[s].rb > max_rb ? (uint32_t)segs[s].rb : max_rb;
    if ((size_t)off + 2 * ((size_t)max_rb + 160) > budget) return 0;                            // needs >= 2 stages of one row
    const size_t ring_budget = budget - off;
    // stage: whole rows, about ring/32 bytes, at least one row
    const uint32_t target = (uint32_t)(ring_budget / BS1_MAX_STAGES);
    uint32_t stage = 0;
    for (int s = 0; s < nseg; s++) {
        Bs1Seg &g = p.seg[s];
        g.W = segs[s].W; g.dst = segs[s].dst; g.residual = segs[s].residual; g.expert_id = segs[s].expert_id; g.expert_stride = segs[s].expert_stride;
        g.rb = (uint32_t)segs[s].rb; g.type = segs[s].type; g.N = (int)segs[s].N;
        int R = (int)(target / g.rb);
        R = R < 1 ? 1 : (R > 8 ? 8 : R);
        if (g.type != B200_TYPE_Q6_K && R < 2 && (K < 8192 || g_bs1_lpr32 == 0) && 2 * (size_t)g.rb <= 16384) R = 2;      // pair decoder (rows shorter than 32 blocks): two rows per stage
        int lg = 0;
        while ((2 << lg) <= R) lg++;
        g.R = 1 << lg; g.lgR = lg;
        const uint32_t sb = (uint32_t)(((size_t)g.R * g.rb + 32 + 127) & ~(size_t)127);       // +16 misalignment, +16 over-read
        stage = sb > stage ? sb : stage;
    }
    int ns = (int)(ring_budget / stage);
    if (ns > BS1_MAX_STAGES) ns = BS1_MAX_STAGES;
    const int ncw = g_bs1_warps == 16 ? 15 : 31;
    p.ncw = ncw;
    if (ns >= ncw) ns = ns / ncw * ncw;                  // every consumer warp owns the same number of stages
    if (ns < 2) return 0;
    p.nstages = ns; p.stage_bytes = stage;
    // window in bytes, not stages: GGML_B200_BS1_WINDOW is in KB per SM
    p.window = g_bs1_window > 0 ? (int)(((size_t)g_bs1_window * 1024 + stage - 1) / stage) : 0;
    if (p.window >= ns) p.window = 0;
    const size_t smem_bytes = off + (size_t)ns * stage;
    if (l2pf && pf) {
        // l2pf 1: the next launch's first matrix, issued with this launch's first copies (round 1: measured neutral);
        // l2pf 2: every range the graph handed down, issued AFTER this launch's own copies
        static const size_t cap_mb = getenv("GGML_B200_L2PF_MB") ? (size_t)atoi(getenv("GGML_B200_L2PF_MB")) : 96;
        size_t budget_pf = l2pf == 1 ? ((size_t)48 << 20) : (cap_mb << 20);
        p.pf_late = l2pf >= 2;
        for (int r = 0; r < npf && r < (l2pf == 1 ? 1 : GEMV_MAX_PF) && budget_pf > 0; r++) {
            if (!pf[r].ptr || pf[r].bytes < 64) continue;
            const uint8_t *q = (const uint8_t *)pf[r].ptr;
            size_t nb = pf[r].bytes < budget_pf ? pf[r].bytes : budget_pf;
            const uintptr_t mis = (uintptr_t)q & 15;
            if (mis) { q += 16 - mis; nb -= 16; }
            p.pf_ptr[p.npf] = q; p.pf_bytes[p.npf] = nb; p.npf++;
            budget_pf -= nb < budget_pf ? nb : budget_pf;
        }
    }
    if (ctx->prof_buf) {     // rotating per-launch slots so consecutive launches can be laid on one timeline
        p.prof = (unsigned long long *)ctx->prof_buf + (size_t)(ctx->prof_launch % 8) * 296 * 32;
        ctx->prof_launch++;
    }
    int64_t min_rows = segs[0].N;
    for (int s = 1; s < nseg; s++) min_rows = segs[s].N < min_rows ? segs[s].N : min_rows;
    int64_t grid = (int64_t)ctx->sm_count * cps;
    if (grid > min_rows) grid = min_rows;                // every CTA gets at least one row of every segment
    // long activation vectors (a warp would quantise two blocks, every CTA would re-read 50+ KB): share the prologue in a cluster
    p.cs = 1;
    // Only the swiglu prologue (two vectors + expf per element) is worth the cluster barrier, which waits for the LAST member to
    // start (CTAs replace the previous kernel's CTAs one by one: 2 us of skew in a real step); plain f32 vectors -- the down projection
    // after a pair-mode gate|up launch -- are loaded and quantised by every CTA itself: 557 vs 546 tok/s (GGML_B200_BS1_CLUSTER_F32=1 restores)
    static const int cluster_f32 = getenv("GGML_B200_BS1_CLUSTER_F32") ? atoi(getenv("GGML_B200_BS1_CLUSTER_F32")) : 0;
    if (g_bs1_cluster > 1 && !p.pair && (ga.mode == ACT_F32_SWIGLU || (ga.mode == ACT_F32 && cluster_f32)) && (K >> 8) > ncw && grid >= ctx->sm_count / 2) {
        const int cs = g_bs1_cluster >= 4 ? 4 : 2;
        static int max_cl[5] = {0, 0, -1, 0, -1};
        if (max_cl[cs] < 0) {
            switch (mask) {
                case TB_Q4_K: max_cl[cs] = bs1_max_clusters<TB_Q4_K>(ctx, cs, (ncw + 1) * 32, (size_t)220 * 1024); break;
                default:      max_cl[cs] = bs1_max_clusters<TB_Q6_K>(ctx, cs, (ncw + 1) * 32, (size_t)220 * 1024); break;
            }
        }
        int64_t gcl = grid / cs * cs;
        if (max_cl[cs] > 0 && gcl > (int64_t)max_cl[cs] * cs) gcl = (int64_t)max_cl[cs] * cs;      // one wave of co-resident clusters
        if (max_cl[cs] > 0 && gcl >= ctx->sm_count * 3 / 4) { p.cs = cs; grid = gcl; }
    }
    for (int s = 0; s < nseg; s++) { p.seg[s].q = (int)(segs[s].N / grid); p.seg[s].rem = (int)(segs[s].N % grid); }
    if (p.pair && (p.cs > 1 || (segs[0].N + grid - 1) / grid > segs[0].N / ctx->sm_count + 1)) { b200_set_error("gemv_bs1: pair-mode row table too small"); return B200_ERR_FAILED; }
    if (pair) *pair = p.pair != 0;
    int rc;
    switch (mask) {
        case TB_Q4_K: rc = bs1_launch_t<TB_Q4_K>(ctx, p, (int)grid, smem_bytes); break;
        case TB_Q6_K: rc = bs1_launch_t<TB_Q6_K>(ctx, p, (int)grid, smem_bytes); break;
        case TB_Q5_K: rc = bs1_launch_t<TB_Q5_K>(ctx, p, (int)grid, smem_bytes); break;
        case TB_Q4_K | TB_Q6_K: rc = bs1_launch_t<TB_Q4_K | TB_Q6_K>(ctx, p, (int)grid, smem_bytes); break;
        default: rc = bs1_launch_t<TB_Q4_K | TB_Q5_K | TB_Q6_K>(ctx, p, (int)grid, smem_bytes); break;
    }
    return rc ? rc : 1;
}
