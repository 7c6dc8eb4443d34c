// gemv.cu -- decode GEMV (batch <= 4 per launch) over GGUF-layout quantised weights.
//
// Replaces mul_mat_vec_q (ggml-cuda/mmvq.cu:130-204: one row per 128-thread CTA, 2/4-byte loads, q8_1
// activations quantised by a separate kernel) with a B200 design:
//   * persistent CTAs, one per SM; a launch covers up to 3 weight matrices that share their activations
//     (wq|wk|wv, gate|up: "segments", possibly of different quantisation types).  CTA c owns a contiguous,
//     byte-balanced range of the concatenated rows, i.e. at most a few contiguous byte ranges of the weight
//     tensors (rows are stored back to back in GGUF);
//   * a dedicated producer warp streams those byte ranges into a deep shared-memory ring with 1-D bulk async
//     copies (cp.async.bulk + mbarrier complete_tx; SASS UBLKCP), L2 evict_first -- bytes in flight per SM
//     = ring size, independent of register pressure (Little: 6.5 TB/s x ~1 us => >= 44 KB/SM); once its own
//     range is queued it asks the L2 to fetch the NEXT matmul's weights (cp.async.bulk.prefetch.L2), so HBM
//     keeps streaming across the kernel boundary;
//   * every ring stage (1-4 whole rows) is OWNED by one consumer warp: it waits on that stage's mbarrier,
//     decodes the blocks straight out of shared memory in their file layout (gemv_items.cuh) with int8
//     dp4a block dots, shuffle-reduces, adds the optional residual, stores, releases the stage.  No
//     cross-warp synchronisation, and the result of a row does not depend on scheduling (bit-reproducible);
//   * the activation quantisation (q8_K / q8_0, bit-exact vs the CPU oracle) is fused into the prologue:
//     each CTA quantises the f32 activations itself while the producer is already streaming weights
//     (optionally after an on-the-fly rms_norm*weight or silu(gate)*up), so a matmul is ONE launch;
//   * MoE: the expert matrix of a segment can be chosen on the device (`expert_id`);
//   * programmatic dependent launch: weights are constants, so the producer starts before griddepcontrol.wait.
// Algorithmic bytes per launch: sum N*K*bpw (weights) + ncols*K*4 (f32 activations) + ncols*N*4 (output).
#include "common.cuh"
#include "gemv_items.cuh"
#include "quant_warp.cuh"
#include "gemv.h"

namespace {

using namespace gemv;

constexpr int MAX_STAGES = 48;

struct GemvSeg {
    const uint8_t *W;                 // row 0 of the weight matrix (of expert 0 for MUL_MAT_ID)
    uint32_t       rb;                // bytes per row
    int            type, N, rpw;      // rows per ring stage
    float *        dst;
    size_t         dst_stride;        // elements between columns
    const float *  residual;          // optional: dst = W.x + residual (same layout as dst)
    const int32_t *expert_id;         // MUL_MAT_ID: device pointer to the expert index (NULL: plain matmul)
    size_t         expert_stride;     // bytes between expert matrices (as->nb[2])
    int32_t *      dbgP, *dbgM;       // debug (block sums)
};

struct GemvParams {
    GemvSeg        seg[GEMV_MAX_SEG];
    int            nseg;
    int            K, q8k, act_mode;
    const uint8_t *act;               // ACT_PREQ: activation scratch (ActLayout), ncols columns
    ActLayout      L;
    const float *  x;                 // ACT_F32*: f32 activations, column stride x_stride bytes
    size_t         x_stride;
    const float *  x2;                // ACT_F32_NORM: norm weight [K]; ACT_F32_SWIGLU: `up` (same strides as x)
    float          eps;
    int            nstages;
    uint32_t       stage_bytes;
    int            w_const;           // weights are constant across launches (PDL may prefetch them early)
    int            use_pdl;
    // shared memory carve-up (bytes from the 128-aligned base); an aq offset of 0 means "layout not needed"
    uint32_t off_aq64, off_aq128, off_ad, off_as, off_ring;
    uint32_t aq64_col, aq128_col, ad_col, as_col;     // per-column sizes in smem: bytes / bytes / floats / int16
    const uint8_t *pf_ptr;            // L2 prefetch of the next launch's weights
    unsigned long long pf_bytes;
    unsigned long long *prof;         // optional [grid][16] globaltimer stamps (tools/gemv_prof.py)
};

// first global row (over the concatenated segments) of CTA c: ranges are balanced by BYTES, cut at row boundaries.
// 32-bit arithmetic in units of 16 bytes (64-bit divisions cost ~0.3 us each at kernel start); total < 64 GB.
__device__ __forceinline__ int split_row(const GemvParams &p, uint32_t share16, int total_rows, int c, int G) {
    if (c >= G) return total_rows;
    uint32_t target = share16 * (uint32_t)c;          // <= total bytes / 16
    int before = 0;
    for (int s = 0; s < p.nseg; s++) {
        const uint32_t rb16 = p.seg[s].rb >> 4 ? p.seg[s].rb >> 4 : 1;     // row bytes in 16-byte units (>= 1; exact for K-quants)
        const uint32_t sb = (uint32_t)p.seg[s].N * rb16;
        if (target < sb || s == p.nseg - 1) {
            const int r = (int)(target / rb16);
            return before + (r < p.seg[s].N ? r : p.seg[s].N);
        }
        target -= sb;
        before += p.seg[s].N;
    }
    return total_rows;
}

// ---- fused prologue: f32 activations -> quantised shared-memory layouts --------------------------------
__device__ __forceinline__ void store_act_q(const GemvParams &p, uint8_t *smem, int col, int e0, uint2 qp) {
    if (p.off_aq64)  *(uint2 *)(smem + p.off_aq64 + (size_t)col * p.aq64_col + (size_t)(e0 >> 6) * 80 + (e0 & 63)) = qp;
    if (p.off_aq128) *(uint2 *)(smem + p.off_aq128 + (size_t)col * p.aq128_col + (size_t)(e0 >> 7) * 144 + (e0 & 127)) = qp;
}

__device__ __forceinline__ void quantize_col_to_smem(const GemvParams &p, int col, uint8_t *smem, float *s_ad, int16_t *s_as,
                                                     int cwarp, int ncw, int lane, float norm_scale) {
    const float *xp = (const float *)((const char *)p.x + (size_t)col * p.x_stride);
    const float *up = p.act_mode == ACT_F32_SWIGLU ? (const float *)((const char *)p.x2 + (size_t)col * p.x_stride) : nullptr;
    const int nchunk = (p.K + 255) / 256;
    for (int b0 = cwarp; b0 < nchunk; b0 += 4 * ncw) {
        float4 ra[4][2], rb2[4][2];     // up to 4 chunks (x 2 operands) of loads in flight per warp
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int e0 = (b0 + u * ncw) * 256 + lane * 8;
            if (b0 + u * ncw < nchunk && e0 < p.K) {
                ra[u][0] = *(const float4 *)(xp + e0); ra[u][1] = *(const float4 *)(xp + e0 + 4);
                if (p.act_mode == ACT_F32_NORM) { rb2[u][0] = *(const float4 *)(p.x2 + e0); rb2[u][1] = *(const float4 *)(p.x2 + e0 + 4); }
                else if (p.act_mode == ACT_F32_SWIGLU) { rb2[u][0] = *(const float4 *)(up + e0); rb2[u][1] = *(const float4 *)(up + e0 + 4); }
            }
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int b = b0 + u * ncw;
            if (b >= nchunk) break;
            const int e0 = b * 256 + lane * 8;
            const bool valid = e0 < p.K;
            float v[8];
            if (valid) {
                v[0] = ra[u][0].x; v[1] = ra[u][0].y; v[2] = ra[u][0].z; v[3] = ra[u][0].w;
                v[4] = ra[u][1].x; v[5] = ra[u][1].y; v[6] = ra[u][1].z; v[7] = ra[u][1].w;
                if (p.act_mode == ACT_F32_NORM || p.act_mode == ACT_F32_SWIGLU) {
                    const float w[8] = {rb2[u][0].x, rb2[u][0].y, rb2[u][0].z, rb2[u][0].w, rb2[u][1].x, rb2[u][1].y, rb2[u][1].z, rb2[u][1].w};
                    if (p.act_mode == ACT_F32_NORM) {
#pragma unroll
                        for (int j = 0; j < 8; j++) v[j] = __fmul_rn(__fmul_rn(v[j], norm_scale), w[j]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 8; j++) v[j] = __fmul_rn(ggml_silu_lane(v[j]), w[j]);
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < 8; j++) v[j] = 0.0f;
            }
            uint2 qp;
            if (p.q8k) {
                float d; int pair;
                warp_quant_q8k(v, lane, qp, d, pair);
                if ((lane & 1) == 0) s_as[(size_t)col * p.as_col + b * 16 + (lane >> 1)] = (int16_t)pair;
                if (lane == 0) s_ad[(size_t)col * p.ad_col + b] = d;
            } else {
                float d16; int bsum;
                warp_quant_q80(v, qp, d16, bsum);
                if (valid && (lane & 3) == 0) {
                    s_ad[(size_t)col * p.ad_col + (e0 >> 5)] = d16;
                    s_as[(size_t)col * p.as_col + (e0 >> 5)] = (int16_t)bsum;
                }
            }
            if (valid) store_act_q(p, smem, col, e0, qp);
        }
    }
}

// ---- one ring stage = RPW rows of one segment, all NC columns -------------------------------------------
template <int TYPE, int NC, int RPW, bool DBG>
__device__ __forceinline__ void consume_chunk(const GemvParams &p, const GemvSeg &sg, const uint8_t *rowp, int row, int nr,
                                              const ActView &A, int lane, uint64_t *empty_bar) {
    const int nitems = num_items<TYPE>(p.K);
    float acc[RPW][NC];
#pragma unroll
    for (int r = 0; r < RPW; r++)
#pragma unroll
        for (int j = 0; j < NC; j++) acc[r][j] = 0.0f;
    DbgSink dbg[RPW];
    if (DBG) {
        const int nblk = p.K / Traits<TYPE>::BLOCK;
#pragma unroll
        for (int r = 0; r < RPW; r++) { dbg[r].P = sg.dbgP + (size_t)(row + r) * nblk; dbg[r].M = sg.dbgM + (size_t)(row + r) * nblk; }
    }
    constexpr bool TWO = (TYPE == T_Q4_K || TYPE == T_Q5_K) && RPW * NC <= 2;   // second item in flight only where registers allow
    for (int it = lane; it < nitems; it += TWO ? 64 : 32) {
        const bool two = TWO && it + 32 < nitems;
#pragma unroll
        for (int j = 0; j < NC; j++) {
            ActRegs<TYPE> ar0, ar1;
            load_act<TYPE>(A, j, it, ar0);
            if (two) load_act<TYPE>(A, j, it + 32, ar1);
#pragma unroll
            for (int r = 0; r < RPW; r++)
                if (r < nr) {
                    const DbgSink ds = j == 0 ? dbg[r] : DbgSink{nullptr, nullptr};
                    float v = item_dot<TYPE, DBG>(rowp + (size_t)r * sg.rb, it, p.K, ar0, ds);
                    if (two) v += item_dot<TYPE, DBG>(rowp + (size_t)r * sg.rb, it + 32, p.K, ar1, ds);
                    acc[r][j] += v;
                }
        }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty_bar);       // stage bytes are in registers/accumulated: release before reducing
#pragma unroll
    for (int r = 0; r < RPW; r++)
#pragma unroll
        for (int j = 0; j < NC; j++) acc[r][j] = warp_reduce_sum(acc[r][j]);
    if (lane == 0) {
#pragma unroll
        for (int r = 0; r < RPW; r++)
            if (r < nr) {
#pragma unroll
                for (int j = 0; j < NC; j++) {
                    const size_t o = (size_t)j * sg.dst_stride + row + r;
                    float v = acc[r][j];
                    if (sg.residual) v = __fadd_rn(v, sg.residual[o]);
                    sg.dst[o] = v;
                }
            }
    }
}

template <int TYPE, int NC, bool DBG>
__device__ __forceinline__ void consume_rpw(const GemvParams &p, const GemvSeg &sg, const uint8_t *rowp, int row, int nr, uint8_t *smem,
                                            const float *s_ad, const int16_t *s_as, int lane, uint64_t *empty_bar) {
    ActView A;
    constexpr bool L64 = Traits<TYPE>::ITEM == 64;
    A.q = (const int8_t *)(smem + (L64 ? p.off_aq64 : p.off_aq128));
    A.q_stride = L64 ? p.aq64_col : p.aq128_col;
    A.d = s_ad; A.s = s_as; A.d_stride = p.ad_col; A.s_stride = p.as_col;
    if constexpr (NC == 1) {
        if (sg.rpw == 4) { consume_chunk<TYPE, NC, 4, DBG>(p, sg, rowp, row, nr, A, lane, empty_bar); return; }
    }
    if constexpr (NC <= 2) {
        if (sg.rpw == 2) { consume_chunk<TYPE, NC, 2, DBG>(p, sg, rowp, row, nr, A, lane, empty_bar); return; }
    }
    consume_chunk<TYPE, NC, 1, DBG>(p, sg, rowp, row, nr, A, lane, empty_bar);
}

// TYPES: bit mask of the segment types this instantiation can meet (bit 0 Q4_K, 1 Q5_K, 2 Q6_K, 3 Q4_0, 4 Q8_0); single-type
// launches compile to straight-line code, mixed launches (wq|wk|wv of a K_M file) dispatch per ring stage.
constexpr int TM_Q4_K = 1, TM_Q5_K = 2, TM_Q6_K = 4, TM_Q4_0 = 8, TM_Q8_0 = 16;
constexpr int GEMV_THREADS = 640;
static_assert(GEMV_THREADS / 32 - 1 <= 32, "s_red holds one double per consumer warp");        // 19 consumer warps + 1 producer warp, one CTA per SM, <= 96 registers per thread

template <int TYPES, int NC, bool DBG>
__global__ void __launch_bounds__(GEMV_THREADS, 1) b200_gemv_kernel(const GemvParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *full  = (uint64_t *)smem;
    uint64_t *empty = full + MAX_STAGES;
    double *  s_red = (double *)(empty + MAX_STAGES);      // 32 doubles: rms_norm reduction, one per consumer warp
    volatile int *s_seq = (volatile int *)(s_red + 32);    // chunk index currently held by each stage
    float *   s_ad  = (float *)(smem + p.off_ad);
    int16_t * s_as  = (int16_t *)(smem + p.off_as);
    uint8_t * ring  = smem + p.off_ring;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ncw = (blockDim.x >> 5) - 1;                 // consumer warps; the last warp is the producer
#define PROF(slot) do { if (p.prof && lane == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); p.prof[(size_t)blockIdx.x * 16 + (slot)] = t_; } } while (0)
    if (warp == 0) PROF(0);
    const int G = gridDim.x, c = blockIdx.x;

    // ---- this CTA's share: per segment a row range [lo, hi) and its first chunk index (kept in shared memory: the hot
    //      loops need the registers) ------------------------------------------------------------------------------
    volatile int *s_lo = s_seq + MAX_STAGES, *s_hi = s_lo + GEMV_MAX_SEG, *s_ch0 = s_hi + GEMV_MAX_SEG;   // [3], [3], [4]
    if (threadIdx.x == 0) {
        uint32_t total16 = 0;
        int total_rows = 0;
        for (int s = 0; s < p.nseg; s++) { total16 += (uint32_t)p.seg[s].N * (p.seg[s].rb >> 4 ? p.seg[s].rb >> 4 : 1); total_rows += p.seg[s].N; }
        const uint32_t share16 = (total16 + (uint32_t)G - 1) / (uint32_t)G;
        const int g0 = split_row(p, share16, total_rows, c, G), g1 = split_row(p, share16, total_rows, c + 1, G);
        int base = 0, chunks = 0;
        for (int s = 0; s < GEMV_MAX_SEG; s++) {
            int a = 0, b = 0;
            s_ch0[s] = chunks;
            if (s < p.nseg) {
                a = max(g0, base) - base; b = min(g1, base + p.seg[s].N) - base;
                if (b > a) chunks += (b - a + p.seg[s].rpw - 1) / p.seg[s].rpw; else a = b = 0;
                base += p.seg[s].N;
            }
            s_lo[s] = a; s_hi[s] = b;
        }
        s_ch0[GEMV_MAX_SEG] = chunks;
    }
    if (threadIdx.x < p.nstages) { mbar_init(&full[threadIdx.x], 1); mbar_init(&empty[threadIdx.x], 1); }
    mbar_fence_init();
    __syncthreads();
    const int nchunks = s_ch0[GEMV_MAX_SEG];
    if (warp == 0) PROF(1);
    // Programmatic dependent launch: let the next kernel of the stream become resident right away (its producer streams
    // its constant weights, everything else blocks in griddepcontrol.wait until this grid has completed and flushed).
    if (p.use_pdl) pdl_trigger();

    if (warp == ncw) {
        // ------------------------------------------------------------------ producer
        // lanes issue the copies of `rw` consecutive chunks in parallel (a single thread tops out near 250 ns per
        // copy, i.e. ~5 TB/s chip-wide); rw <= nstages so no lane waits on a stage another lane of the same round fills
        bool waited = false;
        bool any_expert = false;
        for (int s = 0; s < p.nseg; s++) any_expert |= p.seg[s].expert_id != nullptr;
        if (p.use_pdl && (!p.w_const || any_expert)) { pdl_wait(); waited = true; }
        const uint64_t pol = l2_policy_evict_first();
        // Round r fills chunks [r*nstages, (r+1)*nstages); lane l always owns ring stages l and l+32.  A stage is therefore
        // re-armed by the SAME lane, in order, so the parity wait below can only refer to the immediately preceding use of
        // that stage (a lane that ran a full round ahead of a slow consumer would otherwise see the 1-bit phase alias and
        // overwrite a stage that is still being read).
        for (int base = 0; base < nchunks; base += p.nstages) {
            for (int st = lane; st < p.nstages; st += 32) {
                const int i = base + st;
                if (i >= nchunks) break;
                int s = 0;
#pragma unroll
                for (int t = 1; t < GEMV_MAX_SEG; t++) if (t < p.nseg && i >= s_ch0[t]) s = t;
                const GemvSeg &sg = p.seg[s];
                if (base > 0) mbar_wait(&empty[st], ((base / p.nstages) - 1) & 1);
                const int row = s_lo[s] + (i - s_ch0[s]) * sg.rpw;
                const int nr = min(sg.rpw, s_hi[s] - row);
                // MoE: the expert matrix is chosen on the device (no host round trip on `ids`, unlike ggml-cuda.cu:1976-1979)
                const uint8_t *Wb = sg.expert_id ? sg.W + (size_t)(*sg.expert_id) * sg.expert_stride : sg.W;
                const uint8_t *src = Wb + (size_t)row * sg.rb;
                const uint32_t extra = (uint32_t)((uintptr_t)src & 15);
                const uint32_t bytes = (extra + (uint32_t)nr * sg.rb + 15u) & ~15u;
                s_seq[st] = i;                                   // published by the release of the arrive below
                mbar_arrive_expect_tx(&full[st], bytes);
                bulk_g2s_hint(ring + (size_t)st * p.stage_bytes, src - extra, bytes, &full[st], pol);
            }
            __syncwarp();
            if (base == 0) {
                PROF(2);
                // weights of the NEXT matmul: ask the L2 to start fetching this CTA's 1/G of them now
                if (p.pf_bytes) {
                    const unsigned long long per = ((p.pf_bytes / G) + 15ull) & ~15ull;
                    const unsigned long long b0 = per * c;
                    const unsigned long long lim = p.pf_bytes & ~15ull;
                    const unsigned long long b1 = b0 + per < lim ? b0 + per : lim;
                    constexpr unsigned long long PIECE = 8192;
                    for (unsigned long long o = b0 + (unsigned long long)lane * PIECE; o < b1; o += 32 * PIECE) {
                        const uint32_t n = (uint32_t)(b1 - o < PIECE ? b1 - o : PIECE);
                        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p.pf_ptr + o), "r"(n) : "memory");
                    }
                }
            }
        }
        PROF(3);
        if (p.use_pdl && !waited) pdl_wait();      // every thread orders itself after the previous grid before exiting
        return;
    }

    // ---------------------------------------------------------------------- consumers: prologue
    if (p.use_pdl) pdl_wait();     // activations (and the memory we are about to overwrite) belong to the previous kernels
    if (nchunks == 0) return;
    const int nct = ncw * 32;
    if (p.act_mode == ACT_PREQ) {
        const int tid = threadIdx.x;
        const int nvec = p.K / 8;
        for (int col = 0; col < NC; col++) {
            const uint8_t *g = p.act + (size_t)col * p.L.col_bytes;
            for (int v = tid; v < nvec; v += nct) store_act_q(p, smem, col, v * 8, *(const uint2 *)(g + v * 8));
            const int nd = p.K / (p.q8k ? 256 : 32), ns = p.K / (p.q8k ? 16 : 32);
            for (int i = tid; i < nd; i += nct) s_ad[(size_t)col * p.ad_col + i] = ((const float *)(g + p.L.off_d))[i];
            for (int i = tid; i < ns; i += nct) s_as[(size_t)col * p.as_col + i] = ((const int16_t *)(g + p.L.off_sums))[i];
        }
    } else {
        for (int col = 0; col < NC; col++) {
            float norm_scale = 1.0f;
            if (p.act_mode == ACT_F32_NORM) {
                // rms_norm exactly as glue.cu / the CPU oracle: sum of squares in double, fixed reduction order
                const float *xp = (const float *)((const char *)p.x + (size_t)col * p.x_stride);
                double s = 0.0;
                for (int i = threadIdx.x; i < p.K; i += nct) { const float v = xp[i]; s += (double)__fmul_rn(v, v); }
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                double *sd = s_red;
                named_bar_sync(1, nct);
                if (lane == 0) sd[warp] = s;
                named_bar_sync(1, nct);
                double t = 0.0;
                for (int i = 0; i < ncw; i++) t += sd[i];
                const float mean = (float)(t / (double)p.K);
                norm_scale = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(mean, p.eps)));
            }
            quantize_col_to_smem(p, col, smem, s_ad, s_as, warp, ncw, lane, norm_scale);
        }
    }
    if (warp == 0) PROF(4);
    named_bar_sync(1, nct);
    if (warp == 0) PROF(5);

    // ---------------------------------------------------------------------- consumers: main loop
    for (int i = warp; i < nchunks; i += ncw) {
        int s = 0;
#pragma unroll
        for (int t = 1; t < GEMV_MAX_SEG; t++) if (t < p.nseg && i >= s_ch0[t]) s = t;
        const GemvSeg &sg = p.seg[s];
        const int st = i % p.nstages;
        const int row = s_lo[s] + (i - s_ch0[s]) * sg.rpw;
        const int nr = min(sg.rpw, s_hi[s] - row);
        // A warp that runs far ahead of the owner of this slot's previous use could be fooled by the 1-bit phase
        // parity (use u and u+2 look alike); the stage's sequence number disambiguates.
        do { mbar_wait(&full[st], (i / p.nstages) & 1); } while (s_seq[st] != i);
        if (i == 0) PROF(6);
        const uint8_t *Wb = sg.expert_id ? sg.W + (size_t)(*sg.expert_id) * sg.expert_stride : sg.W;
        const uint32_t extra = (uint32_t)((uintptr_t)(Wb + (size_t)row * sg.rb) & 15);
        const uint8_t *rowp = ring + (size_t)st * p.stage_bytes + extra;
        const int ty = sg.type;
        if ((TYPES & TM_Q4_K) && (TYPES == TM_Q4_K || ty == T_Q4_K)) consume_rpw<T_Q4_K, NC, DBG>(p, sg, rowp, row, nr, smem, s_ad, s_as, lane, &empty[st]);
        else if ((TYPES & TM_Q5_K) && (TYPES == TM_Q5_K || ty == T_Q5_K)) consume_rpw<T_Q5_K, NC, DBG>(p, sg, rowp, row, nr, smem, s_ad, s_as, lane, &empty[st]);
        else if ((TYPES & TM_Q6_K) && (TYPES == TM_Q6_K || ty == T_Q6_K)) consume_rpw<T_Q6_K, NC, DBG>(p, sg, rowp, row, nr, smem, s_ad, s_as, lane, &empty[st]);
        else if ((TYPES & TM_Q4_0) && (TYPES == TM_Q4_0 || ty == T_Q4_0)) consume_rpw<T_Q4_0, NC, DBG>(p, sg, rowp, row, nr, smem, s_ad, s_as, lane, &empty[st]);
        else if (TYPES & TM_Q8_0) consume_rpw<T_Q8_0, NC, DBG>(p, sg, rowp, row, nr, smem, s_ad, s_as, lane, &empty[st]);
        if (i == 0) PROF(7);
        if (i + ncw >= nchunks && warp == (nchunks - 1) % ncw) PROF(8);
    }
#undef PROF
}

bool item64(int type) { return type == B200_TYPE_Q4_K || type == B200_TYPE_Q5_K; }

int g_gemv_warps = 0, g_gemv_stage_kb = 0, g_gemv_smem_kb = 0, g_gemv_ctas = 0, g_gemv_l2pf = -1;     // tuning overrides (env GGML_B200_GEMV_*)

// rows per stage for a given column count: keep a stage around 8-12 KB so the ring holds >= 16 stages
int choose_rpw(uint32_t rb, int ncols, int64_t rows_per_cta, int nwarps) {
    const uint32_t target = (uint32_t)(g_gemv_stage_kb > 0 ? g_gemv_stage_kb : 10) * 1024;
    const int maxr = ncols == 1 ? 4 : (ncols == 2 ? 2 : 1);
    int r = maxr;
    // small stages when a CTA owns few rows (every consumer warp should get >= 2 chunks), bounded stage bytes otherwise
    while (r > 1 && ((size_t)r * rb > target || rows_per_cta / r < 2 * nwarps)) r >>= 1;
    return r;
}

// stage geometry + smem carve-up for `ncols` columns; false if it does not fit.  p.seg[].type/rb/rpw and p.q8k must be set.
bool plan(const b200_ctx *ctx, int64_t K, int ncols, GemvParams &p, size_t &smem_bytes) {
    bool need64 = false, need128 = false;
    uint32_t max_stage = 0;
    for (int s = 0; s < p.nseg; s++) {
        if (item64(p.seg[s].type)) need64 = true; else need128 = true;
        const uint32_t sb = (uint32_t)(((size_t)p.seg[s].rpw * p.seg[s].rb + 32 + 127) & ~(size_t)127);   // +16 misalignment, +16 over-read
        if (sb > max_stage) max_stage = sb;
    }
    const int q8k = p.q8k;
    p.aq64_col = (uint32_t)(((K + 63) / 64) * 80);
    p.aq128_col = (uint32_t)(((K + 127) / 128) * 144);
    p.ad_col = (uint32_t)(((K / (q8k ? 256 : 32)) + 4 + 3) & ~3);
    p.as_col = (uint32_t)(((K / (q8k ? 16 : 32)) + 8 + 7) & ~7);
    uint32_t off = 2 * MAX_STAGES * 8 + 256 + MAX_STAGES * 4 + 64;      // barriers, s_red, s_seq, s_lo/s_hi/s_ch0
    off = (off + 15) & ~15u;
    p.off_aq64 = 0; p.off_aq128 = 0;
    if (need64)  { p.off_aq64 = off;  off += p.aq64_col * ncols;  off = (off + 15) & ~15u; }
    if (need128) { p.off_aq128 = off; off += p.aq128_col * ncols; off = (off + 15) & ~15u; }
    p.off_ad = off;   off += p.ad_col * 4 * ncols;
    off = (off + 15) & ~15u;
    p.off_as = off;   off += p.as_col * 2 * ncols;
    off = (off + 127) & ~127u;
    p.off_ring = off;
    size_t budget = g_gemv_smem_kb > 0 ? (size_t)g_gemv_smem_kb * 1024 : ctx->smem_optin;
    if (budget > ctx->smem_optin) budget = ctx->smem_optin;
    if ((size_t)off + 1024 > budget) return false;
    const size_t ring_budget = budget - off;
    int ns = (int)(ring_budget / max_stage);
    if (ns < 2) return false;
    if (ns > MAX_STAGES) ns = MAX_STAGES;
    p.nstages = ns; p.stage_bytes = max_stage;
    smem_bytes = off + (size_t)ns * max_stage;
    return true;
}

template <int TYPES, int NC, bool DBG>
int launch_t(b200_ctx *ctx, const GemvParams &p, int grid, int nwarps, size_t smem_bytes) {
    auto kern = b200_gemv_kernel<TYPES, NC, DBG>;
    static bool attr_set[16] = {false};   // per device
    if (!attr_set[ctx->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->smem_optin));
        attr_set[ctx->device & 15] = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)(nwarps + 1) * 32);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    int nattr = 0;
    if (p.use_pdl) {
        attr[nattr].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[nattr].val.programmaticStreamSerializationAllowed = 1;
        nattr++;
    }
    cfg.attrs = attr;
    cfg.numAttrs = nattr;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, p));
    ctx->launches++;
    return B200_OK;
}

template <int TYPES>
int launch_cols(b200_ctx *ctx, const GemvParams &p, int ncols, bool dbg, int grid, int nwarps, size_t smem) {
    if (dbg) {
        if constexpr (TYPES == TM_Q4_K || TYPES == TM_Q5_K || TYPES == TM_Q6_K || TYPES == TM_Q4_0 || TYPES == TM_Q8_0)
            if (ncols == 1) return launch_t<TYPES, 1, true>(ctx, p, grid, nwarps, smem);
        return B200_ERR_UNSUPPORTED;
    }
    switch (ncols) {
        case 1: return launch_t<TYPES, 1, false>(ctx, p, grid, nwarps, smem);
        case 2: return launch_t<TYPES, 2, false>(ctx, p, grid, nwarps, smem);
        case 3: return launch_t<TYPES, 3, false>(ctx, p, grid, nwarps, smem);
        case 4: return launch_t<TYPES, 4, false>(ctx, p, grid, nwarps, smem);
    }
    b200_set_error("gemv: ncols=%d", ncols);
    return B200_ERR_UNSUPPORTED;
}

int type_bit(int type) {
    switch (type) {
        case B200_TYPE_Q4_K: return TM_Q4_K; case B200_TYPE_Q5_K: return TM_Q5_K; case B200_TYPE_Q6_K: return TM_Q6_K;
        case B200_TYPE_Q4_0: return TM_Q4_0; default: return TM_Q8_0;
    }
}

int launch_mask(b200_ctx *ctx, const GemvParams &p, int ncols, bool dbg, int grid, int nwarps, size_t smem) {
    int mask = 0;
    for (int s = 0; s < p.nseg; s++) mask |= type_bit(p.seg[s].type);
    switch (mask) {
        case TM_Q4_K: return launch_cols<TM_Q4_K>(ctx, p, ncols, dbg, grid, nwarps, smem);
        case TM_Q5_K: return launch_cols<TM_Q5_K>(ctx, p, ncols, dbg, grid, nwarps, smem);
        case TM_Q6_K: return launch_cols<TM_Q6_K>(ctx, p, ncols, dbg, grid, nwarps, smem);
        case TM_Q4_0: return launch_cols<TM_Q4_0>(ctx, p, ncols, dbg, grid, nwarps, smem);
        case TM_Q8_0: return launch_cols<TM_Q8_0>(ctx, p, ncols, dbg, grid, nwarps, smem);
        case TM_Q4_K | TM_Q6_K: return launch_cols<TM_Q4_K | TM_Q6_K>(ctx, p, ncols, dbg, grid, nwarps, smem);
        case TM_Q4_0 | TM_Q8_0: return launch_cols<TM_Q4_0 | TM_Q8_0>(ctx, p, ncols, dbg, grid, nwarps, smem);
        default:
            if (mask & (TM_Q4_0 | TM_Q8_0)) { b200_set_error("gemv: type mix %d", mask); return B200_ERR_UNSUPPORTED; }
            return launch_cols<TM_Q4_K | TM_Q5_K | TM_Q6_K>(ctx, p, ncols, dbg, grid, nwarps, smem);
    }
}

void read_env() {
    static bool env_read = false;
    if (env_read) return;
    if (const char *e = getenv("GGML_B200_GEMV_WARPS")) g_gemv_warps = atoi(e);
    if (const char *e = getenv("GGML_B200_GEMV_STAGE_KB")) g_gemv_stage_kb = atoi(e);
    if (const char *e = getenv("GGML_B200_GEMV_SMEM_KB")) g_gemv_smem_kb = atoi(e);
    if (const char *e = getenv("GGML_B200_GEMV_CTAS")) g_gemv_ctas = atoi(e);
    if (const char *e = getenv("GGML_B200_L2_PREFETCH")) g_gemv_l2pf = atoi(e);
    env_read = true;
}

}  // namespace

int gemv_max_cols(const b200_ctx *ctx, int type, size_t rb, int64_t K) {
    GemvParams p = {};
    size_t smem;
    p.nseg = 1; p.seg[0].type = type; p.seg[0].rb = (uint32_t)rb; p.seg[0].rpw = 1; p.q8k = b200_act_mode_q8k(type);
    for (int nc = 4; nc >= 1; nc--) if (plan(ctx, K, nc, p, smem)) return nc;
    return 0;
}

// General entry: up to GEMV_MAX_SEG weight matrices that share K and the activation columns.
int gemv_launch(b200_ctx *ctx, const GemvSegDesc *segs, int nseg, int64_t K, const GemvActDesc &ga, int ncols, bool w_const,
                const GemvPf *pf, int npf, bool *pair) {
    if (pair && ncols != 1) { *pair = false; pair = nullptr; }
    const void *pf_ptr = pf && npf > 0 ? pf[0].ptr : nullptr;
    const size_t pf_bytes = pf && npf > 0 ? pf[0].bytes : 0;
    if (nseg <= 0 || nseg > GEMV_MAX_SEG || ncols <= 0) return B200_OK;
    read_env();
    const int q8k = b200_act_mode_q8k(segs[0].type);
    int64_t total_rows = 0;
    for (int s = 0; s < nseg; s++) {
        if (!b200_type_is_quant(segs[s].type) || b200_act_mode_q8k(segs[s].type) != q8k) { b200_set_error("gemv: segment types do not share an activation format"); return B200_ERR_UNSUPPORTED; }
        if (item64(segs[s].type) && (((uintptr_t)segs[s].W & 15) || (segs[s].rb & 15) || (segs[s].expert_stride & 15))) {
            b200_set_error("gemv: K-quant rows must be 16-byte aligned");
            return B200_ERR_UNSUPPORTED;
        }
        total_rows += segs[s].N;
    }
    if (total_rows <= 0) return B200_OK;
    if (ncols > 4) {
        // continuous-batching step (5..32 token columns): one producer launch quantises the activations, then every segment streams
        // its weights once through the mma.sync kernel (gemv_mma.cu); the residual is added by its epilogue / split-K reduction
        bool ok = ncols <= 32;
        for (int s = 0; s < nseg; s++) ok = ok && gemv_mma_supported(segs[s].type, segs[s].N, K, ncols) && !segs[s].expert_id && !segs[s].dbgP;
        if (ok) {
            const ActLayout Lb = ActLayout::make(q8k, K);
            const uint8_t *act = ga.act;
            if (ga.mode != ACT_PREQ) {
                uint8_t *scr = (uint8_t *)ctx->get_scratch(SCRATCH_ACT, Lb.col_bytes * (size_t)ncols);
                if (!scr) return B200_ERR_ALLOC;
                int rc = launch_act_prologue(ctx, ga.mode, ga.x, ga.x_stride, ga.x2, ga.eps, K, ncols, q8k, scr);
                if (rc) return rc;
                act = scr;
            }
            for (int s = 0; s < nseg; s++) {
                int rc = launch_gemv_mma(ctx, segs[s].type, segs[s].W, segs[s].rb, segs[s].N, K, act, ncols, segs[s].dst, segs[s].dst_stride, true, w_const,
                                         segs[s].residual);
                if (rc) return rc;
            }
            return B200_OK;
        }
    }
    if (ncols == 1) {
        // batch-1 decode over K-quants: the compact half-SM kernel (gemv_bs1.cu); anything it does not take falls through
        const int l2pf = g_gemv_l2pf >= 0 ? g_gemv_l2pf : ctx->opt_l2_prefetch;
        const int rc = gemv_bs1_try_launch(ctx, segs, nseg, K, ga, w_const, pf, npf, l2pf, pair);
        if (rc != 0) return rc < 0 ? rc : B200_OK;
        if (pair) *pair = false;
    }
    const ActLayout L = ActLayout::make(q8k, K);
    constexpr int MAXW = GEMV_THREADS / 32 - 1;
    const int nwarps = g_gemv_warps > 0 ? (g_gemv_warps > MAXW ? MAXW : g_gemv_warps) : MAXW;
    // one persistent CTA per SM: 19 consumer warps hide the shared-memory / dp4a latency of the block decoders
    const int ctas_per_sm = 1;
    const bool dbg = segs[0].dbgP != nullptr;
    GemvParams p = {};
    size_t smem = 0;
    for (int c0 = 0; c0 < ncols;) {
        int nc = ncols - c0 < 4 ? ncols - c0 : 4;
        // geometry for this column count (shrinks nc until the activations fit shared memory)
        for (;; nc--) {
            if (nc == 0) { b200_set_error("gemv: K=%lld does not fit shared memory", (long long)K); return B200_ERR_UNSUPPORTED; }
            p = GemvParams();
            p.nseg = nseg; p.q8k = q8k;
            for (int s = 0; s < nseg; s++) {
                GemvSeg &g = p.seg[s];
                g.W = segs[s].W; g.rb = (uint32_t)segs[s].rb; g.type = segs[s].type; g.N = (int)segs[s].N;
                g.rpw = choose_rpw(g.rb, nc, total_rows / ((int64_t)ctx->sm_count * ctas_per_sm), nwarps);
                g.dst = segs[s].dst + (size_t)c0 * segs[s].dst_stride; g.dst_stride = segs[s].dst_stride;
                g.residual = segs[s].residual ? segs[s].residual + (size_t)c0 * segs[s].dst_stride : nullptr;
                g.expert_id = segs[s].expert_id; g.expert_stride = segs[s].expert_stride;
                g.dbgP = segs[s].dbgP; g.dbgM = segs[s].dbgM;
            }
            if (plan(ctx, K, nc, p, smem)) break;
        }
        const int cps = ctas_per_sm;
        p.K = (int)K;
        p.act_mode = ga.mode;
        p.act = ga.act ? ga.act + (size_t)c0 * L.col_bytes : nullptr;
        p.L = L;
        p.x = ga.x ? (const float *)((const char *)ga.x + (size_t)c0 * ga.x_stride) : nullptr;
        p.x_stride = ga.x_stride;
        p.x2 = ga.mode == ACT_F32_SWIGLU && ga.x2 ? (const float *)((const char *)ga.x2 + (size_t)c0 * ga.x_stride) : ga.x2;
        p.eps = ga.eps;
        p.w_const = w_const ? 1 : 0;
        p.use_pdl = ctx->opt_pdl;
        const bool last = c0 + nc >= ncols;
        const int l2pf = g_gemv_l2pf >= 0 ? g_gemv_l2pf : ctx->opt_l2_prefetch;
        if (last && l2pf && pf_ptr && pf_bytes) {
            p.pf_ptr = (const uint8_t *)pf_ptr;
            p.pf_bytes = pf_bytes < ((size_t)48 << 20) ? pf_bytes : ((size_t)48 << 20);
            const uintptr_t mis = (uintptr_t)p.pf_ptr & 15;
            if (mis) { p.pf_ptr += 16 - mis; p.pf_bytes = p.pf_bytes > 16 ? p.pf_bytes - 16 : 0; }
        }
        p.prof = (unsigned long long *)ctx->prof_buf;
        int64_t min_chunks = 0;
        for (int s = 0; s < nseg; s++) min_chunks += (segs[s].N + p.seg[s].rpw - 1) / p.seg[s].rpw;
        const int64_t maxg = (int64_t)ctx->sm_count * cps;
        const int grid = (int)(min_chunks < maxg ? min_chunks : maxg);
        int rc = launch_mask(ctx, p, nc, dbg, grid, nwarps, smem);
        if (rc) return rc;
        c0 += nc;
    }
    return B200_OK;
}

int launch_gemv(b200_ctx *ctx, int type, const uint8_t *W, size_t row_bytes, int64_t N, int64_t K, const uint8_t *act, int ncols,
                float *dst, size_t dst_col_stride, bool w_const) {
    GemvSegDesc sg = {};
    sg.type = type; sg.W = W; sg.rb = row_bytes; sg.N = N; sg.dst = dst; sg.dst_stride = dst_col_stride;
    GemvActDesc ga = {};
    ga.mode = ACT_PREQ; ga.act = act;
    return gemv_launch(ctx, &sg, 1, K, ga, ncols, w_const, nullptr, 0);
}

// fused: dst = W . quant(f(x)) (+ residual); fuse_mode 0: f = id, 1: f = rms_norm(x)*x2, 2: f = silu(x)*x2
int launch_gemv_f32(b200_ctx *ctx, int type, const uint8_t *W, size_t row_bytes, int64_t N, int64_t K, const float *x, size_t x_stride_bytes,
                    int ncols, float *dst, size_t dst_col_stride, bool w_const, int fuse_mode, const float *x2, float eps,
                    const float *residual) {
    GemvSegDesc sg = {};
    sg.type = type; sg.W = W; sg.rb = row_bytes; sg.N = N; sg.dst = dst; sg.dst_stride = dst_col_stride; sg.residual = residual;
    GemvActDesc ga = {};
    ga.mode = fuse_mode == 1 ? ACT_F32_NORM : fuse_mode == 2 ? ACT_F32_SWIGLU : ACT_F32;
    ga.x = x; ga.x_stride = x_stride_bytes; ga.x2 = x2; ga.eps = eps;
    return gemv_launch(ctx, &sg, 1, K, ga, ncols, w_const, nullptr, 0);
}

// MUL_MAT_ID building block: dst[N] = W[*expert_id] . quant(x), one column, expert chosen on the device
int launch_gemv_expert(b200_ctx *ctx, int type, const uint8_t *W, size_t row_bytes, size_t expert_stride, const int32_t *expert_id, int64_t N,
                       int64_t K, const float *x, float *dst) {
    GemvSegDesc sg = {};
    sg.type = type; sg.W = W; sg.rb = row_bytes; sg.N = N; sg.dst = dst; sg.dst_stride = (size_t)N;
    sg.expert_id = expert_id; sg.expert_stride = expert_stride;
    GemvActDesc ga = {};
    ga.mode = ACT_F32; ga.x = x; ga.x_stride = (size_t)K * 4;
    return gemv_launch(ctx, &sg, 1, K, ga, 1, true, nullptr, 0);
}

// test hook: exact integer block sums computed by the SAME item decoders through the SAME pipeline
extern "C" int b200_block_sums(b200_ctx *ctx, int32_t type, const void *W, const float *x, int64_t N, int64_t K, int32_t *P, int32_t *M) {
    if (!ctx || !b200_type_is_quant(type)) { b200_set_error("block_sums: type %d", type); return B200_ERR_UNSUPPORTED; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int64_t nblk = K / b200_type_block_elems(type);
    float *dummy = (float *)ctx->get_scratch(SCRATCH_MISC, (size_t)N * 4);
    if (!dummy) return B200_ERR_ALLOC;
    CUDA_TRY(cudaMemsetAsync(P, 0, (size_t)N * nblk * 4, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(M, 0, (size_t)N * nblk * 4, ctx->stream));
    GemvSegDesc sg = {};
    sg.type = type; sg.W = (const uint8_t *)W; sg.rb = b200_row_bytes(type, K); sg.N = N; sg.dst = dummy; sg.dst_stride = (size_t)N;
    sg.dbgP = P; sg.dbgM = M;
    GemvActDesc ga = {};
    ga.mode = ACT_F32; ga.x = x; ga.x_stride = (size_t)K * 4;
    return gemv_launch(ctx, &sg, 1, K, ga, 1, false, nullptr, 0);
}
