// gemv_f16.cu -- F16/BF16 weight matmul for 1..32 token columns (bs1 decode up to continuous-batching steps): a weight-streaming
// problem (every weight byte is used by at most 32 columns), built like gemv_mma.cu:
//   * unit of work = 128 weight rows x one K slice; CTA (g, r) keeps the x columns of K slice r resident in shared memory, rounded to
//     the weight's 16-bit type (the CPU's vec_dot_type: f16 or bf16, round-to-nearest-even) and walks the 128-row blocks of group g;
//     several K slices are combined by a fixed-order reduction (split-K), so results are bit-reproducible;
//   * a producer warp streams the rows through a shared-memory ring, one 2-D TMA tile of 128 rows x 64 k (16 KB) per stage,
//     SWIZZLE_128B (ldmatrix conflict-free), completing on the stage's mbarrier; the tensor map's zero fill covers the K and N tails.
//     Weights (B200_TENSOR_FLAG_WEIGHT) are requested before griddepcontrol.wait, so the previous kernel's tail overlaps them;
//   * 8 consumer warps own 16 rows each and multiply them into all token columns with mma.sync m16n8k16 (.f16 / .bf16, f32
//     accumulate): the weight rows are M, the token columns N (8 per n-tile).  Products of two 16-bit floats are exact in f32, so
//     the result differs from the CPU only in the order of the f32 additions.
// Grouped mode (MUL_MAT_ID, b200_gemv_f16_grouped_kernel): blockIdx.y = a chunk of <= 32 (token, slot) pairs of one expert from the
// device-side routing tables; the chunk's x columns are gathered into the slice and the expert's rows streamed through a 3-D TMA map.
// Roofline: HBM; algorithmic bytes = 2 N K + 4 M (K + N).
#include "float_mm.h"
#include "tc05.cuh"
#include <cuda_bf16.h>
#include <algorithm>

namespace {

constexpr int GF_ROWS = 128;                     // rows per block (8 consumer warps x the mma M of 16)
constexpr int GF_KS = 64;                        // k per stage: one 128-byte swizzle row
constexpr uint32_t GF_STAGE = GF_ROWS * GF_KS * 2;      // 16 KB
constexpr int GF_CONS = 8;
constexpr int GF_THREADS = (GF_CONS + 1) * 32;
constexpr int GF_MAX_STAGES = 12;
constexpr uint32_t GF_X_BYTES = 64 * 1024;      // resident x slice: (8 * NT) columns x slice k x 2 bytes

struct GfParams {
    const float *x; size_t x_stride;             // floats between columns
    int N, K, ncols;
    float *dst; size_t dst_stride;
    float *part;                                 // [nslices][ncols][N] when nslices > 1
    int nslices, ngroups, nblocks, kslice, nstages;
    uint32_t xpitch, off_x, off_bar;
    int use_pdl, w_const;
};
// grouped (MUL_MAT_ID) mode: blockIdx.y = chunk of <= 32 (token, slot) pairs of one expert; part = [nslices][npairs][N] in sorted order.
// A second kernel argument: a larger GfParams would change how the dense kernel loads its parameters.
struct GfGroup {
    const int32_t *off, *pairs; int E, n_used, b_ne1, npairs; size_t d_nb1, d_nb2;
};

// grouped mode: chunk -> (expert, first sorted pair, pairs in the chunk); cnt = 0: the chunk does not exist (fewer than the upper bound)
__device__ __forceinline__ void gf_chunk(const GfGroup &g, int chunk, int &e, int &first, int &cnt) {
    cnt = 0; first = 0;
    for (e = 0; e < g.E; e++) {
        const int o0 = g.off[e], n = g.off[e + 1] - o0, nch = (n + 31) / 32;
        if (chunk < nch) { first = o0 + chunk * 32; cnt = min(32, n - chunk * 32); return; }
        chunk -= nch;
    }
}

__device__ __forceinline__ void ldsm_x4(uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3, uint32_t saddr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(saddr));
}
__device__ __forceinline__ void ldsm_x2(uint32_t &r0, uint32_t &r1, uint32_t saddr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(saddr));
}
template <bool BF>
__device__ __forceinline__ void mma_k16(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    if (BF)
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
    else
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// two floats -> two 16-bit values (round-to-nearest-even), low half first
template <bool BF> __device__ __forceinline__ uint32_t pack2(float a, float b) {
    if (BF) { __nv_bfloat162 h = __floats2bfloat162_rn(a, b); return *(uint32_t *)&h; }
    __half2 h = __floats2half2_rn(a, b);
    return *(uint32_t *)&h;
}

template <bool BF, int NT>
__global__ void __launch_bounds__(GF_THREADS, 1) b200_gemv_f16_kernel(const __grid_constant__ CUtensorMap tmw, const GfParams p) {
    extern __shared__ uint8_t gf_smem_raw[];
    uint8_t *smem = gf_smem_raw + ((1024u - (smem_u32(gf_smem_raw) & 1023u)) & 1023u);      // SWIZZLE_128B destinations: 1024-byte aligned
    uint8_t *ring = smem;
    uint8_t *xs = smem + p.off_x;
    uint64_t *full = (uint64_t *)(smem + p.off_bar), *empty = full + GF_MAX_STAGES;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ns = p.nstages;
    if (p.use_pdl) pdl_trigger();
    const int r = blockIdx.x % p.nslices, g = blockIdx.x / p.nslices;
    const int b0 = (int)((long long)p.nblocks * g / p.ngroups), b1 = (int)((long long)p.nblocks * (g + 1) / p.ngroups);
    const int k0 = r * p.kslice;
    const int nst = (min(p.kslice, p.K - k0) + GF_KS - 1) / GF_KS;          // stages per block
    const int nunits = (b1 - b0) * nst;
    if (threadIdx.x == 0) {
        for (int i = 0; i < ns; i++) { mbar_init(&full[i], 1); mbar_init(&empty[i], GF_CONS); }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == GF_CONS) {
        // ------------------------------------------------------------ producer: one TMA tile per stage
        if (p.use_pdl && !p.w_const) pdl_wait();          // src0 written earlier in the same graph: no early streaming
        for (int u = 0; u < nunits; u++) {
            const int st = u % ns, use = u / ns;
            if (use > 0) mbar_wait_bounded(&empty[st], (use - 1) & 1);
            if (elect_one_sync()) {
                mbar_arrive_expect_tx(&full[st], GF_STAGE);
                tma_load_2d(ring + (size_t)st * GF_STAGE, &tmw, k0 + (u % nst) * GF_KS, (b0 + u / nst) * GF_ROWS, &full[st]);
            }
            __syncwarp();
        }
        return;
    }
    // ---------------------------------------------------------------- consumers: x slice -> shared memory, rounded once
    if (p.use_pdl) pdl_wait();
    {
        const int q4 = p.kslice / 4;                      // float4 groups per column
        for (int i = threadIdx.x; i < NT * 8 * q4; i += GF_CONS * 32) {
            const int col = i / q4, k = k0 + (i % q4) * 4;
            float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            if (col < p.ncols && k < p.K) v = *(const float4 *)(p.x + (size_t)col * p.x_stride + k);      // K % 8 == 0: whole float4
            *(uint2 *)(xs + (size_t)col * p.xpitch + (size_t)(i % q4) * 8) = make_uint2(pack2<BF>(v.x, v.y), pack2<BF>(v.z, v.w));
        }
    }
    named_bar_sync(1, GF_CONS * 32);
    const uint32_t xs_saddr = smem_u32(xs), ring_saddr = smem_u32(ring);
    // ldmatrix lanes: A row (l & 7) + 8 ((l >> 3) & 1) of this warp's 16, 16-byte chunk (l >> 4) of the k16 step; B row l & 7 of n-tile
    const int arow = (lane & 7) + ((lane >> 3) & 1) * 8, achunk = lane >> 4;
    const uint32_t a_off = (uint32_t)(warp * 16 + arow) * 128u;
    const int mi = lane >> 3, rr = lane & 7;
    int u = 0;
    for (int blk = b0; blk < b1; blk++) {
        float acc[NT][4];
#pragma unroll
        for (int nt = 0; nt < NT; nt++) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.0f;
        for (int s = 0; s < nst; s++, u++) {
            const int st = u % ns, use = u / ns;
            mbar_wait_bounded(&full[st], use & 1);
            const uint32_t tile = ring_saddr + (uint32_t)st * GF_STAGE + a_off;
#pragma unroll
            for (int ks = 0; ks < GF_KS / 16; ks++) {
                uint32_t a0, a1, a2, a3;
                ldsm_x4(a0, a1, a2, a3, tile + (uint32_t)(((2 * ks + achunk) ^ (arow & 7)) * 16));
                const uint32_t kb = (uint32_t)(s * GF_KS + ks * 16) * 2u;
                uint32_t b[NT][2];
                if (NT == 1) {
                    ldsm_x2(b[0][0], b[0][1], xs_saddr + (uint32_t)rr * p.xpitch + kb + (uint32_t)(mi & 1) * 16);
                } else {
#pragma unroll
                    for (int n2 = 0; n2 < NT / 2; n2++)
                        ldsm_x4(b[2 * n2][0], b[2 * n2][1], b[2 * n2 + (NT > 1)][0], b[2 * n2 + (NT > 1)][1],
                                xs_saddr + (uint32_t)((2 * n2 + (mi >> 1)) * 8 + rr) * p.xpitch + kb + (uint32_t)(mi & 1) * 16);
                }
#pragma unroll
                for (int nt = 0; nt < NT; nt++) mma_k16<BF>(acc[nt], a0, a1, a2, a3, b[nt][0], b[nt][1]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[st]);
        }
        // ---- store: rows R, R + 8 of this warp's 16; columns nt * 8 + cq + {0, 1} ----
        const int R = lane >> 2, cq = (lane & 3) * 2, row = blk * GF_ROWS + warp * 16 + R;
#pragma unroll
        for (int nt = 0; nt < NT; nt++)
#pragma unroll
            for (int cc = 0; cc < 2; cc++) {
                const int col = nt * 8 + cq + cc;
                if (col >= p.ncols) continue;
                float *dp = p.nslices > 1 ? p.part + ((size_t)r * p.ncols + col) * p.N : p.dst + (size_t)col * p.dst_stride;
                if (row < p.N) dp[row] = acc[nt][cc];
                if (row + 8 < p.N) dp[row + 8] = acc[nt][2 + cc];
            }
    }
}

// MUL_MAT_ID: blockIdx.y = chunk of <= 32 pairs of one expert, tmw the 3-D (K, N, expert) map; otherwise the dense kernel above (a
// body shared with it changes how the dense kernel loads its parameters)
template <bool BF, int NT>
__global__ void __launch_bounds__(GF_THREADS, 1) b200_gemv_f16_grouped_kernel(const __grid_constant__ CUtensorMap tmw, const GfParams p, const GfGroup gr) {
    extern __shared__ uint8_t gf_smem_raw[];
    uint8_t *smem = gf_smem_raw + ((1024u - (smem_u32(gf_smem_raw) & 1023u)) & 1023u);      // SWIZZLE_128B destinations: 1024-byte aligned
    uint8_t *ring = smem;
    uint8_t *xs = smem + p.off_x;
    uint64_t *full = (uint64_t *)(smem + p.off_bar), *empty = full + GF_MAX_STAGES;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ns = p.nstages;
    if (p.use_pdl) pdl_trigger();
    // the routing tables come from the grouping kernel just before: no table read and no weight copy before this wait
    if (p.use_pdl) pdl_wait();
    int e, first, cnt;
    gf_chunk(gr, blockIdx.y, e, first, cnt);
    if (cnt == 0) return;
    const int r = blockIdx.x % p.nslices, g = blockIdx.x / p.nslices;
    const int b0 = (int)((long long)p.nblocks * g / p.ngroups), b1 = (int)((long long)p.nblocks * (g + 1) / p.ngroups);
    const int k0 = r * p.kslice;
    const int nst = (min(p.kslice, p.K - k0) + GF_KS - 1) / GF_KS;          // stages per block
    const int nunits = (b1 - b0) * nst;
    if (threadIdx.x == 0) {
        for (int i = 0; i < ns; i++) { mbar_init(&full[i], 1); mbar_init(&empty[i], GF_CONS); }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == GF_CONS) {
        // ------------------------------------------------------------ producer: one TMA tile per stage
        for (int u = 0; u < nunits; u++) {
            const int st = u % ns, use = u / ns;
            if (use > 0) mbar_wait_bounded(&empty[st], (use - 1) & 1);
            if (elect_one_sync()) {
                mbar_arrive_expect_tx(&full[st], GF_STAGE);
                tma_load_3d(ring + (size_t)st * GF_STAGE, &tmw, k0 + (u % nst) * GF_KS, (b0 + u / nst) * GF_ROWS, e, &full[st]);
            }
            __syncwarp();
        }
        return;
    }
    // ---------------------------------------------------------------- consumers: x slice -> shared memory, rounded once
    {
        const int q4 = p.kslice / 4;                      // float4 groups per column
        for (int i = threadIdx.x; i < NT * 8 * q4; i += GF_CONS * 32) {
            const int col = i / q4, k = k0 + (i % q4) * 4;
            float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            if (col < cnt && k < p.K) {                   // column of the pair: its token's (b_ne1 == 1) or its own
                const int pair = gr.pairs[first + col];
                v = *(const float4 *)(p.x + (size_t)(gr.b_ne1 == 1 ? pair / gr.n_used : pair) * p.x_stride + k);
            }
            *(uint2 *)(xs + (size_t)col * p.xpitch + (size_t)(i % q4) * 8) = make_uint2(pack2<BF>(v.x, v.y), pack2<BF>(v.z, v.w));
        }
    }
    named_bar_sync(1, GF_CONS * 32);
    const uint32_t xs_saddr = smem_u32(xs), ring_saddr = smem_u32(ring);
    // ldmatrix lanes: A row (l & 7) + 8 ((l >> 3) & 1) of this warp's 16, 16-byte chunk (l >> 4) of the k16 step; B row l & 7 of n-tile
    const int arow = (lane & 7) + ((lane >> 3) & 1) * 8, achunk = lane >> 4;
    const uint32_t a_off = (uint32_t)(warp * 16 + arow) * 128u;
    const int mi = lane >> 3, rr = lane & 7;
    int u = 0;
    for (int blk = b0; blk < b1; blk++) {
        float acc[NT][4];
#pragma unroll
        for (int nt = 0; nt < NT; nt++) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.0f;
        for (int s = 0; s < nst; s++, u++) {
            const int st = u % ns, use = u / ns;
            mbar_wait_bounded(&full[st], use & 1);
            const uint32_t tile = ring_saddr + (uint32_t)st * GF_STAGE + a_off;
#pragma unroll
            for (int ks = 0; ks < GF_KS / 16; ks++) {
                uint32_t a0, a1, a2, a3;
                ldsm_x4(a0, a1, a2, a3, tile + (uint32_t)(((2 * ks + achunk) ^ (arow & 7)) * 16));
                const uint32_t kb = (uint32_t)(s * GF_KS + ks * 16) * 2u;
                uint32_t b[NT][2];
                if (NT == 1) {
                    ldsm_x2(b[0][0], b[0][1], xs_saddr + (uint32_t)rr * p.xpitch + kb + (uint32_t)(mi & 1) * 16);
                } else {
#pragma unroll
                    for (int n2 = 0; n2 < NT / 2; n2++)
                        ldsm_x4(b[2 * n2][0], b[2 * n2][1], b[2 * n2 + (NT > 1)][0], b[2 * n2 + (NT > 1)][1],
                                xs_saddr + (uint32_t)((2 * n2 + (mi >> 1)) * 8 + rr) * p.xpitch + kb + (uint32_t)(mi & 1) * 16);
                }
#pragma unroll
                for (int nt = 0; nt < NT; nt++) mma_k16<BF>(acc[nt], a0, a1, a2, a3, b[nt][0], b[nt][1]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[st]);
        }
        // ---- store: rows R, R + 8 of this warp's 16; columns nt * 8 + cq + {0, 1} ----
        const int R = lane >> 2, cq = (lane & 3) * 2, row = blk * GF_ROWS + warp * 16 + R;
#pragma unroll
        for (int nt = 0; nt < NT; nt++)
#pragma unroll
            for (int cc = 0; cc < 2; cc++) {
                const int col = nt * 8 + cq + cc;
                if (col >= cnt) continue;
                float *dp;                                // partials in sorted-pair order; results scattered to (slot, token)
                if (p.nslices > 1) dp = p.part + ((size_t)r * gr.npairs + first + col) * p.N;
                else {
                    const int pair = gr.pairs[first + col];
                    dp = p.dst + (size_t)(pair % gr.n_used) * gr.d_nb1 + (size_t)(pair / gr.n_used) * gr.d_nb2;
                }
                if (row < p.N) dp[row] = acc[nt][cc];
                if (row + 8 < p.N) dp[row + 8] = acc[nt][2 + cc];
            }
    }
}

// dst[col][row] = sum over the K slices in slice order (deterministic)
__global__ void __launch_bounds__(256) b200_gemv_f16_reduce_kernel(const float *__restrict__ part, int nslices, int N, int ncols, float *dst, size_t dst_stride,
                                                                   int use_pdl) {
    if (use_pdl) { pdl_trigger(); pdl_wait(); }
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)ncols * N) return;
    const int col = (int)(i / N), row = (int)(i % N);
    float a = part[i];
    for (int r = 1; r < nslices; r++) a += part[(size_t)r * ncols * N + i];
    dst[(size_t)col * dst_stride + row] = a;
}

// grouped: part[slice][sorted pair][N] -> dst[:, slot, token] of the pair, summed in slice order (deterministic); off[E] = routed pairs
__global__ void __launch_bounds__(256) b200_f16_grouped_reduce_kernel(const float *__restrict__ part, int nslices, int N, int npairs, const int32_t *off,
                                                                      const int32_t *pairs, int E, int n_used, float *dst, size_t d_nb1, size_t d_nb2, int use_pdl) {
    if (use_pdl) { pdl_trigger(); pdl_wait(); }
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)off[E] * N) return;
    const int q = (int)(i / N), row = (int)(i % N), pair = pairs[q];
    float a = part[i];
    for (int r = 1; r < nslices; r++) a += part[(size_t)r * npairs * N + i];
    dst[(size_t)(pair % n_used) * d_nb1 + (size_t)(pair / n_used) * d_nb2 + row] = a;
}

template <bool BF, int NT, bool G>
int launch_gf(b200_ctx *ctx, const CUtensorMap &tm, const GfParams &p, const GfGroup *g, dim3 grid, size_t smem) {
    auto kern = G ? (void *)b200_gemv_f16_grouped_kernel<BF, NT> : (void *)b200_gemv_f16_kernel<BF, NT>;
    static bool attr_set[16] = {false};
    if (!attr_set[ctx->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->smem_optin));
        attr_set[ctx->device & 15] = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = dim3(GF_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = p.use_pdl ? 1 : 0;
    if (G) CUDA_TRY(cudaLaunchKernelEx(&cfg, b200_gemv_f16_grouped_kernel<BF, NT>, tm, p, *g));
    else   CUDA_TRY(cudaLaunchKernelEx(&cfg, b200_gemv_f16_kernel<BF, NT>, tm, p));
    ctx->launches++;
    return B200_OK;
}

// K slicing and shared-memory geometry.  ctas: the CTAs one set of (row-block group, K slice) CTAs may occupy -- the machine (dense) or
// its share per chunk (grouped).  Among 1..32 slices whose x slice fits its 64 KB, take the one with the least stages on the busiest CTA,
// the fewest slices on a tie.
int gf_plan(b200_ctx *ctx, GfParams &p, int NT, int64_t K, int64_t ctas, size_t &smem) {
    const int64_t kmax = (int64_t)(GF_X_BYTES / (NT * 8 * 2)) / GF_KS * GF_KS;
    const int64_t K64 = (K + GF_KS - 1) / GF_KS * GF_KS;
    int64_t best = INT64_MAX;
    for (int n = 1; n <= 32; n++) {
        const int64_t ks = ((K64 / GF_KS + n - 1) / n) * GF_KS;
        if (ks > kmax) continue;
        const int ns_eff = (int)((K + ks - 1) / ks);
        if (ns_eff != n) continue;
        int64_t groups = std::max<int64_t>(1, std::min<int64_t>(p.nblocks, ctas / ns_eff));
        const int64_t cost = (p.nblocks + groups - 1) / groups * (ks / GF_KS);
        if (cost < best) { best = cost; p.kslice = (int)ks; p.nslices = ns_eff; p.ngroups = (int)groups; }
    }
    if (best == INT64_MAX) { b200_set_error("gemv_f16: no K slicing"); return B200_ERR_FAILED; }
    p.xpitch = (uint32_t)p.kslice * 2u + 16u;            // (pitch / 16) odd: ldmatrix conflict-free
    // shared memory: [ring: nstages x 16 KB][x: 8 NT columns x xpitch][barriers]; + 1 KB for the manual 1024-byte alignment
    const uint32_t xbytes = (uint32_t)(NT * 8) * p.xpitch;
    const size_t fixed = 1024 + xbytes + 2 * GF_MAX_STAGES * 8;
    int ns = (int)((ctx->smem_optin - fixed) / GF_STAGE);
    if (ns > GF_MAX_STAGES) ns = GF_MAX_STAGES;
    if (ns < 2) { b200_set_error("gemv_f16: shared memory"); return B200_ERR_FAILED; }
    p.nstages = ns;
    p.off_x = (uint32_t)ns * GF_STAGE;
    p.off_bar = p.off_x + ((xbytes + 15u) & ~15u);
    smem = 1024 + (size_t)p.off_bar + 2 * GF_MAX_STAGES * 8;
    return B200_OK;
}

// g: the routing of the grouped kernel; nullptr: the dense kernel
template <bool G>
int launch_gf_any(b200_ctx *ctx, bool bf, int NT, const CUtensorMap &tm, const GfParams &p, const GfGroup *g, dim3 grid, size_t smem) {
    if (bf) return NT == 1 ? launch_gf<true, 1, G>(ctx, tm, p, g, grid, smem) : NT == 2 ? launch_gf<true, 2, G>(ctx, tm, p, g, grid, smem) : launch_gf<true, 4, G>(ctx, tm, p, g, grid, smem);
    return NT == 1 ? launch_gf<false, 1, G>(ctx, tm, p, g, grid, smem) : NT == 2 ? launch_gf<false, 2, G>(ctx, tm, p, g, grid, smem) : launch_gf<false, 4, G>(ctx, tm, p, g, grid, smem);
}

}  // namespace

int gemv_f16_run(b200_ctx *ctx, int type, const uint16_t *W, int64_t N, int64_t K, const float *x, size_t x_stride_bytes, int ncols, float *dst,
                 size_t dst_stride, bool w_const) {
    if ((type != B200_TYPE_F16 && type != B200_TYPE_BF16) || ncols < 1 || ncols > (int)F16MM_STREAM_MAX_M || K % 8 || ((uintptr_t)W & 15) ||
        ((uintptr_t)x & 15) || (x_stride_bytes & 15) || N < 1 || N > INT32_MAX || K > INT32_MAX) {
        b200_set_error("gemv_f16: unsupported shape");
        return B200_ERR_UNSUPPORTED;
    }
    const int NT = ncols <= 8 ? 1 : ncols <= 16 ? 2 : 4;
    GfParams p = {};
    p.x = x; p.x_stride = x_stride_bytes / 4; p.N = (int)N; p.K = (int)K; p.ncols = ncols;
    p.dst = dst; p.dst_stride = dst_stride;
    p.nblocks = (int)((N + GF_ROWS - 1) / GF_ROWS);
    p.use_pdl = ctx->opt_pdl; p.w_const = w_const ? 1 : 0;
    size_t smem = 0;
    int rc = gf_plan(ctx, p, NT, K, ctx->sm_count, smem);
    if (rc) return rc;
    if (p.nslices > 1) {
        p.part = (float *)ctx->get_scratch(SCRATCH_MISC, (size_t)p.nslices * ncols * N * 4);
        if (!p.part) return B200_ERR_ALLOC;
    }
    CUtensorMap tm;
    rc = make_tmap_16bit(&tm, type, W, K, N, GF_KS, GF_ROWS);
    if (rc) return rc;
    rc = launch_gf_any<false>(ctx, type == B200_TYPE_BF16, NT, tm, p, nullptr, dim3((unsigned)(p.ngroups * p.nslices)), smem);
    if (rc || p.nslices == 1) return rc;
    const int64_t total = (int64_t)ncols * N;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((total + 255) / 256)); cfg.blockDim = dim3(256); cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = p.use_pdl ? 1 : 0;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, b200_gemv_f16_reduce_kernel, (const float *)p.part, p.nslices, (int)N, ncols, dst, dst_stride, p.use_pdl));
    ctx->launches++;
    return B200_OK;
}

// every chunk of <= 32 pairs of one expert streams that expert's rows once; the grid covers g.max_chunks chunks and the ones beyond the
// routed count exit at once
int gemv_f16_run_grouped(b200_ctx *ctx, int type, const uint16_t *As, int64_t N, int64_t K, const float *x, size_t x_stride_bytes, const MmGroupDesc &g,
                         int64_t npairs, float *dst) {
    if ((type != B200_TYPE_F16 && type != B200_TYPE_BF16) || K % 8 || (((uintptr_t)As | g.expert_stride | (uintptr_t)x | x_stride_bytes) & 15) ||
        N < 1 || N > INT32_MAX || K > INT32_MAX || npairs < 1 || npairs > INT32_MAX / 32 || g.max_chunks < 1) {
        b200_set_error("gemv_f16 grouped: unsupported shape");
        return B200_ERR_UNSUPPORTED;
    }
    const int64_t most = std::min<int64_t>(32, npairs);         // pairs in the fullest chunk
    const int NT = most <= 8 ? 1 : most <= 16 ? 2 : 4;
    GfParams p = {};
    p.x = x; p.x_stride = x_stride_bytes / 4; p.N = (int)N; p.K = (int)K; p.ncols = 0;
    p.dst = dst;
    p.nblocks = (int)((N + GF_ROWS - 1) / GF_ROWS);
    p.use_pdl = ctx->opt_pdl; p.w_const = 0;
    const GfGroup gg = {g.off, g.pairs, g.E, g.n_used, g.b_ne1, (int)npairs, g.d_nb1, g.d_nb2};
    size_t smem = 0;
    int rc = gf_plan(ctx, p, NT, K, std::max<int64_t>(1, ctx->sm_count / g.max_chunks), smem);      // the chunks share one wave
    if (rc) return rc;
    if (p.nslices > 1) {
        p.part = (float *)ctx->get_scratch(SCRATCH_MISC, (size_t)p.nslices * npairs * N * 4);
        if (!p.part) return B200_ERR_ALLOC;
    }
    CUtensorMap tm;
    rc = make_tmap_16bit_3d(&tm, type, As, K, N, g.E, g.expert_stride, GF_KS, GF_ROWS);
    if (rc) return rc;
    rc = launch_gf_any<true>(ctx, type == B200_TYPE_BF16, NT, tm, p, &gg, dim3((unsigned)(p.ngroups * p.nslices), (unsigned)g.max_chunks), smem);
    if (rc || p.nslices == 1) return rc;
    return launch_f16_grouped_reduce(ctx, p.part, p.nslices, N, g, npairs, dst, p.use_pdl);
}

int launch_f16_grouped_reduce(b200_ctx *ctx, const float *part, int nslices, int64_t N, const MmGroupDesc &g, int64_t npairs, float *dst, int use_pdl) {
    const int64_t total = npairs * N;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((total + 255) / 256)); cfg.blockDim = dim3(256); cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = use_pdl ? 1 : 0;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, b200_f16_grouped_reduce_kernel, part, nslices, (int)N, (int)npairs, g.off, (const int32_t *)g.pairs, g.E, g.n_used, dst,
                                g.d_nb1, g.d_nb2, use_pdl));
    ctx->launches++;
    return B200_OK;
}
