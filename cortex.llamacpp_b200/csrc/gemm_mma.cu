// gemm_mma.cu -- prompt-batch GEMM (more than 32 token columns) for all five GGUF formats on the warp-level tensor-core path.
//
// Replaces mul_mat_q (ggml-cuda/mmq.cuh:2501-2657: 128 x mmq_x tiles, weights de-nibbled to int8 in shared memory, q8_1 activations,
// float fix-up per 32-k block).  Round 1's tcgen05 kind::i8 GEMM (since removed) kept the tensor pipe 6 % busy: its CUDA-core stages -- expanding
// every weight block to hi/lo int8 operand tiles once per 128-token tile, and a ~16-instruction drain per output element per
// 256 k -- bound it at 112 TOPS, below the reference's own MMQ on the same B200 (profiles/r2_ref_cuda_vs_plugin.txt).  This kernel
// removes both stages:
//   * weights stay in their GGUF bytes in shared memory (a stage = the 256-k block of 128 rows = 128 pieces of 144..272 bytes, brought
//     in by 16-byte cp.async from all threads, completion on the stage's mbarrier); every warp expands the nibbles of ITS 32 rows
//     straight into mma A fragments in registers -- no operand tiles are written;
//   * activations are quantised once per matmul exactly like the CPU (q8_K / q8_0, quant_warp.cuh) into [token tile][super-block]
//     stage images (int8 rows padded for ldmatrix + block scales + per-32 sums) that ONE bulk copy brings in;
//   * mma.sync.m16n8k32.s8 per 32-wide sub-block, the 6-bit sub-scale applied to the int32 product (4 IMADs per IMMA): the CPU's
//     per-block integer  sum_j sc_j sum_l q a  exactly; q6_K / q4_0 / q8_0 use signed quants (no offset term); once per 256 k the
//     integers are folded into f32 accumulators with d_w * d_a (and the dp2a min term), all in registers.
// CTA tile 128 rows x 128 tokens, 8 warps (4 x 2, warp tile 32 x 64; every thread issues its share of the next stages' cp.async copies, up to `nstages`
// stages ahead), persistent over (row tile, token tile, K slice) work items; deterministic split-K for matrices whose tile grid would leave SMs idle.
// Roofline: tensor (int8).  Algorithmic work 2*N*K*M.  The legacy IMMA pipe peaks at 1150 TOPS on B200 (tools/micro/imma_bench.cu).
#include "common.cuh"
#include "quant_warp.cuh"

namespace {

constexpr int GT_M = 128, GT_N = 128;                 // CTA tile: weight rows x tokens
constexpr int G_BSTRIDE = 256 + 16;                   // bytes per token row of a stage image: (stride / 16) odd -> ldmatrix conflict-free
constexpr int G_THREADS = 8 * 32;                     // 8 warps: 255 registers per thread (a 9th producer warp would round the block to 384 threads: 168)

// stage image of the activations of one (token tile, super-block), written by the pack kernel, copied by one bulk copy:
//   [128 tokens][272] int8 quants | d: q8_K [128] floats, q8_0 mode [128][8] floats | q8_K only: per-32 sums [128][8] int16
__host__ __device__ inline uint32_t img_off_d() { return GT_N * G_BSTRIDE; }
__host__ __device__ inline uint32_t img_off_s(int q8k) { return img_off_d() + (q8k ? GT_N * 4 : GT_N * 8 * 4); }
__host__ __device__ inline uint32_t img_bytes(int q8k) { return (img_off_s(q8k) + (q8k ? GT_N * 8 * 2 : 0) + 127u) & ~127u; }

struct GParams {
    const uint8_t *W; uint32_t rb, bbytes; int type, N, K, M, q8k;
    int tn;                                            // = GT_N.  g_lookup reads it from here: with the constant folded in, ptxas spills twice as much in the Q5_K GEMM
    const uint8_t *img;                                // [ntile][nsb] stage images
    float *dst; size_t dst_stride;
    float *part;                                       // [ksplit][M][N] when ksplit > 1
    int nsb, ntile, nrt, ksplit, sb_per_split, nitems;
    int nstages; uint32_t stage_bytes, a_bytes, rstride;
    // grouped (MUL_MAT_ID) mode: a "token tile" is a chunk of <= 128 (token, slot) pairs routed to one expert
    const int32_t *g_off, *g_pairs; int g_E, g_n_used, g_b_ne1, g_chunks;       // g_E == 0: dense
    size_t g_expert_stride, g_d_nb1, g_d_nb2;
};

// grouped mode: chunk -> (expert, first pair, pairs in the chunk; 0 = the chunk does not exist)
__device__ __forceinline__ void g_lookup(const GParams &p, int chunk, int &e, int &first, int &cnt) {
    cnt = 0; first = 0;
    for (e = 0; e < p.g_E; e++) {
        const int o0 = p.g_off[e], n = p.g_off[e + 1] - o0, nch = (n + p.tn - 1) / p.tn;
        if (chunk < nch) { first = o0 + chunk * p.tn; cnt = min(p.tn, n - chunk * p.tn); return; }
        chunk -= nch;
    }
}

__device__ __forceinline__ void ldsm4(uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3, uint32_t saddr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(saddr));
}
__device__ __forceinline__ void imma32(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.s8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
                 : "=r"(c[0]), "=r"(c[1]), "=r"(c[2]), "=r"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "r"(0));
}
__device__ __forceinline__ void imma16(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t b0) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.s32.s8.s8.s32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%7,%7,%7,%7};"
                 : "=r"(c[0]), "=r"(c[1]), "=r"(c[2]), "=r"(c[3]) : "r"(a0), "r"(a1), "r"(b0), "r"(0));
}
__device__ __forceinline__ uint32_t lds2(const uint8_t *p) { return (uint32_t)*(const unsigned short *)p | ((uint32_t)*(const unsigned short *)(p + 2) << 16); }
__device__ __forceinline__ float hf(uint32_t bits) { return __half2float(__ushort_as_half((unsigned short)bits)); }

// ---------------------------------------------------------------------------------------------------------------- activation pack
// one warp per (token, super-block): quantise 256 floats like the CPU and write them into the stage image of the token's tile
__global__ void __launch_bounds__(256) b200_gemm_mma_pack_kernel(const float *__restrict__ x, size_t x_stride, int K, int M, int q8k, int nsb, uint8_t *__restrict__ img) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int ntile = (M + GT_N - 1) / GT_N;
    if (gw >= (int64_t)ntile * GT_N * nsb) return;
    const int b = (int)(gw % nsb), tok = (int)(gw / nsb), tile = tok / GT_N, t = tok % GT_N;
    uint8_t *im = img + ((size_t)tile * nsb + b) * img_bytes(q8k);
    float v[8];
    if (tok < M) {
        const float *xp = (const float *)((const char *)x + (size_t)tok * x_stride) + b * 256 + lane * 8;
        const float4 a = *(const float4 *)xp, c = *(const float4 *)(xp + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
    } else {
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = 0.0f;
    }
    uint2 qp;
    if (q8k) {
        float d; int pair;
        warp_quant_q8k(v, lane, qp, d, pair);
        const int s32 = pair + __shfl_down_sync(0xffffffffu, pair, 2);           // even lanes hold per-16 sums: lanes 0, 4, 8, ... add their neighbour pair
        if ((lane & 3) == 0) ((int16_t *)(im + img_off_s(1)))[t * 8 + (lane >> 2)] = (int16_t)s32;
        if (lane == 0) ((float *)(im + img_off_d()))[t] = d;
    } else {
        float d16; int bsum;
        warp_quant_q80(v, qp, d16, bsum);
        if ((lane & 3) == 0) ((float *)(im + img_off_d()))[t * 8 + (lane >> 2)] = d16;
    }
    *(uint2 *)(im + (size_t)t * G_BSTRIDE + lane * 8) = qp;
}

// one 256-k super-block of a warp tile: 2 m-tiles (rows R, R+8 of each from rowp[mt][h], raw GGUF block bytes) x NTW n-tiles of 8 tokens
// starting at token `tokbase` of the stage image (b_lane: this lane's ldmatrix address, bd / bs: block scales and per-32 sums)
template <int TYPE, int NTW>
__device__ __forceinline__ void sb_compute(const uint8_t *const (&rowp)[2][2], uint32_t b_lane, const float *bd, const int16_t *bs, int tokbase, int lane,
                                           float (&out)[2][NTW][4]) {
    const int kq = (lane & 3) * 4, cq = (lane & 3) * 2;
    if (TYPE == B200_TYPE_Q4_K || TYPE == B200_TYPE_Q5_K) {
        int P[2][NTW][4];
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
            for (int nt = 0; nt < NTW; nt++) P[mt][nt][0] = P[mt][nt][1] = P[mt][nt][2] = P[mt][nt][3] = 0;
        uint32_t sc_lo[2][2], sc_hi[2][2], mn_lo[2][2], mn_hi[2][2];
        float dd[2][2], dm[2][2];
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const uint4 hd = *(const uint4 *)rowp[mt][h];
                sc_lo[mt][h] = hd.y & 0x3f3f3f3fu; mn_lo[mt][h] = hd.z & 0x3f3f3f3fu;
                sc_hi[mt][h] = (hd.w & 0x0f0f0f0fu) | ((hd.y >> 2) & 0x30303030u);
                mn_hi[mt][h] = ((hd.w >> 4) & 0x0f0f0f0fu) | ((hd.z >> 2) & 0x30303030u);
                dd[mt][h] = hf(hd.x); dm[mt][h] = -hf(hd.x >> 16);
            }
        constexpr int QO = TYPE == B200_TYPE_Q5_K ? 48 : 16;
#pragma unroll
        for (int g = 0; g < 4; g++) {
            uint32_t w[2][2][2];
#pragma unroll
            for (int mt = 0; mt < 2; mt++)
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    w[mt][h][0] = *(const uint32_t *)(rowp[mt][h] + QO + 32 * g + kq);
                    w[mt][h][1] = *(const uint32_t *)(rowp[mt][h] + QO + 32 * g + 16 + kq);
                }
#pragma unroll
            for (int sub = 0; sub < 2; sub++) {
                const int j = 2 * g + sub;
                uint32_t a[2][4]; int s[2][2];
#pragma unroll
                for (int mt = 0; mt < 2; mt++) {
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        uint32_t x0 = sub ? (w[mt][h][0] >> 4) & 0x0f0f0f0fu : w[mt][h][0] & 0x0f0f0f0fu;
                        uint32_t x1 = sub ? (w[mt][h][1] >> 4) & 0x0f0f0f0fu : w[mt][h][1] & 0x0f0f0f0fu;
                        if (TYPE == B200_TYPE_Q5_K) {
                            const uint32_t hb0 = *(const uint32_t *)(rowp[mt][h] + 16 + kq), hb1 = *(const uint32_t *)(rowp[mt][h] + 32 + kq);
                            x0 |= ((hb0 >> j) & 0x01010101u) << 4; x1 |= ((hb1 >> j) & 0x01010101u) << 4;
                        }
                        a[mt][h] = x0; a[mt][2 + h] = x1;
                        s[mt][h] = (int)(((j < 4 ? sc_lo[mt][h] : sc_hi[mt][h]) >> (8 * (j & 3))) & 0xffu);
                    }
                }
#pragma unroll
                for (int np = 0; np < NTW / 2; np++) {
                    uint32_t b0, b1, b2, b3;
                    ldsm4(b0, b1, b2, b3, b_lane + (uint32_t)(np * 16) * G_BSTRIDE + (uint32_t)(j * 32));
#pragma unroll
                    for (int mt = 0; mt < 2; mt++) {
                        int c[4];
                        imma32(c, a[mt][0], a[mt][1], a[mt][2], a[mt][3], b0, b1);
                        P[mt][2 * np][0] += s[mt][0] * c[0]; P[mt][2 * np][1] += s[mt][0] * c[1]; P[mt][2 * np][2] += s[mt][1] * c[2]; P[mt][2 * np][3] += s[mt][1] * c[3];
                        imma32(c, a[mt][0], a[mt][1], a[mt][2], a[mt][3], b2, b3);
                        P[mt][2 * np + 1][0] += s[mt][0] * c[0]; P[mt][2 * np + 1][1] += s[mt][0] * c[1]; P[mt][2 * np + 1][2] += s[mt][1] * c[2]; P[mt][2 * np + 1][3] += s[mt][1] * c[3];
                    }
                }
            }
        }
        // fold the super-block: out += da * (d * P - dmin * M), M = sum_j m_j * (sum of the token's quants over sub-block j)
#pragma unroll
        for (int nt = 0; nt < NTW; nt++)
#pragma unroll
            for (int cc = 0; cc < 2; cc++) {
                const int tok = tokbase + nt * 8 + cq + cc;
                const uint4 sv = *(const uint4 *)(bs + tok * 8);
                const float da = bd[tok];
#pragma unroll
                for (int mt = 0; mt < 2; mt++)
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        int Mv = __dp2a_lo((int)sv.x, (int)mn_lo[mt][h], 0); Mv = __dp2a_hi((int)sv.y, (int)mn_lo[mt][h], Mv);
                        Mv = __dp2a_lo((int)sv.z, (int)mn_hi[mt][h], Mv); Mv = __dp2a_hi((int)sv.w, (int)mn_hi[mt][h], Mv);
                        out[mt][nt][2 * h + cc] = fmaf(da, fmaf(dd[mt][h], (float)P[mt][nt][2 * h + cc], dm[mt][h] * (float)Mv), out[mt][nt][2 * h + cc]);
                    }
            }
    } else if (TYPE == B200_TYPE_Q6_K) {
        int P[2][NTW][4];
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
            for (int nt = 0; nt < NTW; nt++) P[mt][nt][0] = P[mt][nt][1] = P[mt][nt][2] = P[mt][nt][3] = 0;
#pragma unroll
        for (int hh = 0; hh < 2; hh++) {
#pragma unroll
            for (int t = 0; t < 4; t++) {
                const int j = 4 * hh + t;
                uint32_t a[2][4]; int sA[2][2], sB[2][2];
#pragma unroll
                for (int mt = 0; mt < 2; mt++)
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        const uint8_t *bp = rowp[mt][h];
                        const uint32_t l0 = lds2(bp + 64 * hh + 32 * (t & 1) + kq), l1 = lds2(bp + 64 * hh + 32 * (t & 1) + 16 + kq);
                        const uint32_t q0 = lds2(bp + 128 + 32 * hh + kq), q1 = lds2(bp + 128 + 32 * hh + 16 + kq);
                        a[mt][h]     = __vsub4(((t < 2 ? l0 : l0 >> 4) & 0x0f0f0f0fu) | (((q0 >> (2 * t)) & 0x03030303u) << 4), 0x20202020u);
                        a[mt][2 + h] = __vsub4(((t < 2 ? l1 : l1 >> 4) & 0x0f0f0f0fu) | (((q1 >> (2 * t)) & 0x03030303u) << 4), 0x20202020u);
                        sA[mt][h] = (int)(int8_t)bp[192 + 2 * j]; sB[mt][h] = (int)(int8_t)bp[193 + 2 * j];
                    }
#pragma unroll
                for (int np = 0; np < NTW / 2; np++) {
                    uint32_t b0, b1, b2, b3;
                    ldsm4(b0, b1, b2, b3, b_lane + (uint32_t)(np * 16) * G_BSTRIDE + (uint32_t)(j * 32));
#pragma unroll
                    for (int mt = 0; mt < 2; mt++) {
                        int c[4], e[4];
                        imma16(c, a[mt][0], a[mt][1], b0); imma16(e, a[mt][2], a[mt][3], b1);
                        P[mt][2 * np][0] += sA[mt][0] * c[0] + sB[mt][0] * e[0]; P[mt][2 * np][1] += sA[mt][0] * c[1] + sB[mt][0] * e[1];
                        P[mt][2 * np][2] += sA[mt][1] * c[2] + sB[mt][1] * e[2]; P[mt][2 * np][3] += sA[mt][1] * c[3] + sB[mt][1] * e[3];
                        imma16(c, a[mt][0], a[mt][1], b2); imma16(e, a[mt][2], a[mt][3], b3);
                        P[mt][2 * np + 1][0] += sA[mt][0] * c[0] + sB[mt][0] * e[0]; P[mt][2 * np + 1][1] += sA[mt][0] * c[1] + sB[mt][0] * e[1];
                        P[mt][2 * np + 1][2] += sA[mt][1] * c[2] + sB[mt][1] * e[2]; P[mt][2 * np + 1][3] += sA[mt][1] * c[3] + sB[mt][1] * e[3];
                    }
                }
            }
        }
        float dd[2][2];
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
            for (int h = 0; h < 2; h++) dd[mt][h] = hf(*(const unsigned short *)(rowp[mt][h] + 208));
#pragma unroll
        for (int nt = 0; nt < NTW; nt++)
#pragma unroll
            for (int cc = 0; cc < 2; cc++) {
                const float da = bd[tokbase + nt * 8 + cq + cc];
#pragma unroll
                for (int mt = 0; mt < 2; mt++)
#pragma unroll
                    for (int h = 0; h < 2; h++) out[mt][nt][2 * h + cc] = fmaf(dd[mt][h] * da, (float)P[mt][nt][2 * h + cc], out[mt][nt][2 * h + cc]);
            }
    } else {
        // q4_0 (18 B) / q8_0 (34 B) blocks of 32: one float scale per (row, block) and per (token, block)
        constexpr int SB = TYPE == B200_TYPE_Q4_0 ? 18 : 34;
#pragma unroll 2
        for (int j = 0; j < 8; j++) {
            uint32_t a[2][4]; float dw[2][2];
#pragma unroll
            for (int mt = 0; mt < 2; mt++)
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const uint8_t *bp = rowp[mt][h] + j * SB;
                    dw[mt][h] = hf(*(const unsigned short *)bp);
                    if (TYPE == B200_TYPE_Q4_0) {
                        const uint32_t wv = lds2(bp + 2 + kq);
                        a[mt][h] = __vsub4(wv & 0x0f0f0f0fu, 0x08080808u); a[mt][2 + h] = __vsub4((wv >> 4) & 0x0f0f0f0fu, 0x08080808u);
                    } else {
                        a[mt][h] = lds2(bp + 2 + kq); a[mt][2 + h] = lds2(bp + 18 + kq);
                    }
                }
#pragma unroll
            for (int np = 0; np < NTW / 2; np++) {
                uint32_t b0, b1, b2, b3;
                ldsm4(b0, b1, b2, b3, b_lane + (uint32_t)(np * 16) * G_BSTRIDE + (uint32_t)(j * 32));
#pragma unroll
                for (int q = 0; q < 2; q++) {
                    const int nt = 2 * np + q;
                    const float da0 = bd[(tokbase + nt * 8 + cq) * 8 + j], da1 = bd[(tokbase + nt * 8 + cq + 1) * 8 + j];
#pragma unroll
                    for (int mt = 0; mt < 2; mt++) {
                        int c[4];
                        imma32(c, a[mt][0], a[mt][1], a[mt][2], a[mt][3], q ? b2 : b0, q ? b3 : b1);
                        out[mt][nt][0] = fmaf((float)c[0], dw[mt][0] * da0, out[mt][nt][0]); out[mt][nt][1] = fmaf((float)c[1], dw[mt][0] * da1, out[mt][nt][1]);
                        out[mt][nt][2] = fmaf((float)c[2], dw[mt][1] * da0, out[mt][nt][2]); out[mt][nt][3] = fmaf((float)c[3], dw[mt][1] * da1, out[mt][nt][3]);
                    }
                }
            }
        }
    }
}

// grouped: one warp per (chunk slot, super-block); the slot's pair gives the activation column
__global__ void __launch_bounds__(256) b200_gemm_mma_pack_grouped_kernel(const float *__restrict__ x, size_t x_stride, GParams p, uint8_t *__restrict__ img) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (gw >= (int64_t)p.g_chunks * GT_N * p.nsb) return;
    const int b = (int)(gw % p.nsb), slot = (int)(gw / p.nsb), chunk = slot / GT_N, t = slot % GT_N;
    int e, first, cnt;
    g_lookup(p, chunk, e, first, cnt);
    if (cnt == 0) return;
    uint8_t *im = img + ((size_t)chunk * p.nsb + b) * img_bytes(p.q8k);
    float v[8];
    if (t < cnt) {
        const int pair = p.g_pairs[first + t];
        const int64_t colidx = p.g_b_ne1 == 1 ? pair / p.g_n_used : pair;
        const float *xp = (const float *)((const char *)x + (size_t)colidx * x_stride) + b * 256 + lane * 8;
        const float4 a = *(const float4 *)xp, c = *(const float4 *)(xp + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
    } else {
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = 0.0f;
    }
    uint2 qp;
    if (p.q8k) {
        float d; int pair;
        warp_quant_q8k(v, lane, qp, d, pair);
        const int s32 = pair + __shfl_down_sync(0xffffffffu, pair, 2);
        if ((lane & 3) == 0) ((int16_t *)(im + img_off_s(1)))[t * 8 + (lane >> 2)] = (int16_t)s32;
        if (lane == 0) ((float *)(im + img_off_d()))[t] = d;
    } else {
        float d16; int bsum;
        warp_quant_q80(v, qp, d16, bsum);
        if ((lane & 3) == 0) ((float *)(im + img_off_d()))[t * 8 + (lane >> 2)] = d16;
    }
    *(uint2 *)(im + (size_t)t * G_BSTRIDE + lane * 8) = qp;
}

// ---------------------------------------------------------------------------------------------------------------- the GEMM
template <int TYPE>
__global__ void __launch_bounds__(G_THREADS, 1) b200_gemm_mma_kernel(const GParams p) {
    constexpr int NTW = GT_N / 16;                      // n-tiles per warp: the two token halves of the tile belong to warps wn = 0, 1
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *full = (uint64_t *)smem, *empty = full + 8;
    uint8_t *ring = smem + 128;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ns = p.nstages;
    if (threadIdx.x == 0) {
        for (int i = 0; i < ns; i++) { mbar_init(&full[i], G_THREADS + 1); mbar_init(&empty[i], 8); }
        mbar_fence_init();
    }
    __syncthreads();
    const uint32_t ibytes = img_bytes(p.q8k);

    // ------------------------------------------------------------ producer side, ALL threads: stage iteration p_it stands for (p_item, p_b).
    // The 128 row pieces of a stage (144..272 bytes each) go through 16-byte cp.async issued by every thread -- a bulk copy per piece
    // costs ~60 ns of TMA issue each and starved the pipeline (profiles/r2_ncu_summaries.md) -- and complete on the stage's mbarrier
    // (cp.async.mbarrier.arrive.noinc); the 37 KB activation image is one bulk copy.
    constexpr int CPR = TYPE == B200_TYPE_Q4_K ? 9 : TYPE == B200_TYPE_Q5_K ? 11 : TYPE == B200_TYPE_Q6_K ? 15 : TYPE == B200_TYPE_Q4_0 ? 9 : 17;   // 16-byte chunks per row piece
    int p_it = 0, p_item = blockIdx.x, p_b = 0, p_b1 = 0;
    if (p_item < p.nitems) { const int ks = p_item % p.ksplit; p_b = ks * p.sb_per_split; p_b1 = min(p.nsb, p_b + p.sb_per_split); }
    auto produce_upto = [&](int limit) {
        while (p_item < p.nitems && p_it < limit) {
            const int rt = (p_item / p.ksplit) % p.nrt, tt = p_item / (p.ksplit * p.nrt);
            const uint8_t *Wb = p.W;
            if (p.g_E) {                    // grouped: token tile tt = chunk of one expert; chunks beyond the routed pairs do not exist
                int e, first, cnt;
                g_lookup(p, tt, e, first, cnt);
                if (cnt == 0) { p_item += gridDim.x; if (p_item < p.nitems) { p_b = 0; p_b1 = p.nsb; } continue; }
                Wb += (size_t)e * p.g_expert_stride;
            }
            const int st = p_it % ns, use = p_it / ns;
            if (use > 0) mbar_wait(&empty[st], (use - 1) & 1);
            uint8_t *stage = ring + (size_t)st * p.stage_bytes;
            const uint8_t *wbase = Wb + (size_t)(rt * GT_M) * p.rb + (size_t)p_b * p.bbytes;
            for (int c = threadIdx.x; c < GT_M * CPR; c += G_THREADS) {
                const int r = c / CPR, ch = c % CPR;
                const uint8_t *src = wbase + (size_t)r * p.rb;
                src -= (uintptr_t)src & 15;                       // the piece keeps its 16-byte phase inside the stage row
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(stage + (size_t)r * p.rstride + ch * 16)), "l"(src + ch * 16) : "memory");
            }
            asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(&full[st])) : "memory");
            if (threadIdx.x == 0) {
                mbar_arrive_expect_tx(&full[st], ibytes);
                bulk_g2s(stage + p.a_bytes, p.img + ((size_t)tt * p.nsb + p_b) * ibytes, ibytes, &full[st]);
            }
            p_it++;
            if (++p_b >= p_b1) {
                p_item += gridDim.x;
                if (p_item < p.nitems) { const int ks = p_item % p.ksplit; p_b = ks * p.sb_per_split; p_b1 = min(p.nsb, p_b + p.sb_per_split); }
            }
        }
    };
    // ---------------------------------------------------------------- consumers: warp (wm, wn) owns rows wm*32.. (2 m-tiles) x tokens wn*64.. (8 n-tiles)
    const int wm = warp & 3, wn = warp >> 2;
    const int R = lane >> 2, cq = (lane & 3) * 2;
    int it = 0;
    for (int item = blockIdx.x; item < p.nitems; item += gridDim.x) {
        const int ks = item % p.ksplit, rt = (item / p.ksplit) % p.nrt, tt = item / (p.ksplit * p.nrt);
        const int sb0 = ks * p.sb_per_split, sb1 = min(p.nsb, sb0 + p.sb_per_split);
        const uint8_t *Wc = p.W;
        int g_first = 0, g_cnt = GT_N;
        if (p.g_E) {
            int e;
            g_lookup(p, tt, e, g_first, g_cnt);
            if (g_cnt == 0) continue;
            Wc += (size_t)e * p.g_expert_stride;
        }
        float out[2][NTW][4];
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
            for (int nt = 0; nt < NTW; nt++) out[mt][nt][0] = out[mt][nt][1] = out[mt][nt][2] = out[mt][nt][3] = 0.0f;
        for (int b = sb0; b < sb1; b++, it++) {
            const int st = it % ns;
            produce_upto(it + ns);
            mbar_wait(&full[st], (it / ns) & 1);
            const uint8_t *stage = ring + (size_t)st * p.stage_bytes;
            const uint8_t *bimg = stage + p.a_bytes;
            const uint32_t bq = smem_u32(bimg) + (uint32_t)(wn * (GT_N / 2)) * G_BSTRIDE;
            const float *bd = (const float *)(bimg + img_off_d());
            const int16_t *bs = (const int16_t *)(bimg + img_off_s(p.q8k));
            // B fragment address of this lane for ldmatrix.x4 over two n-tiles: matrix mi = lane >> 3 -> (n-tile pair member, k half)
            const uint32_t b_lane = bq + (uint32_t)(((lane >> 4) & 1) * 8 + (lane & 7)) * G_BSTRIDE + (uint32_t)((lane >> 3) & 1) * 16;
            const uint8_t *rowp[2][2];
#pragma unroll
            for (int mt = 0; mt < 2; mt++)
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int r = wm * 32 + mt * 16 + h * 8 + R;
                    const uintptr_t g = (uintptr_t)(Wc + (size_t)(rt * GT_M + r) * p.rb + (size_t)b * p.bbytes);
                    rowp[mt][h] = stage + (size_t)r * p.rstride + (g & 15);
                }
            sb_compute<TYPE, NTW>(rowp, b_lane, bd, bs, wn * (GT_N / 2), lane, out);
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[st]);
        }
        // ---- store the tile: rows rt*128 + wm*32 + mt*16 + h*8 + R, tokens tt*128 + wn*64 + nt*8 + cq + cc ----
        float *base = p.ksplit > 1 ? p.part + (size_t)ks * p.M * p.N : p.dst;
        const size_t stride = p.ksplit > 1 ? (size_t)p.N : p.dst_stride;
#pragma unroll
        for (int nt = 0; nt < NTW; nt++)
#pragma unroll
            for (int cc = 0; cc < 2; cc++) {
                const int tl = wn * (GT_N / 2) + nt * 8 + cq + cc, tok = tt * GT_N + tl;
                if (p.g_E) {
                    if (tl < g_cnt) {
                        const int pair = p.g_pairs[g_first + tl];
                        float *dp = p.dst + (size_t)(pair % p.g_n_used) * p.g_d_nb1 + (size_t)(pair / p.g_n_used) * p.g_d_nb2 + rt * GT_M + wm * 32 + R;
#pragma unroll
                        for (int mt = 0; mt < 2; mt++) { dp[mt * 16] = out[mt][nt][cc]; dp[mt * 16 + 8] = out[mt][nt][2 + cc]; }
                    }
                } else if (tok < p.M) {
                    float *dp = base + (size_t)tok * stride + rt * GT_M + wm * 32 + R;
#pragma unroll
                    for (int mt = 0; mt < 2; mt++) { dp[mt * 16] = out[mt][nt][cc]; dp[mt * 16 + 8] = out[mt][nt][2 + cc]; }
                }
            }
    }
}

__global__ void __launch_bounds__(256) b200_gemm_mma_reduce_kernel(const float *__restrict__ part, int ksplit, int N, int M, float *__restrict__ dst, size_t dst_stride) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)M * N) return;
    const int tok = (int)(i / N), n = (int)(i % N);
    float a = part[i];
    for (int z = 1; z < ksplit; z++) a += part[(size_t)z * M * N + i];
    dst[(size_t)tok * dst_stride + n] = a;
}

template <int TYPE>
int launch_g(b200_ctx *ctx, const GParams &p, int grid, size_t smem) {
    auto kern = b200_gemm_mma_kernel<TYPE>;
    static bool attr_set[16] = {false};
    if (!attr_set[ctx->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->smem_optin));
        attr_set[ctx->device & 15] = true;
    }
    kern<<<grid, G_THREADS, smem, ctx->stream>>>(p);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return B200_OK;
}
// stage geometry + grid shared by the dense and the grouped entry
static size_t gemm_geometry(b200_ctx *ctx, GParams &p) {
    const uint32_t ibytes = img_bytes(p.q8k);
    p.rstride = ((p.bbytes + 15u) & ~15u) + 16;            // >= 16 x chunks per row piece (gemm kernel CPR)
    p.a_bytes = (GT_M * p.rstride + 127u) & ~127u;
    p.stage_bytes = p.a_bytes + ibytes;
    int ns = (int)((ctx->smem_optin - 128) / p.stage_bytes);
    if (ns > 4) ns = 4;
    p.nstages = ns;
    return ns < 2 ? 0 : 128 + (size_t)ns * p.stage_bytes;
}

}  // namespace

bool gemm_mma_supported(int type, int64_t N, int64_t K, int64_t M) {
    if (!b200_type_is_quant(type) || getenv("GGML_B200_NO_GEMM_MMA")) return false;
    return N % GT_M == 0 && K % 256 == 0 && M >= 1;
}

// dst[tok * dst_stride + n] = sum_k W[n, k] * x[k, tok]; x f32 with column stride x_stride bytes
int gemm_mma_run(b200_ctx *ctx, int type, const uint8_t *W, size_t rb, int64_t N, int64_t K, const float *x, size_t x_stride, int64_t M, float *dst, size_t dst_stride) {
    if (!gemm_mma_supported(type, N, K, M)) { b200_set_error("gemm_mma: unsupported shape"); return B200_ERR_UNSUPPORTED; }
    GParams p = {};
    p.W = W; p.rb = (uint32_t)rb; p.type = type; p.N = (int)N; p.K = (int)K; p.M = (int)M; p.q8k = b200_act_mode_q8k(type);
    p.bbytes = type == B200_TYPE_Q4_K ? 144u : type == B200_TYPE_Q5_K ? 176u : type == B200_TYPE_Q6_K ? 210u : type == B200_TYPE_Q4_0 ? 144u : 272u;
    p.tn = GT_N;
    p.nsb = (int)(K / 256); p.ntile = (int)((M + GT_N - 1) / GT_N); p.nrt = (int)(N / GT_M);
    p.dst = dst; p.dst_stride = dst_stride;
    const uint32_t ibytes = img_bytes(p.q8k);
    uint8_t *img = (uint8_t *)ctx->get_scratch(SCRATCH_ACT, (size_t)p.ntile * p.nsb * ibytes);
    if (!img) return B200_ERR_ALLOC;
    p.img = img;
    {
        const int64_t warps = (int64_t)p.ntile * GT_N * p.nsb;
        b200_gemm_mma_pack_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, ctx->stream>>>(x, x_stride, (int)K, (int)M, p.q8k, p.nsb, img);
        ctx->launches++;
        CUDA_TRY(cudaGetLastError());
    }
    const size_t smem = gemm_geometry(ctx, p);
    if (!smem) { b200_set_error("gemm_mma: shared memory"); return B200_ERR_FAILED; }
    // split K when the tile grid would leave most of the machine idle (slices of >= 4 super-blocks); partials reduced in slice order
    const int64_t tiles = (int64_t)p.nrt * p.ntile;
    int ksplit = 1;
    while (ksplit < 8 && tiles * ksplit * 2 <= ctx->sm_count && p.nsb / (ksplit * 2) >= 4) ksplit *= 2;
    p.sb_per_split = (p.nsb + ksplit - 1) / ksplit;
    p.ksplit = (p.nsb + p.sb_per_split - 1) / p.sb_per_split;
    if (p.ksplit > 1) {
        p.part = (float *)ctx->get_scratch(SCRATCH_MISC, (size_t)p.ksplit * M * N * 4);
        if (!p.part) return B200_ERR_ALLOC;
    }
    p.nitems = (int)(tiles * p.ksplit);
    const int grid = p.nitems < ctx->sm_count ? p.nitems : ctx->sm_count;
    int rc;
    switch (type) {
        case B200_TYPE_Q4_K: rc = launch_g<B200_TYPE_Q4_K>(ctx, p, grid, smem); break;
        case B200_TYPE_Q5_K: rc = launch_g<B200_TYPE_Q5_K>(ctx, p, grid, smem); break;
        case B200_TYPE_Q6_K: rc = launch_g<B200_TYPE_Q6_K>(ctx, p, grid, smem); break;
        case B200_TYPE_Q4_0: rc = launch_g<B200_TYPE_Q4_0>(ctx, p, grid, smem); break;
        default:             rc = launch_g<B200_TYPE_Q8_0>(ctx, p, grid, smem); break;
    }
    if (rc || p.ksplit == 1) return rc;
    const int64_t total = M * N;
    b200_gemm_mma_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(p.part, p.ksplit, (int)N, (int)M, dst, dst_stride);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return B200_OK;
}

// MUL_MAT_ID for prompt batches: the (token, slot) pairs counting-sorted by expert on the device (mulmat.cu) become token tiles of <= 128
// pairs per expert; every tile runs the same GEMM against its expert's matrix.  g.max_chunks: upper bound of sum_e ceil(count_e / 128).
int gemm_mma_run_grouped(b200_ctx *ctx, int type, const uint8_t *W, size_t rb, int64_t N, int64_t K, const float *x, size_t x_stride, const MmGroupDesc &g, float *dst) {
    GParams p = {};
    p.W = W; p.rb = (uint32_t)rb; p.type = type; p.N = (int)N; p.K = (int)K; p.M = 0; p.q8k = b200_act_mode_q8k(type);
    p.bbytes = type == B200_TYPE_Q4_K ? 144u : type == B200_TYPE_Q5_K ? 176u : type == B200_TYPE_Q6_K ? 210u : type == B200_TYPE_Q4_0 ? 144u : 272u;
    p.tn = GT_N;
    p.nsb = (int)(K / 256); p.ntile = g.max_chunks; p.nrt = (int)(N / GT_M);
    p.dst = dst;
    p.g_off = g.off; p.g_pairs = g.pairs; p.g_E = g.E; p.g_n_used = g.n_used; p.g_b_ne1 = g.b_ne1; p.g_chunks = g.max_chunks;
    p.g_expert_stride = g.expert_stride; p.g_d_nb1 = g.d_nb1; p.g_d_nb2 = g.d_nb2;
    const uint32_t ibytes = img_bytes(p.q8k);
    uint8_t *img = (uint8_t *)ctx->get_scratch(SCRATCH_ACT, (size_t)p.ntile * p.nsb * ibytes);
    if (!img) return B200_ERR_ALLOC;
    p.img = img;
    {
        const int64_t warps = (int64_t)p.ntile * GT_N * p.nsb;
        b200_gemm_mma_pack_grouped_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, ctx->stream>>>(x, x_stride, p, img);
        ctx->launches++;
        CUDA_TRY(cudaGetLastError());
    }
    const size_t smem = gemm_geometry(ctx, p);
    if (!smem) { b200_set_error("gemm_mma: shared memory"); return B200_ERR_FAILED; }
    p.ksplit = 1; p.sb_per_split = p.nsb;
    p.nitems = p.nrt * p.ntile;
    const int grid = p.nitems < ctx->sm_count ? p.nitems : ctx->sm_count;
    switch (type) {
        case B200_TYPE_Q4_K: return launch_g<B200_TYPE_Q4_K>(ctx, p, grid, smem);
        case B200_TYPE_Q5_K: return launch_g<B200_TYPE_Q5_K>(ctx, p, grid, smem);
        case B200_TYPE_Q6_K: return launch_g<B200_TYPE_Q6_K>(ctx, p, grid, smem);
        case B200_TYPE_Q4_0: return launch_g<B200_TYPE_Q4_0>(ctx, p, grid, smem);
        default:             return launch_g<B200_TYPE_Q8_0>(ctx, p, grid, smem);
    }
}
