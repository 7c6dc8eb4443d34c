// gemm_f16_tc.cu -- F16/BF16 weight matmul for prompt batches (more than 32 token columns) on the 5th-generation tensor cores:
// tcgen05.mma cta_group::1 kind::f16 with f16 or bf16 operands (chosen by the instruction descriptor), f32 accumulators in TMEM.
//   * x is rounded once per matmul to the weight's 16-bit type (the CPU's vec_dot_type, round-to-nearest-even) by a pack kernel that
//     writes a dense [M][K] image into context scratch;
//   * both operands come in through 2-D TMA tensor maps (SWIZZLE_128B, K-major, 64 k per stage): the weight tile of 128 rows straight
//     from the GGUF rows, the activation tile of 128 tokens from the image.  The tensor maps' zero fill covers the N, M and K tails;
//   * warp-specialised CTA of one 128 x 128 output tile: warp 0 issues the TMA loads into a ring of operand stages (full / empty
//     mbarriers), warp 1 allocates TMEM and issues 4 MMAs of K = 16 per stage from one elected lane, warps 2..5 drain the accumulator
//     (tcgen05.ld) and store f32;
//   * when the tile grid leaves most SMs idle, K is split into slices whose partials a second kernel adds in slice order
//     (deterministic).
//   * grouped mode (MUL_MAT_ID): the image holds the (token, slot) pairs sorted by expert, a token tile is a chunk of <= 128 pairs of
//     one expert and the weight tile comes from a 3-D (K, N, expert) map; only the chunk's pairs are stored.
// Products of two 16-bit floats are exact in f32: the result differs from the CPU only in the order of the f32 additions.
// Roofline: tensor pipe for prompt batches; algorithmic work 2 N K M flops, bytes 2 N K + 4 M K + 4 M N.
#include "float_mm.h"
#include "tc05.cuh"
#include <cuda_bf16.h>
#include <algorithm>

namespace {

constexpr int FT_M = 128, FT_N = 128, FT_K = 64;                 // weight rows, token columns, k per stage
constexpr uint32_t FT_TILE = FT_M * FT_K * 2;                     // 16 KB per operand tile
constexpr int FT_THREADS = 6 * 32;
constexpr int FT_MAX_STAGES = 8;

struct FtParams {
    int N, M, K;
    float *dst; size_t dst_stride;
    float *part;                        // [ksplit][M][N] when gridDim.z > 1
    int st_per_split, nst, nstages;     // k stages per slice, in all
    // grouped (MUL_MAT_ID) mode: blockIdx.y = chunk of <= 128 pairs of one expert, M = the pair-sorted image's rows
    const int32_t *g_off, *g_pairs; int g_E, g_n_used; size_t g_d_nb1, g_d_nb2;
};

// grouped mode: chunk -> (expert, first sorted pair = image row, pairs in the chunk); cnt = 0: the chunk does not exist
__device__ __forceinline__ void ft_chunk(const FtParams &p, int chunk, int &e, int &first, int &cnt) {
    cnt = 0; first = 0;
    for (e = 0; e < p.g_E; e++) {
        const int o0 = p.g_off[e], n = p.g_off[e + 1] - o0, nch = (n + FT_N - 1) / FT_N;
        if (chunk < nch) { first = o0 + chunk * FT_N; cnt = min(FT_N, n - chunk * FT_N); return; }
        chunk -= nch;
    }
}

struct FtBars { uint64_t full[FT_MAX_STAGES], empty[FT_MAX_STAGES], acc_full; uint32_t tmem_base; };

// G: grouped mode (MUL_MAT_ID); the dense instantiation compiles none of its branches
template <bool BF, bool G>
__device__ __forceinline__ void ft_body(const CUtensorMap &tmw, const CUtensorMap &tmx, const FtParams &p) {
    extern __shared__ uint8_t ft_smem_raw[];
    uint8_t *smem = ft_smem_raw + ((1024u - (smem_u32(ft_smem_raw) & 1023u)) & 1023u);      // SWIZZLE_128B tiles: 1024-byte aligned
    const int ns = p.nstages;
    FtBars *S = (FtBars *)(smem + (size_t)ns * 2 * FT_TILE);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row0 = blockIdx.x * FT_M;
    int tok0 = blockIdx.y * FT_N, e = 0, cnt = 0;
    if constexpr (G) {
        ft_chunk(p, blockIdx.y, e, tok0, cnt);
        if (cnt == 0) return;
    }
    const int st0 = blockIdx.z * p.st_per_split, nst = min(p.st_per_split, p.nst - st0);
    if (threadIdx.x == 0) {
        for (int i = 0; i < ns; i++) { mbar_init(&S->full[i], 1); mbar_init(&S->empty[i], 1); }
        mbar_init(&S->acc_full, 1);
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc(&S->tmem_base, FT_N);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = S->tmem_base;

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer: weight tile + activation tile per stage
        for (int i = 0; i < nst; i++) {
            const int st = i % ns, use = i / ns;
            if (use > 0) mbar_wait_bounded(&S->empty[st], (use - 1) & 1);
            if (elect_one_sync()) {
                uint8_t *a = smem + (size_t)st * 2 * FT_TILE;
                mbar_arrive_expect_tx(&S->full[st], 2 * FT_TILE);
                if constexpr (G) tma_load_3d(a, &tmw, (st0 + i) * FT_K, row0, e, &S->full[st]);
                else tma_load_2d(a, &tmw, (st0 + i) * FT_K, row0, &S->full[st]);
                tma_load_2d(a + FT_TILE, &tmx, (st0 + i) * FT_K, tok0, &S->full[st]);
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer (warp-uniform loop, one elected lane issues)
        constexpr uint32_t idesc = idesc_f16(BF, FT_M, FT_N);
        const uint32_t base = smem_u32(smem);
        for (int i = 0; i < nst; i++) {
            const int st = i % ns, use = i / ns;
            mbar_wait_bounded(&S->full[st], use & 1);
            tc_fence_after();
            if (elect_one_sync()) {
                const uint32_t a = base + (uint32_t)st * 2 * FT_TILE, b = a + FT_TILE;
#pragma unroll
                for (int k = 0; k < FT_K / 16; k++)
                    mma_f16(tmem, make_desc_sw128(a + 32 * k), make_desc_sw128(b + 32 * k), idesc, (i | k) ? 1u : 0u);
                tc_commit(&S->empty[st]);                      // the stage is free once these MMAs have read it
                if (i == nst - 1) tc_commit(&S->acc_full);     // the accumulator is complete
            }
            __syncwarp();
        }
    } else {
        // ------------------------------------------------------------ drain: TMEM lane = weight row, column = token
        const int q = warp & 3, row = row0 + q * 32 + lane;
        mbar_wait_bounded(&S->acc_full, 0);
        tc_fence_after();
        float *const dstv = gridDim.z > 1 ? p.part + (size_t)blockIdx.z * p.M * p.N : p.dst;
        const size_t stride = gridDim.z > 1 ? (size_t)p.N : p.dst_stride;
#pragma unroll 1
        for (int c0 = 0; c0 < FT_N; c0 += 32) {
            uint32_t v[32];
            tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
            tmem_ld_wait();
            if (row < p.N)
#pragma unroll
                for (int j = 0; j < 32; j++) {
                    const int tok = tok0 + c0 + j;
                    if constexpr (G) {               // only the chunk's pairs: partials in sorted order, results to (slot, token)
                        if (c0 + j >= cnt) continue;
                        if (gridDim.z > 1) { dstv[(size_t)tok * stride + row] = __uint_as_float(v[j]); continue; }
                        const int pair = p.g_pairs[tok];
                        p.dst[(size_t)(pair % p.g_n_used) * p.g_d_nb1 + (size_t)(pair / p.g_n_used) * p.g_d_nb2 + row] = __uint_as_float(v[j]);
                    } else if (tok < p.M) dstv[(size_t)tok * stride + row] = __uint_as_float(v[j]);
                }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, FT_N);
}

template <bool BF>
__global__ void __launch_bounds__(FT_THREADS, 1) b200_gemm_f16_tc_kernel(const __grid_constant__ CUtensorMap tmw, const __grid_constant__ CUtensorMap tmx,
                                                                         const FtParams p) {
    ft_body<BF, false>(tmw, tmx, p);
}
// MUL_MAT_ID: blockIdx.y = chunk of <= 128 pairs of one expert; tmw is the 3-D (K, N, expert) map, tmx the pair-sorted image
template <bool BF>
__global__ void __launch_bounds__(FT_THREADS, 1) b200_gemm_f16_tc_grouped_kernel(const __grid_constant__ CUtensorMap tmw, const __grid_constant__ CUtensorMap tmx,
                                                                                 const FtParams p) {
    ft_body<BF, true>(tmw, tmx, p);
}

// 8 floats -> 8 16-bit values (round-to-nearest-even)
template <bool BF>
__device__ __forceinline__ uint4 round8(const float4 a, const float4 b) {
    uint32_t o[4];
    if (BF) {
        __nv_bfloat162 h[4] = {__floats2bfloat162_rn(a.x, a.y), __floats2bfloat162_rn(a.z, a.w), __floats2bfloat162_rn(b.x, b.y), __floats2bfloat162_rn(b.z, b.w)};
        for (int j = 0; j < 4; j++) o[j] = *(uint32_t *)&h[j];
    } else {
        __half2 h[4] = {__floats2half2_rn(a.x, a.y), __floats2half2_rn(a.z, a.w), __floats2half2_rn(b.x, b.y), __floats2half2_rn(b.z, b.w)};
        for (int j = 0; j < 4; j++) o[j] = *(uint32_t *)&h[j];
    }
    return make_uint4(o[0], o[1], o[2], o[3]);
}

// x f32 [M] columns (stride x_stride floats) -> [M][K] image of 16-bit values, 8 elements per thread
template <bool BF>
__global__ void __launch_bounds__(256) b200_gemm_f16_pack_kernel(const float *__restrict__ x, size_t x_stride, int K, int M, uint16_t *__restrict__ img) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, k8 = K / 8;
    if (i >= (int64_t)M * k8) return;
    const int64_t m = i / k8, k = (i % k8) * 8;
    const float4 a = *(const float4 *)(x + m * x_stride + k), b = *(const float4 *)(x + m * x_stride + k + 4);
    *(uint4 *)(img + m * (int64_t)K + k) = round8<BF>(a, b);
}

// grouped: row q of the image = the column of sorted pair q (its token's when b_ne1 == 1); rows past the routed pairs (off[E]) untouched
template <bool BF>
__global__ void __launch_bounds__(256) b200_gemm_f16_pack_grouped_kernel(const float *__restrict__ x, size_t x_stride, int K, const int32_t *off,
                                                                         const int32_t *pairs, int E, int n_used, int b_ne1, uint16_t *__restrict__ img) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, k8 = K / 8;
    if (i >= (int64_t)off[E] * k8) return;
    const int64_t q = i / k8, k = (i % k8) * 8;
    const int pair = pairs[q];
    const float *xp = x + (int64_t)(b_ne1 == 1 ? pair / n_used : pair) * x_stride + k;
    *(uint4 *)(img + q * (int64_t)K + k) = round8<BF>(*(const float4 *)xp, *(const float4 *)(xp + 4));
}

// dst[tok][n] = sum over the K slices in slice order (deterministic)
__global__ void __launch_bounds__(256) b200_gemm_f16_reduce_kernel(const float *__restrict__ part, int ksplit, int N, int M, float *__restrict__ dst, size_t dst_stride) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)M * N) return;
    float a = part[i];
    for (int z = 1; z < ksplit; z++) a += part[(size_t)z * M * N + i];
    dst[(i / N) * dst_stride + i % N] = a;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

template <bool BF, bool G>
int launch_ft(b200_ctx *ctx, const CUtensorMap &tw, const CUtensorMap &tx, const FtParams &p, dim3 grid, size_t smem) {
    auto kern = G ? b200_gemm_f16_tc_grouped_kernel<BF> : b200_gemm_f16_tc_kernel<BF>;
    static bool attr_set[16] = {false};
    if (!attr_set[ctx->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->smem_optin));
        attr_set[ctx->device & 15] = true;
    }
    kern<<<grid, FT_THREADS, smem, ctx->stream>>>(tw, tx, p);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return B200_OK;
}

// stage ring and split-K of a grid of `tiles` (weight-row tile, token tile) CTAs; p.nst must be set.  Returns the slice count.
int ft_plan(b200_ctx *ctx, FtParams &p, int64_t tiles, size_t &smem) {
    const size_t fixed = 1024 + sizeof(FtBars);
    p.nstages = (int)std::min<size_t>(FT_MAX_STAGES, (ctx->smem_optin - fixed) / (2 * FT_TILE));
    // split K when the tile grid covers less than half of the SMs: slices of >= 8 stages (512 k), partials reduced in slice order
    int ksplit = 1;
    while (ksplit < 8 && tiles * ksplit * 2 <= ctx->sm_count && p.nst / (ksplit * 2) >= 8) ksplit *= 2;
    p.st_per_split = (p.nst + ksplit - 1) / ksplit;
    smem = fixed + (size_t)p.nstages * 2 * FT_TILE;
    return (p.nst + p.st_per_split - 1) / p.st_per_split;
}

EncodeTiledFn tmap_encoder() {
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn) {
            cudaGetLastError();
            b200_set_error("cuTensorMapEncodeTiled: driver entry point not found");
            return nullptr;
        }
        encode = (EncodeTiledFn)fn;
    }
    return encode;
}

int encode_16bit(CUtensorMap *map, int type, const void *base, int rank, const cuuint64_t *dims, const cuuint64_t *strides, const cuuint32_t *box) {
    const EncodeTiledFn encode = tmap_encoder();
    if (!encode) return B200_ERR_FAILED;
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = encode(map, type == B200_TYPE_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, const_cast<void *>(base), dims,
                              strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        b200_set_error("cuTensorMapEncodeTiled failed (%d): %lld x %lld x %lld", (int)r, (long long)dims[0], (long long)dims[1], rank > 2 ? (long long)dims[2] : 1LL);
        return B200_ERR_FAILED;
    }
    return B200_OK;
}

}  // namespace

int make_tmap_16bit(CUtensorMap *map, int type, const void *base, int64_t inner, int64_t outer, uint32_t box_inner, uint32_t box_outer) {
    const cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer}, strides[1] = {(cuuint64_t)inner * 2};
    const cuuint32_t box[2] = {box_inner, box_outer};
    return encode_16bit(map, type, base, 2, dims, strides, box);
}

int make_tmap_16bit_3d(CUtensorMap *map, int type, const void *base, int64_t inner, int64_t outer, int64_t depth, size_t depth_stride,
                       uint32_t box_inner, uint32_t box_outer) {
    const cuuint64_t dims[3] = {(cuuint64_t)inner, (cuuint64_t)outer, (cuuint64_t)depth}, strides[2] = {(cuuint64_t)inner * 2, (cuuint64_t)depth_stride};
    const cuuint32_t box[3] = {box_inner, box_outer, 1};
    return encode_16bit(map, type, base, 3, dims, strides, box);
}

int gemm_f16_tc_run(b200_ctx *ctx, int type, const uint16_t *W, int64_t N, int64_t K, const float *x, size_t x_stride_bytes, int64_t M, float *dst,
                    size_t dst_stride) {
    if ((type != B200_TYPE_F16 && type != B200_TYPE_BF16) || M < 1 || N < 1 || K % 8 || ((uintptr_t)W & 15) || ((uintptr_t)x & 15) || (x_stride_bytes & 15) ||
        N > INT32_MAX || K > INT32_MAX || M > INT32_MAX) {
        b200_set_error("gemm_f16_tc: unsupported shape");
        return B200_ERR_UNSUPPORTED;
    }
    const bool bf = type == B200_TYPE_BF16;
    uint16_t *img = (uint16_t *)ctx->get_scratch(SCRATCH_ACT, (size_t)M * K * 2);
    if (!img) return B200_ERR_ALLOC;
    {
        const int64_t n = M * (K / 8);
        if (bf) b200_gemm_f16_pack_kernel<true><<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(x, x_stride_bytes / 4, (int)K, (int)M, img);
        else    b200_gemm_f16_pack_kernel<false><<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(x, x_stride_bytes / 4, (int)K, (int)M, img);
        ctx->launches++;
        CUDA_TRY(cudaGetLastError());
    }
    CUtensorMap tw, tx;
    int rc = make_tmap_16bit(&tw, type, W, K, N, FT_K, FT_M);
    if (!rc) rc = make_tmap_16bit(&tx, type, img, K, M, FT_K, FT_N);
    if (rc) return rc;
    FtParams p = {};
    p.N = (int)N; p.M = (int)M; p.K = (int)K; p.dst = dst; p.dst_stride = dst_stride;
    p.nst = (int)((K + FT_K - 1) / FT_K);
    size_t smem = 0;
    const int ksplit = ft_plan(ctx, p, ((N + FT_M - 1) / FT_M) * ((M + FT_N - 1) / FT_N), smem);
    if (ksplit > 1) {
        p.part = (float *)ctx->get_scratch(SCRATCH_MISC, (size_t)ksplit * M * N * 4);
        if (!p.part) return B200_ERR_ALLOC;
    }
    const dim3 grid((unsigned)((N + FT_M - 1) / FT_M), (unsigned)((M + FT_N - 1) / FT_N), (unsigned)ksplit);
    rc = bf ? launch_ft<true, false>(ctx, tw, tx, p, grid, smem) : launch_ft<false, false>(ctx, tw, tx, p, grid, smem);
    if (rc || ksplit == 1) return rc;
    const int64_t total = M * N;
    b200_gemm_f16_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(p.part, ksplit, (int)N, (int)M, dst, dst_stride);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return B200_OK;
}

// the pairs of every expert, sorted by the grouping kernel, form chunks of <= 128 rows of a pair-sorted rounded image; each (weight-row
// tile, chunk) CTA multiplies a 128-row box of the image at the chunk's first row (rows past the chunk are multiplied but never stored)
// against its expert's weight tile.  The grid covers g.max_chunks chunks; the ones beyond the routed count exit at once.
int gemm_f16_tc_run_grouped(b200_ctx *ctx, int type, const uint16_t *As, int64_t N, int64_t K, const float *x, size_t x_stride_bytes, const MmGroupDesc &g,
                            int64_t npairs, float *dst) {
    if ((type != B200_TYPE_F16 && type != B200_TYPE_BF16) || npairs < 1 || N < 1 || K % 8 || (((uintptr_t)As | g.expert_stride | (uintptr_t)x | x_stride_bytes) & 15) ||
        N > INT32_MAX || K > INT32_MAX || npairs > INT32_MAX || g.max_chunks < 1) {
        b200_set_error("gemm_f16_tc grouped: unsupported shape");
        return B200_ERR_UNSUPPORTED;
    }
    const bool bf = type == B200_TYPE_BF16;
    uint16_t *img = (uint16_t *)ctx->get_scratch(SCRATCH_ACT, (size_t)npairs * K * 2);
    if (!img) return B200_ERR_ALLOC;
    {
        const int64_t n = npairs * (K / 8);
        const unsigned blocks = (unsigned)((n + 255) / 256);
        if (bf) b200_gemm_f16_pack_grouped_kernel<true><<<blocks, 256, 0, ctx->stream>>>(x, x_stride_bytes / 4, (int)K, g.off, g.pairs, g.E, g.n_used, g.b_ne1, img);
        else    b200_gemm_f16_pack_grouped_kernel<false><<<blocks, 256, 0, ctx->stream>>>(x, x_stride_bytes / 4, (int)K, g.off, g.pairs, g.E, g.n_used, g.b_ne1, img);
        ctx->launches++;
        CUDA_TRY(cudaGetLastError());
    }
    CUtensorMap tw, tx;
    int rc = make_tmap_16bit_3d(&tw, type, As, K, N, g.E, g.expert_stride, FT_K, FT_M);
    if (!rc) rc = make_tmap_16bit(&tx, type, img, K, npairs, FT_K, FT_N);
    if (rc) return rc;
    FtParams p = {};
    p.N = (int)N; p.M = (int)npairs; p.K = (int)K; p.dst = dst;
    p.g_off = g.off; p.g_pairs = g.pairs; p.g_E = g.E; p.g_n_used = g.n_used; p.g_d_nb1 = g.d_nb1; p.g_d_nb2 = g.d_nb2;
    p.nst = (int)((K + FT_K - 1) / FT_K);
    size_t smem = 0;
    const int ksplit = ft_plan(ctx, p, ((N + FT_M - 1) / FT_M) * g.max_chunks, smem);
    if (ksplit > 1) {
        p.part = (float *)ctx->get_scratch(SCRATCH_MISC, (size_t)ksplit * npairs * N * 4);
        if (!p.part) return B200_ERR_ALLOC;
    }
    const dim3 grid((unsigned)((N + FT_M - 1) / FT_M), (unsigned)g.max_chunks, (unsigned)ksplit);
    rc = bf ? launch_ft<true, true>(ctx, tw, tx, p, grid, smem) : launch_ft<false, true>(ctx, tw, tx, p, grid, smem);
    if (rc || ksplit == 1) return rc;
    return launch_f16_grouped_reduce(ctx, p.part, ksplit, N, g, npairs, dst, 0);
}
