// float_mm.h -- host interface of the F16/BF16 weight matmuls: the weight-streaming mma.sync kernel for up to 32 token columns
// (gemv_f16.cu) and the tcgen05 GEMM for more (gemm_f16_tc.cu).  Both round x to the weight's 16-bit type (the CPU's vec_dot_type)
// once and accumulate exact products in f32.  Both have a grouped mode for MUL_MAT_ID over expert-sorted (token, slot) pairs.
#pragma once
#include "common.cuh"
#include <cuda.h>

// token columns up to which the streaming kernel runs; above, the tcgen05 GEMM (profiles/float_weights.md)
constexpr int64_t F16MM_STREAM_MAX_M = 32;

// 2-D tensor map over a row-major [outer][inner] matrix of 16-bit elements (row pitch inner * 2 bytes), SWIZZLE_128B boxes of
// box_inner (64) x box_outer; encoded through the driver entry point (the library does not link libcuda)
int make_tmap_16bit(CUtensorMap *map, int type, const void *base, int64_t inner, int64_t outer, uint32_t box_inner, uint32_t box_outer);
// 3-D variant over `depth` such matrices `depth_stride` bytes apart (16-byte multiple), box depth 1: a stack of MoE expert matrices,
// each zero-filled past its own last row
int make_tmap_16bit_3d(CUtensorMap *map, int type, const void *base, int64_t inner, int64_t outer, int64_t depth, size_t depth_stride,
                       uint32_t box_inner, uint32_t box_outer);
// dst[col * dst_stride + n] = sum_k W[n, k] * round16(x[col][k]) for ncols <= 32 columns; W rows contiguous, 16-byte aligned, K % 8 == 0
int gemv_f16_run(b200_ctx *ctx, int type, const uint16_t *W, int64_t N, int64_t K, const float *x, size_t x_stride_bytes, int ncols, float *dst,
                 size_t dst_stride, bool w_const);
// the same for any M (prompt batches): x packed to a rounded [M][K] image, tcgen05.mma kind::f16 over TMA-loaded tiles
int gemm_f16_tc_run(b200_ctx *ctx, int type, const uint16_t *W, int64_t N, int64_t K, const float *x, size_t x_stride_bytes, int64_t M, float *dst,
                    size_t dst_stride);

// MUL_MAT_ID over (token, slot) pairs counting-sorted by expert on the device (g: b200_moe_group_kernel's tables, g.max_chunks the grid's
// upper bound of chunks): dst[:, slot, tok] = As[expert] . round16(x[:, column(pair)]), column = tok (g.b_ne1 == 1) or the pair itself,
// x_stride_bytes the byte stride of those columns; As: E matrices of N contiguous rows of K, g.expert_stride bytes apart (16-byte
// multiple).  npairs: n_used * n_tok, the most pairs the tables can hold.
// Chunks of <= 32 pairs through the weight-streaming kernel (gemv_f16.cu)
int gemv_f16_run_grouped(b200_ctx *ctx, int type, const uint16_t *As, int64_t N, int64_t K, const float *x, size_t x_stride_bytes, const MmGroupDesc &g,
                         int64_t npairs, float *dst);
// chunks of <= 128 pairs through the tcgen05 GEMM over a pair-sorted rounded image (gemm_f16_tc.cu)
int gemm_f16_tc_run_grouped(b200_ctx *ctx, int type, const uint16_t *As, int64_t N, int64_t K, const float *x, size_t x_stride_bytes, const MmGroupDesc &g,
                            int64_t npairs, float *dst);
// split-K partials of both grouped paths, part[slice][sorted pair][N] -> dst, summed in slice order (gemv_f16.cu)
int launch_f16_grouped_reduce(b200_ctx *ctx, const float *part, int nslices, int64_t N, const MmGroupDesc &g, int64_t npairs, float *dst, int use_pdl);
