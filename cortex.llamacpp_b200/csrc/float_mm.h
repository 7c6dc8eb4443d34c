// float_mm.h -- host interface of the F16/BF16 weight matmuls: the weight-streaming mma.sync kernel for up to 32 token columns
// (gemv_f16.cu) and the tcgen05 GEMM for more (gemm_f16_tc.cu).  Both round x to the weight's 16-bit type (the CPU's vec_dot_type)
// once and accumulate exact products in f32.
#pragma once
#include "common.cuh"
#include <cuda.h>

// token columns up to which the streaming kernel runs; above, the tcgen05 GEMM (profiles/float_weights.md)
constexpr int64_t F16MM_STREAM_MAX_M = 32;

// 2-D tensor map over a row-major [outer][inner] matrix of 16-bit elements (row pitch inner * 2 bytes), SWIZZLE_128B boxes of
// box_inner (64) x box_outer; encoded through the driver entry point (the library does not link libcuda)
int make_tmap_16bit(CUtensorMap *map, int type, const void *base, int64_t inner, int64_t outer, uint32_t box_inner, uint32_t box_outer);
// dst[col * dst_stride + n] = sum_k W[n, k] * round16(x[col][k]) for ncols <= 32 columns; W rows contiguous, 16-byte aligned, K % 8 == 0
int gemv_f16_run(b200_ctx *ctx, int type, const uint16_t *W, int64_t N, int64_t K, const float *x, size_t x_stride_bytes, int ncols, float *dst,
                 size_t dst_stride, bool w_const);
// the same for any M (prompt batches): x packed to a rounded [M][K] image, tcgen05.mma kind::f16 over TMA-loaded tiles
int gemm_f16_tc_run(b200_ctx *ctx, int type, const uint16_t *W, int64_t N, int64_t K, const float *x, size_t x_stride_bytes, int64_t M, float *dst,
                    size_t dst_stride);
