// gemv.h -- host-side interface of the decode GEMV (gemv.cu), shared with mulmat.cu and graph.cu
#pragma once
#include "common.cuh"

constexpr int GEMV_MAX_SEG = 3;
enum { ACT_PREQ = 0, ACT_F32 = 1, ACT_F32_NORM = 2, ACT_F32_SWIGLU = 3 };

// one weight matrix of a launch ("segment"): dst[:, col] = W . act[:, col] (+ residual)
struct GemvSegDesc {
    int            type;
    const uint8_t *W;
    size_t         rb;               // bytes per row
    int64_t        N;                // rows
    float *        dst;
    size_t         dst_stride;       // elements between columns
    const float *  residual;         // optional, laid out like dst
    const int32_t *expert_id;        // MUL_MAT_ID: device pointer to the expert index
    size_t         expert_stride;    // bytes between expert matrices
    int32_t *      dbgP, *dbgM;      // block-sum test hook
};
// where the activations come from
struct GemvActDesc {
    int            mode;             // ACT_*
    const uint8_t *act;              // ACT_PREQ: pre-quantised scratch (ActLayout)
    const float *  x;                // f32 source, column stride x_stride bytes
    size_t         x_stride;
    const float *  x2;               // ACT_F32_NORM: norm weight [K]; ACT_F32_SWIGLU: `up` (strided like x)
    float          eps;
};

// L2 look-ahead: constant weight ranges of the launches that follow this one (graph.cu fills them in)
constexpr int GEMV_MAX_PF = 4;
struct GemvPf { const void *ptr; size_t bytes; };

int gemv_launch(b200_ctx *ctx, const GemvSegDesc *segs, int nseg, int64_t K, const GemvActDesc &ga, int ncols, bool w_const,
                const GemvPf *pf, int npf, bool *pair = nullptr);
// `pair` (FFN gate|up launch, 2 segments): request the paired epilogue -- h = silu(seg0 row) * seg1 row written to seg[0].dst and NOTHING
// else; *pair tells the caller whether the launch did it (only the batch-1 kernel can), so that the down projection reads h directly
// batch-1 K-quant kernel (gemv_bs1.cu): 1 = launched, 0 = not eligible, < 0 = error
int gemv_bs1_try_launch(b200_ctx *ctx, const GemvSegDesc *segs, int nseg, int64_t K, const GemvActDesc &ga, bool w_const,
                        const GemvPf *pf, int npf, int l2pf, bool *pair = nullptr);
int gemv_max_cols(const b200_ctx *ctx, int type, size_t rb, int64_t K);
