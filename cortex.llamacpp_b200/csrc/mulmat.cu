// mulmat.cu -- MUL_MAT / MUL_MAT_ID dispatch.
//
// Replaces ggml_cuda_mul_mat (ggml-cuda.cu:1845-1906) and ggml_cuda_mul_mat_id (:1962-2098).
// Semantics follow the CPU oracle (ggml_compute_forward_mul_mat, ggml-cpu.c:8708-8900): src1 rows are
// quantised to the weight type's vec_dot_type (q8_0 for Q4_0/Q8_0, q8_K for K-quants, f16/bf16 for
// 16-bit float weights) and every dst element is one dot product.
//   quantised W, M <= 4      : streaming GEMV, activation quantisation in its prologue (gemv.cu, gemv_bs1.cu)
//   quantised W, 5 <= M <= 32: quantise (quant.cu) + small-batch mma.sync kernel (gemv_mma.cu)
//   quantised W, M > 32      : K-quants: tcgen05 kind::f16 GEMM (gemm_tc.cu); other formats: prompt-batch GEMM on mma.sync (gemm_mma.cu);
//                              shapes neither takes (N % 128, K % 256): GEMV in column chunks
//   row-split W (B200_TENSOR_FLAG_SPLIT; quantised, F16, BF16): every shard's GPU at once (op_mul_mat_split)
//   F16/BF16 W, rows contiguous and 16-byte aligned, K % 8 == 0 (float_mm_ok):
//                       M <= 32: weight-streaming mma.sync kernel, x rounded to the weight type in its prologue (gemv_f16.cu)
//                       M > 32 : rounded x image + tcgen05 kind::f16 GEMM over TMA tiles (gemm_f16_tc.cu)
//   F32 W, other F16/BF16 layouts (strided or permuted views, odd K, unaligned operands): warp-per-row float kernel below
//   cpu_exact mode           : exact.cu (the reference AVX2 build's summation order)
// MUL_MAT_ID: device-side expert routing -- no host sync on `ids` (the reference copies ids to the host and loops experts there):
//   quantised experts: one GEMV per (token, slot) for decode-sized batches, pairs grouped by expert on the device + grouped gemv_mma for
//                      batches, grouped tile GEMMs for prompt batches;
//   F16/BF16 experts, rows contiguous and 16-byte aligned, K % 8 == 0, dense x (float_mm_id_ok): pairs grouped by expert on the device
//                      at every batch size, then < 32 pairs per expert on average: grouped weight-streaming kernel (gemv_f16.cu);
//                      more: grouped tcgen05 GEMM over a pair-sorted rounded image (gemm_f16_tc.cu);
//   F32 experts, other F16/BF16 layouts, cpu_exact mode: warp-per-(row, pair) float kernel reading the expert from ids on the device.
#include "common.cuh"
#include <algorithm>
#include <cuda_bf16.h>
#include "gemm_tc.h"
#include "float_mm.h"

int gemv_max_cols(const b200_ctx *ctx, int type, size_t rb, int64_t K);
int launch_gemv_f32(b200_ctx *ctx, int type, const uint8_t *W, size_t row_bytes, int64_t N, int64_t K, const float *x, size_t x_stride_bytes,
                    int ncols, float *dst, size_t dst_col_stride, bool w_const, int fuse_mode, const float *x2, float eps,
                    const float *residual);
int launch_gemv_expert(b200_ctx *ctx, int type, const uint8_t *W, size_t row_bytes, size_t expert_stride, const int32_t *expert_id, int64_t N,
                       int64_t K, const float *x, float *dst);

namespace {

// ---------------------------------------------------------------------------------------------------
// float weights: dst[n, m, i2, i3] = sum_k W[k, n, i2/r2, i3/r3] * x[k, m, i2, i3]; one warp per (n, m, batch)
// ---------------------------------------------------------------------------------------------------
template <typename WT> __device__ __forceinline__ float w_to_float(WT v);
template <> __device__ __forceinline__ float w_to_float<float>(float v) { return v; }
template <> __device__ __forceinline__ float w_to_float<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float w_to_float<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
// the CPU converts src1 to the weight's vec_dot_type before the dot
template <typename WT> __device__ __forceinline__ float x_round(float v);
template <> __device__ __forceinline__ float x_round<float>(float v) { return v; }
template <> __device__ __forceinline__ float x_round<__half>(float v) { return __half2float(__float2half_rn(v)); }
template <> __device__ __forceinline__ float x_round<__nv_bfloat16>(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

template <typename WT>
__global__ void __launch_bounds__(128) b200_mul_mat_float_kernel(b200_tensor w, b200_tensor x, b200_tensor d) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int64_t N = d.ne[0], M = d.ne[1];
    const int64_t total = N * M * d.ne[2] * d.ne[3];
    if (gw >= total) return;
    const int64_t n = gw % N, m = (gw / N) % M, i2 = (gw / (N * M)) % d.ne[2], i3 = gw / (N * M * d.ne[2]);
    const int64_t w2 = i2 / (d.ne[2] / w.ne[2]), w3 = i3 / (d.ne[3] / w.ne[3]);
    const char *wp = (const char *)w.data + n * w.nb[1] + w2 * w.nb[2] + w3 * w.nb[3];
    const char *xp = (const char *)x.data + m * x.nb[1] + i2 * x.nb[2] + i3 * x.nb[3];
    float acc = 0.0f;
    for (int64_t k = lane; k < w.ne[0]; k += 32) {
        const float wv = w_to_float<WT>(*(const WT *)(wp + k * w.nb[0]));
        const float xv = x_round<WT>(*(const float *)(xp + k * x.nb[0]));
        acc = fmaf(wv, xv, acc);
    }
    acc = warp_reduce_sum(acc);
    if (lane == 0) *(float *)((char *)d.data + n * d.nb[0] + m * d.nb[1] + i2 * d.nb[2] + i3 * d.nb[3]) = acc;
}

// cpu-exact mode, F32 weights (the MoE router): ggml_vec_dot_f32 of the AVX2 + FMA build (ggml-cpu.c:1454-1494): lane l of accumulator j
// owns elements 32i + 8j + l; 32 threads = the 4 x 8 accumulator lanes; GGML_F32x8_REDUCE; n % 32 leftovers as float mul + add
__global__ void __launch_bounds__(128) b200_mul_mat_f32_exact_kernel(b200_tensor w, b200_tensor x, b200_tensor d) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int64_t N = d.ne[0], M = d.ne[1];
    const int64_t total = N * M * d.ne[2] * d.ne[3];
    if (gw >= total) return;
    const int64_t n = gw % N, m = (gw / N) % M, i2 = (gw / (N * M)) % d.ne[2], i3 = gw / (N * M * d.ne[2]);
    const int64_t w2 = i2 / (d.ne[2] / w.ne[2]), w3 = i3 / (d.ne[3] / w.ne[3]);
    const float *wp = (const float *)((const char *)w.data + n * w.nb[1] + w2 * w.nb[2] + w3 * w.nb[3]);
    const float *xp = (const float *)((const char *)x.data + m * x.nb[1] + i2 * x.nb[2] + i3 * x.nb[3]);
    const int64_t K = w.ne[0], np = K & ~(int64_t)31;
    float acc = 0.0f;                                   // lane = 8 * j + l
    for (int64_t i = 0; i < np; i += 32) acc = __fmaf_rn(wp[i + lane], xp[i + lane], acc);
    // (s0 + s2) + (s1 + s3) lane-wise: lanes l, l+16 then l+8
    float a = __fadd_rn(acc, __shfl_down_sync(0xffffffffu, acc, 16));          // lanes 0..7: s0 + s2; lanes 8..15: s1 + s3
    a = __fadd_rn(a, __shfl_down_sync(0xffffffffu, a, 8));                     // lanes 0..7: x0[l]
    a = __fadd_rn(a, __shfl_down_sync(0xffffffffu, a, 4));                     // lanes 0..3: t[l] = x0[l] + x0[l + 4]
    a = __fadd_rn(a, __shfl_down_sync(0xffffffffu, a, 1));                     // lane 0: t0 + t1, lane 2: t2 + t3
    a = __fadd_rn(a, __shfl_down_sync(0xffffffffu, a, 2));                     // lane 0: (t0 + t1) + (t2 + t3)
    if (lane == 0) {
        for (int64_t i = np; i < K; i++) a = __fadd_rn(a, __fmul_rn(wp[i], xp[i]));
        *(float *)((char *)d.data + n * d.nb[0] + m * d.nb[1] + i2 * d.nb[2] + i3 * d.nb[3]) = a;
    }
}

int mul_mat_float(b200_ctx *ctx, const b200_tensor &w, const b200_tensor &x, const b200_tensor &d) {
    const int64_t total = tensor_nelements(d);
    if (total == 0) return B200_OK;
    if (ctx->opt_cpu_exact && w.type == B200_TYPE_F32 && w.nb[0] == 4 && x.nb[0] == 4) {
        b200_mul_mat_f32_exact_kernel<<<(unsigned)((total + 3) / 4), 128, 0, ctx->stream>>>(w, x, d);
        ctx->launches++;
        CUDA_TRY(cudaGetLastError());
        return B200_OK;
    }
    const unsigned grid = (unsigned)((total + 3) / 4);
    switch (w.type) {
        case B200_TYPE_F32:  b200_mul_mat_float_kernel<float><<<grid, 128, 0, ctx->stream>>>(w, x, d); break;
        case B200_TYPE_F16:  b200_mul_mat_float_kernel<__half><<<grid, 128, 0, ctx->stream>>>(w, x, d); break;
        case B200_TYPE_BF16: b200_mul_mat_float_kernel<__nv_bfloat16><<<grid, 128, 0, ctx->stream>>>(w, x, d); break;
        default: return B200_ERR_UNSUPPORTED;
    }
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return B200_OK;
}

// MUL_MAT_ID with float experts, the arithmetic of b200_mul_mat_float_kernel: one warp per (row n, slot, token); the expert index is read
// from ids on the device (an index outside [0, E) leaves its dst column untouched, as the grouped paths do)
template <typename WT>
__global__ void __launch_bounds__(128) b200_mul_mat_id_float_kernel(b200_tensor as, b200_tensor b, b200_tensor ids, b200_tensor d) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int64_t N = d.ne[0], n_used = d.ne[1];
    if (gw >= N * n_used * d.ne[2]) return;
    const int64_t n = gw % N, s = (gw / N) % n_used, t = gw / (N * n_used);
    const int e = *(const int32_t *)((const char *)ids.data + s * ids.nb[0] + t * ids.nb[1]);
    if (e < 0 || e >= as.ne[2]) return;
    const char *wp = (const char *)as.data + n * as.nb[1] + (int64_t)e * as.nb[2];
    const char *xp = (const char *)b.data + (s % b.ne[1]) * b.nb[1] + t * b.nb[2];
    float acc = 0.0f;
    for (int64_t k = lane; k < as.ne[0]; k += 32) {
        const float wv = w_to_float<WT>(*(const WT *)(wp + k * as.nb[0]));
        const float xv = x_round<WT>(*(const float *)(xp + k * b.nb[0]));
        acc = fmaf(wv, xv, acc);
    }
    acc = warp_reduce_sum(acc);
    if (lane == 0) *(float *)((char *)d.data + n * d.nb[0] + s * d.nb[1] + t * d.nb[2]) = acc;
}

int mul_mat_id_float(b200_ctx *ctx, const b200_tensor &as, const b200_tensor &b, const b200_tensor &ids, const b200_tensor &d) {
    const int64_t total = d.ne[0] * d.ne[1] * d.ne[2];
    if (total == 0) return B200_OK;
    const unsigned grid = (unsigned)((total + 3) / 4);
    switch (as.type) {
        case B200_TYPE_F32:  b200_mul_mat_id_float_kernel<float><<<grid, 128, 0, ctx->stream>>>(as, b, ids, d); break;
        case B200_TYPE_F16:  b200_mul_mat_id_float_kernel<__half><<<grid, 128, 0, ctx->stream>>>(as, b, ids, d); break;
        case B200_TYPE_BF16: b200_mul_mat_id_float_kernel<__nv_bfloat16><<<grid, 128, 0, ctx->stream>>>(as, b, ids, d); break;
        default: return B200_ERR_UNSUPPORTED;
    }
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return B200_OK;
}

// one quantised matmul: W [N rows of K] x cols (already quantised into `act`) -> dst
int mul_mat_q_cols(b200_ctx *ctx, int type, const uint8_t *W, size_t rb, int64_t N, int64_t K, const uint8_t *act, int64_t ncols,
                   float *dst, size_t dst_stride, bool w_const) {
    const size_t col_bytes = ActLayout::make(b200_act_mode_q8k(type), K).col_bytes;
    // GEMV path; launch_gemv chunks columns by what fits in shared memory
    for (int64_t c0 = 0; c0 < ncols; c0 += 64) {
        const int nc = (int)(ncols - c0 < 64 ? ncols - c0 : 64);
        int rc = launch_gemv(ctx, type, W, rb, N, K, act + (size_t)c0 * col_bytes, nc, dst + (size_t)c0 * dst_stride, dst_stride, w_const);
        if (rc) return rc;
    }
    return B200_OK;
}

bool quant_mul_mat_shape_ok(const b200_tensor &w, const b200_tensor &x, const b200_tensor &d) {
    if (!b200_type_is_quant(w.type) || x.type != B200_TYPE_F32 || d.type != B200_TYPE_F32) return false;
    const int64_t K = w.ne[0];
    if (K % b200_type_block_elems(w.type) != 0 || K % 32 != 0) return false;
    if (x.ne[0] != K || x.nb[0] != 4 || d.nb[0] != 4) return false;
    if (w.nb[0] != (uint64_t)b200_type_block_bytes(w.type)) return false;
    if (w.nb[1] != b200_row_bytes(w.type, K)) return false;            // rows back to back (GGUF layout)
    if ((x.nb[1] & 15) || ((uintptr_t)x.data & 15)) return false;     // float4 loads in the quantiser
    if ((w.type == B200_TYPE_Q4_K || w.type == B200_TYPE_Q5_K) && (((uintptr_t)w.data & 15) || (w.nb[2] & 15) || (w.nb[3] & 15))) return false;
    if (w.ne[2] == 0 || w.ne[3] == 0 || x.ne[2] % w.ne[2] || x.ne[3] % w.ne[3]) return false;
    return true;
}

// F16/BF16 weights that the tensor-core kernels take: contiguous 16-byte aligned rows (TMA tiles), K % 8 == 0, f32 x with 16-byte
// aligned columns (float4 loads), f32 dst columns
bool float_mm_ok(const b200_ctx *ctx, const b200_tensor &w, const b200_tensor &x, const b200_tensor &d) {
    if (ctx->opt_cpu_exact || (w.type != B200_TYPE_F16 && w.type != B200_TYPE_BF16)) return false;
    const int64_t K = w.ne[0];
    if (K % 8 || w.nb[0] != 2 || w.nb[1] != (uint64_t)K * 2 || (((uintptr_t)w.data | w.nb[2] | w.nb[3]) & 15)) return false;
    if (x.type != B200_TYPE_F32 || x.ne[0] != K || x.nb[0] != 4 || (((uintptr_t)x.data | x.nb[1] | x.nb[2] | x.nb[3]) & 15)) return false;
    if (d.type != B200_TYPE_F32 || d.nb[0] != 4 || ((d.nb[1] | d.nb[2] | d.nb[3]) & 3)) return false;
    return w.ne[2] > 0 && w.ne[3] > 0 && x.ne[2] % w.ne[2] == 0 && x.ne[3] % w.ne[3] == 0;
}

int mul_mat_f16_tc(b200_ctx *ctx, const b200_tensor &w, const b200_tensor &x, const b200_tensor &d) {
    const int64_t K = w.ne[0], N = w.ne[1], M = x.ne[1];
    if (tensor_nelements(d) == 0) return B200_OK;
    const bool w_const = (w.flags & B200_TENSOR_FLAG_WEIGHT) != 0;
    for (int64_t i3 = 0; i3 < x.ne[3]; i3++)
        for (int64_t i2 = 0; i2 < x.ne[2]; i2++) {
            const int64_t w2 = i2 / (x.ne[2] / w.ne[2]), w3 = i3 / (x.ne[3] / w.ne[3]);
            const uint16_t *wp = (const uint16_t *)((const char *)w.data + w2 * w.nb[2] + w3 * w.nb[3]);
            const float *xp = (const float *)((const char *)x.data + i2 * x.nb[2] + i3 * x.nb[3]);
            float *dp = (float *)((char *)d.data + i2 * d.nb[2] + i3 * d.nb[3]);
            const int rc = M <= F16MM_STREAM_MAX_M ? gemv_f16_run(ctx, w.type, wp, N, K, xp, x.nb[1], (int)M, dp, d.nb[1] / 4, w_const)
                                                   : gemm_f16_tc_run(ctx, w.type, wp, N, K, xp, x.nb[1], M, dp, d.nb[1] / 4);
            if (rc) return rc;
        }
    return B200_OK;
}

}  // namespace

// row-split weight: the shard of every device is a dense GGUF matrix of its row range
static bool split_ok(const b200_op *op) {
    const b200_tensor &w = op->src[0], &x = op->src[1], &d = op->dst;
    const b200_split *sp = (const b200_split *)w.data;
    const bool f16 = w.type == B200_TYPE_F16 || w.type == B200_TYPE_BF16;
    // sp == NULL: llama.cpp probing whether a weight may live in the split buffer type (no shards allocated yet)
    if ((sp && (sp->n_dev < 1 || sp->n_dev > B200_MAX_SPLIT)) || !(b200_type_is_quant(w.type) || f16)) return false;
    if (w.ne[2] != 1 || w.ne[3] != 1 || x.ne[2] != 1 || x.ne[3] != 1) return false;
    // F16/BF16: dense shard rows; any f32 x and dst columns (layouts the tensor-core kernels refuse take the float kernel on every
    // shard); dst rows 4 bytes apart, so that a shard's row range starts row_low * 4 bytes into dst
    if (f16)
        return w.nb[0] == 2 && w.nb[1] == (uint64_t)w.ne[0] * 2 && x.type == B200_TYPE_F32 && x.ne[0] == w.ne[0] && d.type == B200_TYPE_F32 && d.nb[0] == 4;
    b200_tensor w0 = w;                                   // shape checks against an aligned stand-in for the shards (cudaMalloc'd: 256-byte aligned)
    w0.data = (void *)(uintptr_t)0x1000; w0.flags &= ~B200_TENSOR_FLAG_SPLIT;
    return quant_mul_mat_shape_ok(w0, x, d);
}

bool supports_mul_mat(const b200_op *op) {
    const b200_tensor &w = op->src[0], &x = op->src[1], &d = op->dst;
    if (w.flags & B200_TENSOR_FLAG_SPLIT) return split_ok(op);
    if (x.type != B200_TYPE_F32 || d.type != B200_TYPE_F32) return false;
    if (w.type == B200_TYPE_F32 || w.type == B200_TYPE_F16 || w.type == B200_TYPE_BF16) {
        return w.ne[2] > 0 && w.ne[3] > 0 && d.ne[2] % w.ne[2] == 0 && d.ne[3] % w.ne[3] == 0;
    }
    return quant_mul_mat_shape_ok(w, x, d);
}

// MUL_MAT over a row-split weight (replaces the split path of ggml_cuda_op_mul_mat, ggml-cuda.cu:1363-1671): fork on the main stream,
// every device multiplies its shard into its row range of dst -- activations read from and results written to the MAIN device's memory
// through NVLink peer access, no staging copies -- and the main stream joins.  Quantised weights: each dst element is produced by the
// same kernels as on one GPU, so the result does not depend on the split.  F16/BF16 weights: gemv_f16 and gemm_f16_tc choose their K
// slices from the row count they are given, so a shard may sum K in other slices than the whole matrix would: the result equals the
// one-GPU result up to f32 summation order, and is the same bits on every run of the same split.
static int op_mul_mat_split(b200_ctx *ctx, const b200_op *op) {
    const b200_tensor &w = op->src[0];
    const b200_split *sp = (const b200_split *)w.data;
    if (!sp) { b200_set_error("mul_mat split: no shard table"); return B200_ERR_FAILED; }
    if (!ctx->split_fork) CUDA_TRY(cudaEventCreateWithFlags(&ctx->split_fork, cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(ctx->split_fork, ctx->stream));
    int rc = B200_OK;
    for (int i = 0; i < sp->n_dev && !rc; i++) {
        const int64_t r0 = sp->row_low[i], nr = sp->row_low[i + 1] - r0;
        if (nr <= 0) continue;
        const int dev = sp->device[i];
        b200_op sub = *op;
        sub.src[0].data = sp->shard[i]; sub.src[0].flags &= ~B200_TENSOR_FLAG_SPLIT; sub.src[0].ne[1] = nr;
        sub.src[0].nb[2] = sub.src[0].nb[1] * nr; sub.src[0].nb[3] = sub.src[0].nb[2];
        sub.dst.data = (char *)op->dst.data + r0 * 4; sub.dst.ne[0] = nr;
        if (dev == ctx->device) { rc = op_mul_mat(ctx, &sub); continue; }
        if (dev < 0 || dev >= 16) { b200_set_error("mul_mat split: device %d", dev); return B200_ERR_FAILED; }
        b200_ctx *pc = ctx->split_peer[dev];
        if (!pc) {
            pc = b200_ctx_create(dev);
            if (!pc) return B200_ERR_FAILED;
            int can = 0;
            cudaDeviceCanAccessPeer(&can, dev, ctx->device);
            if (!can) { b200_set_error("mul_mat split: device %d cannot access device %d memory", dev, ctx->device); b200_ctx_destroy(pc); return B200_ERR_FAILED; }
            cudaSetDevice(dev);
            cudaError_t e = cudaDeviceEnablePeerAccess(ctx->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { b200_set_error("cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e)); b200_ctx_destroy(pc); return B200_ERR_FAILED; }
            cudaGetLastError();
            CUDA_TRY(cudaEventCreateWithFlags(&ctx->split_join[dev], cudaEventDisableTiming));
            pc->opt_pdl = 0; pc->opt_cuda_graphs = 0;
            ctx->split_peer[dev] = pc;
        }
        pc->opt_cpu_exact = ctx->opt_cpu_exact;
        CUDA_TRY(cudaSetDevice(dev));
        CUDA_TRY(cudaStreamWaitEvent(pc->stream, ctx->split_fork, 0));
        rc = op_mul_mat(pc, &sub);
        if (!rc) {
            CUDA_TRY(cudaEventRecord(ctx->split_join[dev], pc->stream));
            CUDA_TRY(cudaSetDevice(ctx->device));
            CUDA_TRY(cudaStreamWaitEvent(ctx->stream, ctx->split_join[dev], 0));
            ctx->launches += 1;
        }
        cudaSetDevice(ctx->device);
    }
    ctx->split_ops++;
    return rc;
}

int op_mul_mat(b200_ctx *ctx, const b200_op *op) {
    const b200_tensor &w = op->src[0], &x = op->src[1], &d = op->dst;
    if (w.flags & B200_TENSOR_FLAG_SPLIT) return op_mul_mat_split(ctx, op);
    if (!b200_type_is_quant(w.type)) return float_mm_ok(ctx, w, x, d) ? mul_mat_f16_tc(ctx, w, x, d) : mul_mat_float(ctx, w, x, d);
    if (!quant_mul_mat_shape_ok(w, x, d)) { b200_set_error("mul_mat: unsupported layout"); return B200_ERR_UNSUPPORTED; }
    const int64_t K = w.ne[0], N = w.ne[1], M = x.ne[1];
    const int q8k = b200_act_mode_q8k(w.type);
    const ActLayout L = ActLayout::make(q8k, K);
    const size_t rb = b200_row_bytes(w.type, K);
    const bool w_const = (w.flags & B200_TENSOR_FLAG_WEIGHT) != 0;
    const int64_t nbatch = x.ne[2] * x.ne[3];
    // up to this many columns the streaming GEMV (one launch, activations quantised in its prologue); above, the mma.sync small-batch
    // kernel (gemv_mma.cu: 23 us vs 59 us at 8 columns on a 14336 x 4096 Q4_K matrix)
    static const int64_t gemv_max_m = getenv("GGML_B200_GEMV_MAX_M") ? atoi(getenv("GGML_B200_GEMV_MAX_M")) : 4;
    if (ctx->opt_cpu_exact) {
        // parity mode: same quantised activations, float sums in the reference's SIMD order (exact.cu)
        uint8_t *act = (uint8_t *)ctx->get_scratch(SCRATCH_ACT, L.col_bytes * (size_t)(M * nbatch));
        if (!act) return B200_ERR_ALLOC;
        for (int64_t i3 = 0; i3 < x.ne[3]; i3++)
            for (int64_t i2 = 0; i2 < x.ne[2]; i2++) {
                const int64_t w2 = i2 / (x.ne[2] / w.ne[2]), w3 = i3 / (x.ne[3] / w.ne[3]);
                const uint8_t *wp = (const uint8_t *)w.data + w2 * w.nb[2] + w3 * w.nb[3];
                const float *xp = (const float *)((const char *)x.data + i2 * x.nb[2] + i3 * x.nb[3]);
                float *dp = (float *)((char *)d.data + i2 * d.nb[2] + i3 * d.nb[3]);
                uint8_t *ab = act + (size_t)((i3 * x.ne[2] + i2) * M) * L.col_bytes;
                int rc = launch_quantize_act(ctx, q8k, xp, x.nb[1], K, M, ab);
                if (!rc) rc = launch_mul_mat_exact(ctx, w.type, wp, rb, N, K, ab, M, dp, d.nb[1] / 4);
                if (rc) return rc;
            }
        return B200_OK;
    }
    if (M <= gemv_max_m) {
        // decode path: one fused launch per (batch) matmul -- activation quantisation happens in the GEMV prologue
        for (int64_t i3 = 0; i3 < x.ne[3]; i3++)
            for (int64_t i2 = 0; i2 < x.ne[2]; i2++) {
                const int64_t w2 = i2 / (x.ne[2] / w.ne[2]), w3 = i3 / (x.ne[3] / w.ne[3]);
                const uint8_t *wp = (const uint8_t *)w.data + w2 * w.nb[2] + w3 * w.nb[3];
                const float *xp = (const float *)((const char *)x.data + i2 * x.nb[2] + i3 * x.nb[3]);
                float *dp = (float *)((char *)d.data + i2 * d.nb[2] + i3 * d.nb[3]);
                int rc = launch_gemv_f32(ctx, w.type, wp, rb, N, K, xp, x.nb[1], (int)M, dp, d.nb[1] / 4, w_const, 0, nullptr, 0.0f, nullptr);
                if (rc) return rc;
            }
        return B200_OK;
    }
    // continuous-batching decode (9..32 columns): weight-streaming mma.sync kernel (gemv_mma.cu); q4_0 / q8_0, which the tcgen05
    // GEMM does not decode, go through it in chunks of 32 columns at any batch size
    static const int64_t mma_max_m = getenv("GGML_B200_MMA_MAX_M") ? atoi(getenv("GGML_B200_MMA_MAX_M")) : 32;
    // K-quants from tc_min_m token columns up: the tcgen05 kind::f16 GEMM (gemm_tc.cu: exact-integer f16 operands, min term on the tensor core)
    static const int64_t tc_min_m = getenv("GGML_B200_TC_MIN_M") ? atoi(getenv("GGML_B200_TC_MIN_M")) : 33;
    if (M >= tc_min_m && x.nb[0] == 4 && gemm_tc_supported(w.type, N, K, M) && !((uintptr_t)w.data & 15) && !(w.nb[2] & 15) && !(w.nb[3] & 15)) {
        for (int64_t i3 = 0; i3 < x.ne[3]; i3++)
            for (int64_t i2 = 0; i2 < x.ne[2]; i2++) {
                const int64_t w2 = i2 / (x.ne[2] / w.ne[2]), w3 = i3 / (x.ne[3] / w.ne[3]);
                const uint8_t *wp = (const uint8_t *)w.data + w2 * w.nb[2] + w3 * w.nb[3];
                const float *xp = (const float *)((const char *)x.data + i2 * x.nb[2] + i3 * x.nb[3]);
                float *dp = (float *)((char *)d.data + i2 * d.nb[2] + i3 * d.nb[3]);
                int rc = gemm_tc_run(ctx, w.type, wp, rb, N, K, xp, x.nb[1], M, dp, d.nb[1] / 4);
                if (rc) return rc;
            }
        return B200_OK;
    }
    // prompt batches the tcgen05 GEMM does not take: the mma.sync tile GEMM (gemm_mma.cu, all five formats)
    if (M > mma_max_m && gemm_mma_supported(w.type, N, K, M)) {
        for (int64_t i3 = 0; i3 < x.ne[3]; i3++)
            for (int64_t i2 = 0; i2 < x.ne[2]; i2++) {
                const int64_t w2 = i2 / (x.ne[2] / w.ne[2]), w3 = i3 / (x.ne[3] / w.ne[3]);
                const uint8_t *wp = (const uint8_t *)w.data + w2 * w.nb[2] + w3 * w.nb[3];
                const float *xp = (const float *)((const char *)x.data + i2 * x.nb[2] + i3 * x.nb[3]);
                float *dp = (float *)((char *)d.data + i2 * d.nb[2] + i3 * d.nb[3]);
                int rc = gemm_mma_run(ctx, w.type, wp, rb, N, K, xp, x.nb[1], M, dp, d.nb[1] / 4);
                if (rc) return rc;
            }
        return B200_OK;
    }
    if (gemv_mma_supported(w.type, N, K, M)) {
        uint8_t *act = (uint8_t *)ctx->get_scratch(SCRATCH_ACT, L.col_bytes * (size_t)M);
        if (!act) return B200_ERR_ALLOC;
        for (int64_t i3 = 0; i3 < x.ne[3]; i3++)
            for (int64_t i2 = 0; i2 < x.ne[2]; i2++) {
                const int64_t w2 = i2 / (x.ne[2] / w.ne[2]), w3 = i3 / (x.ne[3] / w.ne[3]);
                const uint8_t *wp = (const uint8_t *)w.data + w2 * w.nb[2] + w3 * w.nb[3];
                const float *xp = (const float *)((const char *)x.data + i2 * x.nb[2] + i3 * x.nb[3]);
                float *dp = (float *)((char *)d.data + i2 * d.nb[2] + i3 * d.nb[3]);
                int rc = launch_quantize_act(ctx, q8k, xp, x.nb[1], K, M, act);
                for (int64_t c0 = 0; c0 < M && !rc; c0 += 32)
                    rc = launch_gemv_mma(ctx, w.type, wp, rb, N, K, act + (size_t)c0 * L.col_bytes, (int)(M - c0 < 32 ? M - c0 : 32),
                                         dp + (size_t)c0 * (d.nb[1] / 4), d.nb[1] / 4, M <= 32, w_const);
                if (rc) return rc;
            }
        return B200_OK;
    }
    // quantise every src1 column of every batch once
    uint8_t *act = (uint8_t *)ctx->get_scratch(SCRATCH_ACT, L.col_bytes * (size_t)(M * nbatch));
    if (!act) return B200_ERR_ALLOC;
    for (int64_t i3 = 0; i3 < x.ne[3]; i3++)
        for (int64_t i2 = 0; i2 < x.ne[2]; i2++) {
            const float *xp = (const float *)((const char *)x.data + i2 * x.nb[2] + i3 * x.nb[3]);
            int rc = launch_quantize_act(ctx, q8k, xp, x.nb[1], K, M, act + (size_t)((i3 * x.ne[2] + i2) * M) * L.col_bytes);
            if (rc) return rc;
        }
    for (int64_t i3 = 0; i3 < x.ne[3]; i3++)
        for (int64_t i2 = 0; i2 < x.ne[2]; i2++) {
            const int64_t w2 = i2 / (x.ne[2] / w.ne[2]), w3 = i3 / (x.ne[3] / w.ne[3]);
            const uint8_t *wp = (const uint8_t *)w.data + w2 * w.nb[2] + w3 * w.nb[3];
            float *dp = (float *)((char *)d.data + i2 * d.nb[2] + i3 * d.nb[3]);
            int rc = mul_mat_q_cols(ctx, w.type, wp, rb, N, K, act + (size_t)((i3 * x.ne[2] + i2) * M) * L.col_bytes, M, dp,
                                    d.nb[1] / 4, w_const);
            if (rc) return rc;
        }
    return B200_OK;
}

// ---------------------------------------------------------------------------------------------------
// MUL_MAT_ID (ggml_compute_forward_mul_mat_id, ggml-cpu.c:8902-...): dst[:, slot, tok] = as[ids[slot, tok]] . b[:, slot % b_ne1, tok]
// The expert index is read ON THE DEVICE (no D2H copy of ids + stream sync as in ggml-cuda.cu:1976-1979), so the op is capturable in a
// CUDA graph.  Up to 8 (token, slot) pairs: one streaming GEMV per pair; more: b200_moe_group_kernel counting-sorts the pairs by expert
// and launch_gemv_mma_grouped streams every expert's matrix once per 32 pairs (gemv_mma.cu).
// ---------------------------------------------------------------------------------------------------
bool supports_mul_mat_id(const b200_op *op) {
    const b200_tensor &as = op->src[0], &b = op->src[1], &ids = op->src[2], &d = op->dst;
    if (b.type != B200_TYPE_F32 || d.type != B200_TYPE_F32 || ids.type != B200_TYPE_I32) return false;
    const bool fl = as.type == B200_TYPE_F32 || as.type == B200_TYPE_F16 || as.type == B200_TYPE_BF16;
    if (fl) {                  // any strides: what the tensor-core paths do not take, the float kernel does
        if (as.ne[3] != 1 || b.ne[3] != 1 || d.ne[3] != 1 || b.ne[0] != as.ne[0]) return false;
        if (d.ne[0] != as.ne[1] || d.ne[1] != ids.ne[0] || d.ne[2] != ids.ne[1] || b.ne[2] != ids.ne[1]) return false;
        return b.ne[1] == 1 || b.ne[1] == ids.ne[0];
    }
    if (!b200_type_is_quant(as.type)) return false;
    const int64_t K = as.ne[0];
    if (K % b200_type_block_elems(as.type) != 0 || K % 32 != 0 || b.ne[0] != K) return false;
    if (as.nb[0] != (uint64_t)b200_type_block_bytes(as.type) || as.nb[1] != b200_row_bytes(as.type, K)) return false;
    if ((as.type == B200_TYPE_Q4_K || as.type == B200_TYPE_Q5_K) && (((uintptr_t)as.data & 15) || (as.nb[2] & 15))) return false;
    if (as.ne[3] != 1 || b.ne[3] != 1 || d.ne[3] != 1) return false;
    if (b.nb[0] != 4 || d.nb[0] != 4 || ids.nb[0] != 4) return false;
    if ((b.nb[1] & 15) || (b.nb[2] & 15) || ((uintptr_t)b.data & 15)) return false;
    if (d.ne[0] != as.ne[1] || d.ne[1] != ids.ne[0] || d.ne[2] != ids.ne[1] || b.ne[2] != ids.ne[1]) return false;
    if (b.ne[1] != 1 && b.ne[1] != ids.ne[0]) return false;
    return true;
}

// routing tables for the grouped path: counting sort of the (token, slot) pairs by expert, one CTA (pairs <= a few thousand)
__global__ void __launch_bounds__(1024) b200_moe_group_kernel(const char *ids, uint64_t nb0, uint64_t nb1, int n_used, int n_tok, int E, int32_t *off, int32_t *pairs, int use_pdl) {
    extern __shared__ int sm_cnt[];            // [E] counts, then [E] cursors
    if (use_pdl) { pdl_trigger(); pdl_wait(); }
    int *cnt = sm_cnt, *cur = sm_cnt + E;
    for (int e = threadIdx.x; e < E; e += blockDim.x) cnt[e] = 0;
    __syncthreads();
    const int npairs = n_used * n_tok;
    for (int p = threadIdx.x; p < npairs; p += blockDim.x) {
        const int e = *(const int32_t *)(ids + (uint64_t)(p % n_used) * nb0 + (uint64_t)(p / n_used) * nb1);
        if (e >= 0 && e < E) atomicAdd(&cnt[e], 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int a = 0;
        for (int e = 0; e < E; e++) { off[e] = a; cur[e] = a; a += cnt[e]; }
        off[E] = a;
    }
    __syncthreads();
    // ascending pair order inside an expert (deterministic tables): thread-strided passes would interleave, so one warp per expert scans
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int e = warp; e < E; e += nw) {
        int pos = cur[e];
        for (int p0 = 0; p0 < npairs; p0 += 32) {
            const int p = p0 + lane;
            const bool hit = p < npairs && *(const int32_t *)(ids + (uint64_t)(p % n_used) * nb0 + (uint64_t)(p / n_used) * nb1) == e;
            const uint32_t m = __ballot_sync(0xffffffffu, hit);
            if (hit) pairs[pos + __popc(m & ((1u << lane) - 1))] = p;
            pos += __popc(m);
        }
    }
}

// F16/BF16 experts that the grouped tensor-core paths take: contiguous 16-byte aligned expert rows (3-D TMA map), K % 8 == 0, x columns
// of the pairs 16-byte aligned and dense across tokens (float4 gathers), f32 dst; the routing tables' limits (one grouping CTA)
static bool float_mm_id_ok(const b200_ctx *ctx, const b200_tensor &as, const b200_tensor &b, const b200_tensor &ids, const b200_tensor &d) {
    if (ctx->opt_cpu_exact || (as.type != B200_TYPE_F16 && as.type != B200_TYPE_BF16)) return false;
    const int64_t K = as.ne[0], npairs = ids.ne[0] * ids.ne[1];
    if (K % 8 || K > INT32_MAX || as.ne[1] > INT32_MAX || as.nb[0] != 2 || as.nb[1] != (uint64_t)K * 2 || (((uintptr_t)as.data | as.nb[2]) & 15)) return false;
    const bool b_dense = b.ne[1] == 1 || b.nb[2] == b.ne[1] * b.nb[1];
    if (!b_dense || b.nb[0] != 4 || (((uintptr_t)b.data | b.nb[1] | b.nb[2]) & 15)) return false;
    if (d.nb[0] != 4 || ((d.nb[1] | d.nb[2]) & 3)) return false;
    return as.ne[2] >= 1 && as.ne[2] <= 1024 && npairs >= 1 && npairs <= (1 << 20);
}

// MUL_MAT_ID with F32 / F16 / BF16 experts
static int op_mul_mat_id_float(b200_ctx *ctx, const b200_tensor &as, const b200_tensor &b, const b200_tensor &ids, const b200_tensor &d) {
    if (!float_mm_id_ok(ctx, as, b, ids, d)) return mul_mat_id_float(ctx, as, b, ids, d);
    const int64_t K = as.ne[0], N = as.ne[1], npairs = ids.ne[0] * ids.ne[1], E = as.ne[2];
    int32_t *tab = (int32_t *)ctx->get_scratch(SCRATCH_MOE, (size_t)(E + 1 + npairs) * 4);
    if (!tab) return B200_ERR_ALLOC;
    b200_moe_group_kernel<<<1, 1024, (size_t)2 * E * sizeof(int), ctx->stream>>>((const char *)ids.data, ids.nb[0], ids.nb[1], (int)ids.ne[0], (int)ids.ne[1], (int)E, tab, tab + E + 1, 0);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    MmGroupDesc g = {};
    g.off = tab; g.pairs = tab + E + 1; g.E = (int)E; g.n_used = (int)ids.ne[0]; g.b_ne1 = (int)b.ne[1];
    g.expert_stride = as.nb[2]; g.d_nb1 = d.nb[1] / 4; g.d_nb2 = d.nb[2] / 4;
    const size_t x_stride = b.ne[1] == 1 ? b.nb[2] : b.nb[1];
    // prompt batches (>= 32 pairs per expert on average): token tiles of 128 pairs per expert through the tcgen05 GEMM, as for quantised
    // experts (profiles/moe_float_weights.md)
    if (npairs >= 32 * E) {
        g.max_chunks = (int)std::min<int64_t>(npairs, npairs / 128 + E);
        return gemm_f16_tc_run_grouped(ctx, as.type, (const uint16_t *)as.data, N, K, (const float *)b.data, x_stride, g, npairs, (float *)d.data);
    }
    g.max_chunks = (int)std::min<int64_t>(npairs, npairs / 32 + E);
    return gemv_f16_run_grouped(ctx, as.type, (const uint16_t *)as.data, N, K, (const float *)b.data, x_stride, g, npairs, (float *)d.data);
}

int op_mul_mat_id(b200_ctx *ctx, const b200_op *op) {
    const b200_tensor &as = op->src[0], &b = op->src[1], &ids = op->src[2], &d = op->dst;
    if (!b200_type_is_quant(as.type)) return op_mul_mat_id_float(ctx, as, b, ids, d);
    const int64_t K = as.ne[0], N = as.ne[1], n_used = ids.ne[0], n_tok = ids.ne[1];
    const size_t rb = b200_row_bytes(as.type, K);
    // batches: group the (token, slot) pairs by expert on the device and stream every expert's matrix once per 32 pairs (the reference
    // copies ids to the host, syncs, and loops experts there: ggml-cuda.cu:1976-2096)
    if (ctx->opt_cpu_exact && (b.ne[1] == 1 || b.nb[2] == b.ne[1] * b.nb[1])) {
        // parity mode: same quantised activations, every (token, slot) dot in the reference's SIMD order (exact.cu)
        const int q8k = b200_act_mode_q8k(as.type);
        const ActLayout L = ActLayout::make(q8k, K);
        const int64_t acols = b.ne[1] == 1 ? n_tok : n_used * n_tok;
        uint8_t *act = (uint8_t *)ctx->get_scratch(SCRATCH_ACT, L.col_bytes * (size_t)acols);
        if (!act) return B200_ERR_ALLOC;
        int rc = launch_quantize_act(ctx, q8k, (const float *)b.data, b.ne[1] == 1 ? b.nb[2] : b.nb[1], K, acols, act);
        if (rc) return rc;
        ExactMoe moe = {(const char *)ids.data, ids.nb[0], ids.nb[1], (int)n_used, (int)b.ne[1], (size_t)as.nb[2], (size_t)(d.nb[1] / 4), (size_t)(d.nb[2] / 4)};
        return launch_mul_mat_exact(ctx, as.type, (const uint8_t *)as.data, rb, N, K, act, n_used * n_tok, (float *)d.data, 0, &moe);
    }
    static const int64_t group_min = getenv("GGML_B200_MOE_GROUP_MIN") ? atoi(getenv("GGML_B200_MOE_GROUP_MIN")) : 9;
    const int64_t npairs = n_used * n_tok, E = as.ne[2];
    const bool b_dense = b.ne[1] == 1 || b.nb[2] == b.ne[1] * b.nb[1];
    if (npairs >= group_min && !ctx->opt_cpu_exact && gemv_mma_supported(as.type, N, K, 32) && b_dense && E <= 1024 && npairs <= (1 << 20) && !(d.nb[1] & 3) && !(d.nb[2] & 3)) {
        const int q8k = b200_act_mode_q8k(as.type);
        const ActLayout L = ActLayout::make(q8k, K);
        const int64_t acols = b.ne[1] == 1 ? n_tok : npairs;
        int32_t *tab = (int32_t *)ctx->get_scratch(SCRATCH_MOE, (size_t)(E + 1 + npairs) * 4);
        if (!tab) return B200_ERR_ALLOC;
        b200_moe_group_kernel<<<1, 1024, (size_t)2 * E * sizeof(int), ctx->stream>>>((const char *)ids.data, ids.nb[0], ids.nb[1], (int)n_used, (int)n_tok, (int)E, tab, tab + E + 1, 0);
        ctx->launches++;
        CUDA_TRY(cudaGetLastError());
        MmGroupDesc g = {};
        g.off = tab; g.pairs = tab + E + 1; g.E = (int)E; g.n_used = (int)n_used; g.b_ne1 = (int)b.ne[1];
        g.expert_stride = as.nb[2]; g.d_nb1 = d.nb[1] / 4; g.d_nb2 = d.nb[2] / 4;
        // prompt batches (>= 32 pairs per expert on average): token tiles of 128 pairs per expert through the tile GEMM (gemm_mma.cu)
        if (npairs >= 32 * E && gemm_mma_supported(as.type, N, K, 128)) {
            g.max_chunks = (int)std::min<int64_t>(npairs, npairs / 128 + E);
            // K-quants: the tcgen05 kind::f16 GEMM in grouped mode (gemm_tc.cu); Q4_0 / Q8_0: the mma.sync tile GEMM
            if (gemm_tc_supported(as.type, N, K, 128) && !(((uintptr_t)as.data | as.nb[2]) & 15))
                return gemm_tc_run_grouped(ctx, as.type, (const uint8_t *)as.data, rb, N, K, (const float *)b.data, b.ne[1] == 1 ? b.nb[2] : b.nb[1], g, (float *)d.data);
            return gemm_mma_run_grouped(ctx, as.type, (const uint8_t *)as.data, rb, N, K, (const float *)b.data, b.ne[1] == 1 ? b.nb[2] : b.nb[1], g, (float *)d.data);
        }
        uint8_t *act = (uint8_t *)ctx->get_scratch(SCRATCH_ACT, L.col_bytes * (size_t)acols);
        if (!act) return B200_ERR_ALLOC;
        int rc = launch_quantize_act(ctx, q8k, (const float *)b.data, b.ne[1] == 1 ? b.nb[2] : b.nb[1], K, acols, act);
        if (rc) return rc;
        g.max_chunks = (int)std::min<int64_t>(npairs, npairs / 32 + E);
        return launch_gemv_mma_grouped(ctx, as.type, (const uint8_t *)as.data, rb, N, K, act, g, (float *)d.data);
    }
    for (int64_t t = 0; t < n_tok; t++)
        for (int64_t s = 0; s < n_used; s++) {
            const int32_t *idp = (const int32_t *)((const char *)ids.data + s * ids.nb[0] + t * ids.nb[1]);
            const float *xp = (const float *)((const char *)b.data + (s % b.ne[1]) * b.nb[1] + t * b.nb[2]);
            float *dp = (float *)((char *)d.data + s * d.nb[1] + t * d.nb[2]);
            int rc = launch_gemv_expert(ctx, as.type, (const uint8_t *)as.data, rb, as.nb[2], idp, N, K, xp, dp);
            if (rc) return rc;
        }
    return B200_OK;
}
