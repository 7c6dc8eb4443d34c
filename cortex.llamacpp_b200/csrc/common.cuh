// common.cuh -- internal declarations shared by every translation unit of libggml_b200_kernels.so
// B200 (sm_100a) only.  Replaces the role of ggml-cuda/common.cuh (context, reductions, dp4a) with a
// one-stream-per-context design and Blackwell primitives (mbarrier + cp.async.bulk, PDL).
#pragma once

#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include <unordered_map>

#include "../../include/ggml_b200.h"

// ------------------------------------------------------------------------------------------------
// error handling: nothing throws across the C ABI; failures set a thread-local message
// ------------------------------------------------------------------------------------------------
void b200_set_error(const char *fmt, ...);

#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t err__ = (expr);                                                                 \
        if (err__ != cudaSuccess) {                                                                 \
            b200_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(err__)); \
            return B200_ERR_FAILED;                                                                 \
        }                                                                                           \
    } while (0)

// ------------------------------------------------------------------------------------------------
// block layouts (restated from ggml-common.h:161-328; byte offsets only, no structs shared)
// ------------------------------------------------------------------------------------------------
namespace blk {
constexpr int QK   = 32;
constexpr int QKK  = 256;
constexpr int Q4_0_BYTES = 18;    // half d | qs[16]
constexpr int Q8_0_BYTES = 34;    // half d | int8 qs[32]
constexpr int Q4_K_BYTES = 144;   // half d, half dmin | scales[12] | qs[128]
constexpr int Q5_K_BYTES = 176;   // half d, half dmin | scales[12] | qh[32] | qs[128]
constexpr int Q6_K_BYTES = 210;   // ql[128] | qh[64] | int8 scales[16] | half d
constexpr int Q8_K_BYTES = 292;   // float d | int8 qs[256] | int16 bsums[16]
}  // namespace blk

__host__ __device__ inline int b200_type_block_elems(int type) {
    switch (type) {
        case B200_TYPE_Q4_0: case B200_TYPE_Q8_0: return 32;
        case B200_TYPE_Q4_K: case B200_TYPE_Q5_K: case B200_TYPE_Q6_K: case B200_TYPE_Q8_K: return 256;
        default: return 1;
    }
}
__host__ __device__ inline int b200_type_block_bytes(int type) {
    switch (type) {
        case B200_TYPE_F32: case B200_TYPE_I32: return 4;
        case B200_TYPE_F16: case B200_TYPE_BF16: return 2;
        case B200_TYPE_Q4_0: return 18;
        case B200_TYPE_Q8_0: return 34;
        case B200_TYPE_Q4_K: return 144;
        case B200_TYPE_Q5_K: return 176;
        case B200_TYPE_Q6_K: return 210;
        case B200_TYPE_Q8_K: return 292;
        default: return 0;
    }
}
inline bool b200_type_is_quant(int type) {
    return type == B200_TYPE_Q4_0 || type == B200_TYPE_Q8_0 || type == B200_TYPE_Q4_K || type == B200_TYPE_Q5_K ||
           type == B200_TYPE_Q6_K;
}
inline size_t b200_row_bytes(int type, int64_t k) {
    return (size_t)(k / b200_type_block_elems(type)) * b200_type_block_bytes(type);
}
// activation format the CPU oracle pairs with a weight type (vec_dot_type, ggml-cpu.c:266-341)
inline int b200_act_mode_q8k(int type) { return type == B200_TYPE_Q4_K || type == B200_TYPE_Q5_K || type == B200_TYPE_Q6_K; }

inline bool tensor_is_contiguous(const b200_tensor &t) {
    const int be = b200_type_block_elems(t.type), bb = b200_type_block_bytes(t.type);
    if (t.nb[0] != (uint64_t)bb) return false;
    uint64_t expect = (uint64_t)(t.ne[0] / be) * bb;
    for (int i = 1; i < 4; i++) {
        if (t.ne[i] != 1 && t.nb[i] != expect) return false;
        expect *= t.ne[i];
    }
    return true;
}
inline int64_t tensor_nelements(const b200_tensor &t) { return t.ne[0] * t.ne[1] * t.ne[2] * t.ne[3]; }
inline int64_t tensor_nrows(const b200_tensor &t) { return t.ne[1] * t.ne[2] * t.ne[3]; }

// ------------------------------------------------------------------------------------------------
// activation scratch: the quantised form of src1 that GEMV/GEMM kernels consume.  One column
// (= one token) is laid out as
//     [ qs   : K int8                     ]  (16-byte aligned start)
//     [ d    : K/G floats                 ]  G = 256 (q8_K mode) or 32 (q8_0 mode)
//     [ sums : K/S int16                  ]  S = 16 (q8_K bsums) or 32 (q8_0 mode block sums)
// values are bit-identical to the reference's block_q8_K / block_q8_0 fields (d of q8_0 mode is the
// fp16-rounded scale widened to f32); the split layout is what lets kernels use 128-bit loads.
// ------------------------------------------------------------------------------------------------
struct ActLayout {
    int    q8k;          // 1: q8_K mode, 0: q8_0 mode
    int64_t K;
    size_t off_d, off_sums, col_bytes;
    __host__ __device__ static ActLayout make(int q8k, int64_t K) {
        ActLayout L;
        L.q8k = q8k; L.K = K;
        const size_t nd = (size_t)(K / (q8k ? 256 : 32)), ns = (size_t)(K / (q8k ? 16 : 32));
        L.off_d = ((size_t)K + 15) & ~(size_t)15;
        L.off_sums = L.off_d + ((nd * 4 + 15) & ~(size_t)15);
        L.col_bytes = L.off_sums + ((ns * 2 + 15) & ~(size_t)15);
        return L;
    }
};

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
struct GraphCache;   // graph.cu
struct b200_comm;    // comm.cu

struct b200_ctx {
    int           device   = 0;
    cudaStream_t  stream   = nullptr;
    int           sm_count = 148;
    size_t        smem_optin = 227 * 1024;
    // growable device scratch (activation quantisation, split-KV partials, MoE routing tables)
    void *        scratch[6]      = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    size_t        scratch_size[6] = {0, 0, 0, 0, 0, 0};
    int64_t       launches = 0;
    // options
    int           opt_cuda_graphs = 0;
    int           opt_fusion      = 2;      // 0 off, 1 two-op fusions, 2 + llama layer fusions for decode ubatches
    int           opt_pdl         = 0;
    int           opt_ffn_pair    = 1;      // FFN decode fusion: the gate|up GEMV writes silu(gate) * up itself (gemv_bs1.cu pair mode); 0 = swiglu in the down GEMV's prologue
    int           opt_l2_prefetch = 0;      // L2 look-ahead of the next matmul's weights: measured neutral on B200 (profiles/r1_gemv_diag.md), off
    int           opt_cpu_exact   = 0;      // parity mode (exact.cu, fattn.cu): every float sum in the order of the reference's AVX2 CPU build, the fp16
                                            // V accumulator of f16-cache attention, correctly rounded exp/sin/cos.  Slow; proves summation order is the only difference
    int           opt_debug_skip  = 0;      // timing experiments only: bit 0 flash_attn, 1 rope+store, 2 GEMV are not launched
    GraphCache *  graph_cache = nullptr;
    // live-tile map of the attention mask (fattn.cu): built by the first FLASH_ATTN_EXT of a graph that uses a given mask, reused by
    // the other layers; dropped at every graph_compute / compute_op entry and when an op writes into the mask
    bool          fa_map_valid = false;
    uintptr_t     fa_map_mask = 0, fa_map_mask_end = 0;
    int64_t       fa_map_key[4] = {0, 0, 0, 0};        // m_nb1, n_kv, n_q, QC
    b200_comm *   comm = nullptr;       // tensor-parallel communicator (comm.cu); NULL = single GPU
    // row-split matmuls driven from ONE host thread (ggml_backend_split_buffer_type): a context + join event per peer device
    b200_ctx *    split_peer[16] = {nullptr};
    cudaEvent_t   split_join[16] = {nullptr};
    cudaEvent_t   split_fork = nullptr;
    int64_t       split_ops = 0;                // executed row-split matmuls (tests)
    bool          capturing = false;
    void *        prof_buf = nullptr;   // debug: per-CTA timestamps (b200_debug_set_prof)
    int           prof_launch = 0;

    void *get_scratch(int slot, size_t size);   // grows (sync + realloc) when too small; nullptr on OOM
};

enum { SCRATCH_ACT = 0, SCRATCH_FATTN = 1, SCRATCH_MOE = 2, SCRATCH_MISC = 3, SCRATCH_FUSE = 4, SCRATCH_FAMAP = 5, SCRATCH_COUNT = 6 };

// op entry points (each in its own .cu); all asynchronous on ctx->stream
int op_mul_mat(b200_ctx *ctx, const b200_op *op);
int op_mul_mat_id(b200_ctx *ctx, const b200_op *op);
int op_flash_attn_ext(b200_ctx *ctx, const b200_op *op);
int op_glue(b200_ctx *ctx, const b200_op *op);          // everything else
bool supports_mul_mat(const b200_op *op);
bool supports_mul_mat_id(const b200_op *op);
bool supports_flash_attn_ext(const b200_op *op);
bool supports_glue(const b200_op *op);
int op_allreduce(b200_ctx *ctx, const b200_op *op);     // comm.cu
bool supports_allreduce(const b200_op *op);
int comm_check(b200_ctx *ctx);                          // comm.cu: B200_ERR_FAILED if an all-reduce timed out waiting for a peer

// rope parameters of the rope and rope+store kernels (glue.cu)
struct RopeParams {
    int n_dims, mode, n_ctx_orig;
    float freq_base, freq_scale, ext_factor, attn_factor, beta_fast, beta_slow;
    float theta_scale, corr0, corr1;
    int exact;        // cpu-exact mode: glibc's sinf/cosf restated (common.cuh), which the CPU backend calls; CUDA's sinf/cosf are
                      // 1-2 ulp off here and there and every ulp can flip a KV-store / activation rounding downstream
};

// fused ROPE(q) + ROPE(k) + KV-store of k and v for a decode ubatch (glue.cu); q/k/v are contiguous [D, heads, T] f32
struct RopeStoreDesc {
    const float *q, *k, *v;
    const int32_t *pos;
    const float *freq_factors;          // optional [D/2]
    float *q_out; uint64_t q_out_nb1, q_out_nb2;     // roped q, byte strides of head and token
    void *k_dst, *v_dst;                // cache rows of token 0 of this ubatch (layout [T][Hkv][D] in the cache type)
    void *const *k_dst_ind, *const *v_dst_ind;       // when non-NULL the destinations are read from device memory (CUDA-graph replay)
    int D, H, Hkv, T, kv_type;
    int32_t rope_params[16];
    int use_pdl;
};
int launch_rope_store(b200_ctx *ctx, const RopeStoreDesc &d);

// quantise f32 activations [K, ncols] (column byte stride nb1) into the scratch layout above
int launch_quantize_act(b200_ctx *ctx, int q8k, const float *x, size_t x_col_stride_bytes, int64_t K, int64_t ncols,
                        uint8_t *scratch);
// decode GEMV over pre-quantised activations (gemv.cu)
// cpu-exact matmul over pre-quantised activations (exact.cu)
struct ExactMoe {             // MUL_MAT_ID through the exact kernel: column = (token, slot) pair
    const char *ids; uint64_t ids_nb0, ids_nb1; int n_used, b_ne1; size_t expert_stride, d_nb1, d_nb2;   // d_nb*: dst element strides
};
int launch_mul_mat_exact(b200_ctx *ctx, int type, const uint8_t *W, size_t rb, int64_t N, int64_t K, const uint8_t *act, int64_t ncols,
                         float *dst, size_t dst_stride, const ExactMoe *moe = nullptr);
int launch_gemv(b200_ctx *ctx, int type, const uint8_t *W, size_t row_bytes, int64_t N, int64_t K, const uint8_t *act,
                int ncols, float *dst, size_t dst_col_stride_elems, bool w_const);
// small-batch (<= 32 columns) weight-streaming matmul on mma.sync s8 (gemv_mma.cu)
bool gemv_mma_supported(int type, int64_t N, int64_t K, int64_t M);
int launch_gemv_mma(b200_ctx *ctx, int type, const uint8_t *W, size_t rb, int64_t N, int64_t K, const uint8_t *act, int ncols,
                    float *dst, size_t dst_stride, bool stream_once, bool w_const, const float *residual = nullptr);
// prompt-batch GEMM on mma.sync s8 for all five formats (gemm_mma.cu)
bool gemm_mma_supported(int type, int64_t N, int64_t K, int64_t M);
int gemm_mma_run(b200_ctx *ctx, int type, const uint8_t *W, size_t rb, int64_t N, int64_t K, const float *x, size_t x_stride, int64_t M, float *dst,
                 size_t dst_stride);
// MUL_MAT_ID routing tables built on the device (mulmat.cu) for the grouped small-batch kernel
struct MmGroupDesc {
    const int32_t *off, *pairs;          // [E + 1] first pair of every expert; pair ids (token * n_used + slot) sorted by expert
    int E, n_used, b_ne1, max_chunks;    // max_chunks: upper bound of sum_e ceil(count_e / 32) = grid.y
    size_t expert_stride, d_nb1, d_nb2;  // bytes between expert matrices; dst element strides of slot and token
};
int gemm_mma_run_grouped(b200_ctx *ctx, int type, const uint8_t *W, size_t rb, int64_t N, int64_t K, const float *x, size_t x_stride, const MmGroupDesc &g, float *dst);
int launch_gemv_mma_grouped(b200_ctx *ctx, int type, const uint8_t *W, size_t rb, int64_t N, int64_t K, const uint8_t *act, const MmGroupDesc &g, float *dst);
int launch_act_prologue(b200_ctx *ctx, int mode, const float *x, size_t x_stride_bytes, const float *x2, float eps, int64_t K, int ncols, int q8k,
                        uint8_t *scratch);

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
#ifdef __CUDACC__

// expf exactly as the reference CPU backend computes it inside silu / soft_max on its SIMD builds: ggml_v_expf
// (ggml-cpu.c:2116-2153, the same polynomial on AVX2, AVX512, SSE2 and NEON), restated per lane with explicit FMAs.
// The vector code's result for a lane does not depend on the other lanes, so this scalar form is bit-identical.  Using it
// (instead of CUDA's expf, which differs by an ulp here and there) makes silu(gate)*up identical to the CPU's, so the
// activation quantiser of the down projection sees the same values and rounds the same way.
__device__ __forceinline__ float ggml_v_expf_lane(float x) {
    const float r = 0x1.8p23f;
    const float z = __fmaf_rn(x, 0x1.715476p+0f, r);
    const float n = __fsub_rn(z, r);
    const float b = __fmaf_rn(-n, 0x1.7f7d1cp-20f, __fmaf_rn(-n, 0x1.62e4p-1f, x));
    const uint32_t e = __float_as_uint(z) << 23;
    const float k = __uint_as_float(e + 0x3f800000u);
    const float an = fabsf(n);
    const float u = __fmul_rn(b, b);
    const float j = __fmaf_rn(__fmaf_rn(__fmaf_rn(0x1.0e4020p-7f, b, 0x1.573e2ep-5f), u, __fmaf_rn(0x1.555e66p-3f, b, 0x1.fffdb6p-2f)), u,
                              __fmul_rn(0x1.ffffecp-1f, b));
    if (!(an > 126.0f)) return __fmaf_rn(j, k, k);
    const uint32_t g = n <= 0.0f ? 0x82000000u : 0u;
    const float s1 = __uint_as_float(g + 0x7f000000u), s2 = __uint_as_float(e - g);
    if (an > 192.0f) return __fmul_rn(s1, s1);
    return __fmul_rn(__fmaf_rn(s2, j, s2), s1);
}
// ---- libm of the reference host, restated (cpu-exact mode only) ---------------------------------------------------------
// The CPU backend calls glibc's sinf / cosf (rope) and expf (flash-attention softmax weights).  glibc >= 2.28 implements them
// with the ARM optimized-routines algorithms (sysdeps/ieee754/flt-32/s_sinf.c, s_cosf.c, e_expf.c, sincosf_data.c,
// e_exp2f_data.c: glibc is not part of /root/reference; published algorithm, LGPL): double-precision polynomials on a
// quadrant / 2^(k/32) table reduction, result rounded to float once.  They are accurate to ~0.5 ulp but NOT correctly
// rounded, so neither CUDA's sinf/expf nor a correctly rounded (float)sin((double)x) agrees with them bit for bit (the
// latter differs on ~1.3% of inputs); with a chaotic consumer (fp16 accumulator, q8 quantisers) every such ulp matters.
// These restatements use explicit double FMAs where the x86-64 FMA build of glibc contracts them; they were checked
// bit-identical to the libm of this image over 60M random arguments each, |x| up to 1.4e5 (tools/check_libm_restatement.c).
__device__ __forceinline__ float glibc_sincos_poly(double x, double x2, int tbl, int n) {
    // __sincosf_table[tbl]: tbl 1 negates the cosine coefficients
    const double sg = tbl ? -1.0 : 1.0;
    if ((n & 1) == 0) {
        const double x3 = __dmul_rn(x, x2), s1 = __fma_rn(x2, -0x1.994eb3774cf24p-13, 0x1.1107605230bc4p-7);
        const double x7 = __dmul_rn(x3, x2), s = __fma_rn(x3, -0x1.555545995a603p-3, x);
        return (float)__fma_rn(x7, s1, s);
    }
    const double x4 = __dmul_rn(x2, x2);
    const double c2 = __fma_rn(x2, sg * 0x1.99343027bf8c3p-16, sg * -0x1.6c087e89a359dp-10);
    const double c1 = __fma_rn(x2, sg * -0x1.ffffffd0c621cp-2, sg * 0x1p0);
    const double x6 = __dmul_rn(x4, x2), c = __fma_rn(x4, sg * 0x1.55553e1068f19p-5, c1);
    return (float)__fma_rn(x6, c2, c);
}
__device__ __forceinline__ double glibc_reduce_large(uint32_t xi, int &np) {
    // __inv_pio4: bits of 4/pi, one byte further per entry
    const uint32_t inv_pio4[24] = {0xa2, 0xa2f9, 0xa2f983, 0xa2f9836e, 0xf9836e4e, 0x836e4e44, 0x6e4e4415, 0x4e441529, 0x441529fc, 0x1529fc27,
                                   0x29fc2757, 0xfc2757d1, 0x2757d1f5, 0x57d1f534, 0xd1f534dd, 0xf534ddc0, 0x34ddc0db, 0xddc0db62, 0xc0db6295,
                                   0xdb629599, 0x6295993c, 0x95993c43, 0x993c4390, 0x3c439041};
    const uint32_t *arr = &inv_pio4[(xi >> 26) & 15];
    const int shift = (xi >> 23) & 7;
    xi = (xi & 0xffffffu) | 0x800000u;
    xi <<= shift;
    uint64_t res0 = (uint64_t)(uint32_t)(xi * arr[0]);
    const uint64_t res1 = (uint64_t)xi * arr[4], res2 = (uint64_t)xi * arr[8];
    res0 = (res2 >> 32) | (res0 << 32);
    res0 += res1;
    const uint64_t n = (res0 + (1ULL << 61)) >> 62;
    res0 -= n << 62;
    np = (int)n;
    return __dmul_rn((double)(int64_t)res0, 0x1.921FB54442D18p-62);
}
__device__ __forceinline__ void glibc_sincosf(float y, float &sn, float &cs) {
    const uint32_t top = (__float_as_uint(y) >> 20) & 0x7ffu;
    double x = (double)y;
    if (top < ((0x3f490fdbu >> 20) & 0x7ffu)) {                         // |y| < pi/4
        const double x2 = __dmul_rn(x, x);
        if (top < ((0x39800000u >> 20) & 0x7ffu)) { sn = y; cs = 1.0f; return; }      // |y| < 2^-12
        sn = glibc_sincos_poly(x, x2, 0, 0);
        cs = glibc_sincos_poly(x, x2, 0, 1);
        return;
    }
    int n, add = 0;
    if (top < ((0x42f00000u >> 20) & 0x7ffu)) {                          // |y| < 120: reduce_fast
        const double r = __dmul_rn(x, 0x1.45F306DC9C883p+23);
        n = ((int32_t)r + 0x800000) >> 24;
        x = __fma_rn(-(double)n, 0x1.921FB54442D18p0, x);
    } else {
        const uint32_t xi = __float_as_uint(y);
        add = (int)(xi >> 31);
        x = glibc_reduce_large(xi, n);
    }
    const int q = (n + add) & 3;
    const double sgn = (q == 1 || q == 2) ? -1.0 : 1.0;                   // sign[] = {1, -1, -1, 1}
    const int tbl = ((n + add) & 2) ? 1 : 0;
    const double xs = __dmul_rn(x, sgn), x2 = __dmul_rn(x, x);
    sn = glibc_sincos_poly(xs, x2, tbl, n);
    cs = glibc_sincos_poly(xs, x2, tbl, n ^ 1);
}
__device__ __forceinline__ float glibc_expf(float x) {
    const uint32_t abstop = (__float_as_uint(x) >> 20) & 0x7ffu;
    if (abstop >= (0x42b00000u >> 20)) {                                  // |x| >= 88 or nan
        if (x == -INFINITY) return 0.0f;
        if (abstop >= (0x7f800000u >> 20)) return x + x;
        if (x > 0x1.62e42ep6f) return INFINITY;
        if (x < -0x1.9fe368p6f) return 0.0f;
    }
    // __exp2f_data.tab[i] = bits(2^(i/32)) - (i << 47)
    const uint64_t tab[32] = {
        0x3ff0000000000000, 0x3fefd9b0d3158574, 0x3fefb5586cf9890f, 0x3fef9301d0125b51, 0x3fef72b83c7d517b, 0x3fef54873168b9aa,
        0x3fef387a6e756238, 0x3fef1e9df51fdee1, 0x3fef06fe0a31b715, 0x3feef1a7373aa9cb, 0x3feedea64c123422, 0x3feece086061892d,
        0x3feebfdad5362a27, 0x3feeb42b569d4f82, 0x3feeab07dd485429, 0x3feea47eb03a5585, 0x3feea09e667f3bcd, 0x3fee9f75e8ec5f74,
        0x3feea11473eb0187, 0x3feea589994cce13, 0x3feeace5422aa0db, 0x3feeb737b0cdc5e5, 0x3feec49182a3f090, 0x3feed503b23e255d,
        0x3feee89f995ad3ad, 0x3feeff76f2fb5e47, 0x3fef199bdd85529c, 0x3fef3720dcef9069, 0x3fef5818dcfba487, 0x3fef7c97337b9b5f,
        0x3fefa4afa2a490da, 0x3fefd0765b6e4540};
    const double xd = (double)x, IL = 0x1.71547652b82fep+5;               // InvLn2N = N / ln 2, N = 32
    double kd = __fma_rn(IL, xd, 0x1.8p+52);
    const uint64_t ki = (uint64_t)__double_as_longlong(kd);
    kd = __dadd_rn(kd, -0x1.8p+52);
    const double r = __fma_rn(IL, xd, -kd);
    const uint64_t t = tab[ki & 31] + (ki << 47);
    const double s = __longlong_as_double((long long)t);
    const double z = __fma_rn(0x1.c6af84b912394p-5 / 32 / 32 / 32, r, 0x1.ebfce50fac4f3p-3 / 32 / 32);
    const double r2 = __dmul_rn(r, r);
    double yv = __fma_rn(0x1.62e42ff0c52d6p-1 / 32, r, 1.0);
    yv = __fma_rn(z, r2, yv);
    return (float)__dmul_rn(yv, s);
}

__device__ __forceinline__ void rope_sincos(float th, int exact, float &s, float &c) {
    if (exact) glibc_sincosf(th, s, c);
    else { s = sinf(th); c = cosf(th); }
}

// ggml_v_silu (ggml-cpu.c:2156-2164): x / (1 + expf(0 - x)), IEEE division
__device__ __forceinline__ float ggml_silu_lane(float x) {
    return __fdiv_rn(x, __fadd_rn(1.0f, ggml_v_expf_lane(__fsub_rn(0.0f, x))));
}

__device__ __forceinline__ float warp_reduce_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_reduce_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ int warp_reduce_sum_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ float half_bits_to_float(uint32_t h16) {
    return __half2float(__ushort_as_half((unsigned short)(h16 & 0xffffu)));
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier (Hopper+/Blackwell producer-consumer pipeline) ----
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {}
}
// 1-D bulk async copy global -> shared, completion counted on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_g2s_hint(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(smem_dst)),
        "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
// programmatic dependent launch
__device__ __forceinline__ uint64_t l2_policy_evict_normal() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

#endif  // __CUDACC__
