// glue.cu -- the ops that sit between the matmuls of a llama / mixtral graph.
//
// Replaces norm.cu (rms_norm_f32), rope.cu (rope_norm/neox + YaRN + freq factors), cpy.cu (f32->f16/q8_0/q4_0
// KV store, cont), binbcast.cu, unary.cu (silu), getrows.cu, softmax.cu, argsort.cu, sumrows.cu, scale.cu
// of ggml-cuda.  Arithmetic follows the CPU oracle (ggml-cpu.c), including where it accumulates in double
// (rms_norm, sum_rows, soft_max) and the multiplicative theta recurrence of rope, so results differ from
// the CPU backend only by libm-vs-CUDA expf/sinf/cosf ulps.
#include "common.cuh"
#include <cuda_bf16.h>

namespace {

struct Idx4 { int64_t i0, i1, i2, i3; };
__device__ __forceinline__ Idx4 unravel(int64_t e, const int64_t ne[4]) {
    Idx4 r;
    r.i0 = e % ne[0]; e /= ne[0];
    r.i1 = e % ne[1]; e /= ne[1];
    r.i2 = e % ne[2];
    r.i3 = e / ne[2];
    return r;
}

__device__ __forceinline__ double block_reduce_sum_d(double v, double *sh) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if ((threadIdx.x & 31) == 0) sh[w] = v;
    __syncthreads();
    double t = 0.0;
    for (int i = 0; i < nw; i++) t += sh[i];     // fixed order -> deterministic
    __syncthreads();
    return t;
}
__device__ __forceinline__ float block_reduce_max_f(float v, float *sh) {
    v = warp_reduce_max(v);
    const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if ((threadIdx.x & 31) == 0) sh[w] = v;
    __syncthreads();
    float t = -INFINITY;
    for (int i = 0; i < nw; i++) t = fmaxf(t, sh[i]);
    __syncthreads();
    return t;
}

// ---------------------------------------------------------------------------------------------- rms_norm (+mul)
// ggml_compute_forward_rms_norm_f32: sum(x*x) in double, mean=(float)(sum/n), scale=1/sqrtf(mean+eps), y=x*scale
template <bool MUL>
__global__ void __launch_bounds__(256) b200_rms_norm_kernel(b200_tensor x, b200_tensor w, b200_tensor y, float eps) {
    __shared__ double sh[8];
    const int64_t row = blockIdx.x;
    const int64_t i1 = row % x.ne[1], i2 = (row / x.ne[1]) % x.ne[2], i3 = row / (x.ne[1] * x.ne[2]);
    const float *xp = (const float *)((const char *)x.data + i1 * x.nb[1] + i2 * x.nb[2] + i3 * x.nb[3]);
    float *yp = (float *)((char *)y.data + i1 * y.nb[1] + i2 * y.nb[2] + i3 * y.nb[3]);
    const int64_t n = x.ne[0];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) { const float v = xp[i]; s += (double)__fmul_rn(v, v); }
    s = block_reduce_sum_d(s, sh);
    const float mean = (float)(s / (double)n);
    const float scale = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(mean, eps)));
    const float *wp = nullptr;
    if (MUL) wp = (const float *)((const char *)w.data + (i1 % w.ne[1]) * w.nb[1] + (i2 % w.ne[2]) * w.nb[2] + (i3 % w.ne[3]) * w.nb[3]);
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        float v = __fmul_rn(xp[i], scale);
        if (MUL) v = __fmul_rn(v, wp[i % w.ne[0]]);
        yp[i] = v;
    }
}

// ---------------------------------------------------------------------------------------------- binary broadcast / unary
enum { BIN_ADD, BIN_SUB, BIN_MUL, BIN_DIV };
template <int OP> __device__ __forceinline__ float bin(float a, float b) {
    return OP == BIN_ADD ? __fadd_rn(a, b) : OP == BIN_SUB ? __fsub_rn(a, b) : OP == BIN_MUL ? __fmul_rn(a, b) : __fdiv_rn(a, b);
}
template <int OP>
__global__ void __launch_bounds__(256) b200_bin_bcast_kernel(b200_tensor a, b200_tensor b, b200_tensor d, int64_t total) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const Idx4 i = unravel(e, d.ne);
    const float av = *(const float *)((const char *)a.data + i.i0 * a.nb[0] + i.i1 * a.nb[1] + i.i2 * a.nb[2] + i.i3 * a.nb[3]);
    const float bv = *(const float *)((const char *)b.data + (i.i0 % b.ne[0]) * b.nb[0] + (i.i1 % b.ne[1]) * b.nb[1] +
                                      (i.i2 % b.ne[2]) * b.nb[2] + (i.i3 % b.ne[3]) * b.nb[3]);
    *(float *)((char *)d.data + i.i0 * d.nb[0] + i.i1 * d.nb[1] + i.i2 * d.nb[2] + i.i3 * d.nb[3]) = bin<OP>(av, bv);
}
// fast path: everything contiguous, b is either the same shape or one row broadcast over all rows; n % 4 == 0
template <int OP>
__global__ void __launch_bounds__(256) b200_bin_fast_kernel(const float4 *a, const float4 *b, float4 *d, int64_t n4, int64_t brow4) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n4) return;
    const float4 av = a[e], bv = b[brow4 ? e % brow4 : e];
    float4 r;
    r.x = bin<OP>(av.x, bv.x); r.y = bin<OP>(av.y, bv.y); r.z = bin<OP>(av.z, bv.z); r.w = bin<OP>(av.w, bv.w);
    d[e] = r;
}

enum { UN_SILU, UN_GELU, UN_RELU, UN_TANH, UN_SIGMOID, UN_SCALE, UN_SWIGLU };
template <int OP> __device__ __forceinline__ float unary(float x, float p) {
    switch (OP) {
        case UN_SILU:    return ggml_silu_lane(x);
        case UN_GELU:    return 0.5f * x * (1.0f + tanhf(0.79788456080286535587989211986876f * x * (1.0f + 0.044715f * x * x)));
        case UN_RELU:    return fmaxf(x, 0.0f);
        case UN_TANH:    return tanhf(x);
        case UN_SIGMOID: return __fdiv_rn(1.0f, 1.0f + expf(-x));
        case UN_SCALE:   return __fmul_rn(x, p);
        default:         return x;
    }
}
template <int OP>
__global__ void __launch_bounds__(256) b200_unary_kernel(const float *x, const float *u, float *y, int64_t n, float p) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    if (OP == UN_SWIGLU) y[e] = __fmul_rn(unary<UN_SILU>(x[e], 0.0f), u[e]);
    else y[e] = unary<OP>(x[e], p);
}

// ---------------------------------------------------------------------------------------------- rope
// ggml_compute_forward_rope_f32 (ggml-cpu.c:10671-10800) with ggml_rope_cache_init (:10597-10613): theta starts at
// pos and is multiplied by theta_scale once per pair (sequential product, reproduced here), YaRN mix per rope_yarn.
template <typename T>
__global__ void __launch_bounds__(128) b200_rope_kernel(b200_tensor x, b200_tensor pos, b200_tensor ff, b200_tensor y, RopeParams rp, int has_ff) {
    // grid: (ne2 tokens, ne1 heads, ne3); threads over pairs
    const int64_t i2 = blockIdx.x, i1 = blockIdx.y, i3 = blockIdx.z;
    const char *xp = (const char *)x.data + i1 * x.nb[1] + i2 * x.nb[2] + i3 * x.nb[3];
    char *yp = (char *)y.data + i1 * y.nb[1] + i2 * y.nb[2] + i3 * y.nb[3];
    const int p = ((const int32_t *)pos.data)[i2];
    const bool neox = (rp.mode & 2) != 0;
    const int64_t ne0 = x.ne[0];
    for (int64_t ip = threadIdx.x; ip < ne0 / 2; ip += blockDim.x) {
        const int64_t i0 = 2 * ip;
        if (i0 < rp.n_dims) {
            float theta = (float)p;
            for (int64_t k = 0; k < ip; k++) theta = __fmul_rn(theta, rp.theta_scale);
            const float f = has_ff ? ((const float *)ff.data)[ip] : 1.0f;
            const float te = __fdiv_rn(theta, f);
            float ti = __fmul_rn(rp.freq_scale, te), th = ti, ms = rp.attn_factor;
            if (rp.ext_factor != 0.0f) {
                const float yv = __fdiv_rn((float)(i0 / 2) - rp.corr0, fmaxf(0.001f, rp.corr1 - rp.corr0));
                const float ramp = __fmul_rn(1.0f - fminf(1.0f, fmaxf(0.0f, yv)), rp.ext_factor);
                th = __fadd_rn(__fmul_rn(ti, 1.0f - ramp), __fmul_rn(te, ramp));
                ms = __fmul_rn(ms, 1.0f + 0.1f * logf(__fdiv_rn(1.0f, rp.freq_scale)));
            }
            float sn, cs;
            rope_sincos(th, rp.exact, sn, cs);
            const float c = __fmul_rn(cs, ms), s = __fmul_rn(sn, ms);
            const int64_t ia = neox ? ip : i0, ib = neox ? ip + rp.n_dims / 2 : i0 + 1;
            const float x0 = (float)((const T *)xp)[ia], x1 = (float)((const T *)xp)[ib];
            ((T *)yp)[ia] = (T)__fsub_rn(__fmul_rn(x0, c), __fmul_rn(x1, s));
            ((T *)yp)[ib] = (T)__fadd_rn(__fmul_rn(x0, s), __fmul_rn(x1, c));
        } else {
            ((T *)yp)[i0] = ((const T *)xp)[i0];
            ((T *)yp)[i0 + 1] = ((const T *)xp)[i0 + 1];
        }
    }
}

// ---------------------------------------------------------------------------------------------- cpy / cont / KV store
template <typename TS, typename TD> __device__ __forceinline__ TD cvt(TS v);
template <> __device__ __forceinline__ float cvt<float, float>(float v) { return v; }
template <> __device__ __forceinline__ __half cvt<float, __half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ float cvt<__half, float>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ __half cvt<__half, __half>(__half v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 cvt<float, __nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ float cvt<__nv_bfloat16, float>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ int32_t cvt<int32_t, int32_t>(int32_t v) { return v; }

// flat-index copy: element e of src (src's logical order) -> element e of dst (dst's logical order)
template <typename TS, typename TD>
__global__ void __launch_bounds__(256) b200_cpy_kernel(b200_tensor s, b200_tensor d, int64_t total) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const Idx4 a = unravel(e, s.ne), b = unravel(e, d.ne);
    const TS v = *(const TS *)((const char *)s.data + a.i0 * s.nb[0] + a.i1 * s.nb[1] + a.i2 * s.nb[2] + a.i3 * s.nb[3]);
    *(TD *)((char *)d.data + b.i0 * d.nb[0] + b.i1 * d.nb[1] + b.i2 * d.nb[2] + b.i3 * d.nb[3]) = cvt<TS, TD>(v);
}

__device__ __forceinline__ const char *blk_ptr(const b200_tensor &t, int64_t blk_index, int be) {
    // pointer to block `blk_index` (flat, in blocks of `be` elements along dim 0)
    const int64_t nb0 = t.ne[0] / be;
    int64_t r = blk_index;
    const int64_t b0 = r % nb0; r /= nb0;
    const int64_t i1 = r % t.ne[1]; r /= t.ne[1];
    const int64_t i2 = r % t.ne[2];
    const int64_t i3 = r / t.ne[2];
    return (const char *)t.data + b0 * t.nb[0] * (t.type == B200_TYPE_F32 ? be : 1) + i1 * t.nb[1] + i2 * t.nb[2] + i3 * t.nb[3];
}

// f32 -> q8_0 / q4_0, one thread per 32-element block (quantize_row_q8_0 AVX2 semantics / quantize_row_q4_0_ref)
template <int DT>
__global__ void __launch_bounds__(128) b200_cpy_f32_q_kernel(b200_tensor s, b200_tensor d, int64_t nblocks) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    const float *xp = (const float *)blk_ptr(s, b, 32);
    uint8_t *o = (uint8_t *)blk_ptr(d, b, 32);
    float v[32];
#pragma unroll
    for (int j = 0; j < 32; j += 4) { const float4 t = *(const float4 *)(xp + j); v[j] = t.x; v[j + 1] = t.y; v[j + 2] = t.z; v[j + 3] = t.w; }
    if (DT == B200_TYPE_Q8_0) {
        float amax = 0.0f;
#pragma unroll
        for (int j = 0; j < 32; j++) amax = fmaxf(amax, fabsf(v[j]));
        const float dd = __fdiv_rn(amax, 127.0f);
        const float id = amax != 0.0f ? __fdiv_rn(127.0f, amax) : 0.0f;
        *(__half *)o = __float2half_rn(dd);
#pragma unroll
        for (int j = 0; j < 32; j++) o[2 + j] = (uint8_t)(int8_t)__float2int_rn(__fmul_rn(v[j], id));
    } else {
        float amax = 0.0f, mx = 0.0f;
#pragma unroll
        for (int j = 0; j < 32; j++) { const float a = fabsf(v[j]); if (a > amax) { amax = a; mx = v[j]; } }
        const float dd = __fdiv_rn(mx, -8.0f);
        const float id = dd != 0.0f ? __fdiv_rn(1.0f, dd) : 0.0f;
        *(__half *)o = __float2half_rn(dd);
#pragma unroll
        for (int j = 0; j < 16; j++) {
            const float x0 = __fmul_rn(v[j], id), x1 = __fmul_rn(v[16 + j], id);
            int a = (int)(int8_t)(int)__fadd_rn(x0, 8.5f), c = (int)(int8_t)(int)__fadd_rn(x1, 8.5f);
            a = a > 15 ? 15 : a; c = c > 15 ? 15 : c;
            o[2 + j] = (uint8_t)((a & 0xff) | (c << 4));
        }
    }
}

// dequantise one element of a quantised row (used by get_rows and q->f32 cpy); scalar, not a hot path
__device__ float dequant_elem(int type, const uint8_t *row, int64_t e) {
    switch (type) {
        case B200_TYPE_F32: return ((const float *)row)[e];
        case B200_TYPE_F16: return __half2float(((const __half *)row)[e]);
        case B200_TYPE_BF16: return __bfloat162float(((const __nv_bfloat16 *)row)[e]);
        case B200_TYPE_Q4_0: {
            const uint8_t *b = row + (e / 32) * 18; const int j = (int)(e % 32);
            const float d = __half2float(*(const __half *)b);
            const int q = j < 16 ? (b[2 + j] & 0x0f) : (b[2 + j - 16] >> 4);
            return __fmul_rn((float)(q - 8), d);
        }
        case B200_TYPE_Q8_0: {
            const uint8_t *b = row + (e / 32) * 34;
            return __fmul_rn((float)(int8_t)b[2 + e % 32], __half2float(*(const __half *)b));
        }
        case B200_TYPE_Q4_K: case B200_TYPE_Q5_K: {
            const int bytes = type == B200_TYPE_Q4_K ? 144 : 176;
            const uint8_t *b = row + (e / 256) * bytes; const int r = (int)(e % 256), j = r >> 5;
            const float d = __half2float(*(const __half *)b), dmin = __half2float(*(const __half *)(b + 2));
            const uint8_t *s = b + 4;
            int sc, mn;
            if (j < 4) { sc = s[j] & 63; mn = s[j + 4] & 63; }
            else { sc = (s[j + 4] & 0x0f) | ((s[j - 4] >> 6) << 4); mn = (s[j + 4] >> 4) | ((s[j] >> 6) << 4); }
            const uint8_t *qs = b + (type == B200_TYPE_Q4_K ? 16 : 48);
            const uint8_t byte = qs[32 * (r >> 6) + (r & 31)];
            int q = (r & 32) ? (byte >> 4) : (byte & 0x0f);
            if (type == B200_TYPE_Q5_K) q |= ((b[16 + (r & 31)] >> j) & 1) << 4;
            return __fsub_rn(__fmul_rn(__fmul_rn(d, (float)sc), (float)q), __fmul_rn(dmin, (float)mn));
        }
        case B200_TYPE_Q6_K: {
            const uint8_t *b = row + (e / 256) * 210; const int r = (int)(e % 256);
            const int h = r >> 7, t = (r & 127) >> 5, l = r & 31;
            const uint8_t lb = b[64 * h + l + 32 * (t & 1)];
            const int lo = t < 2 ? (lb & 0x0f) : (lb >> 4);
            const int hi = (b[128 + 32 * h + l] >> (2 * t)) & 3;
            const int q = (lo | (hi << 4)) - 32;
            const float d = __half2float(*(const __half *)(b + 208));
            const int sc = (int8_t)b[192 + 8 * h + 2 * t + l / 16];
            return __fmul_rn(__fmul_rn(d, (float)sc), (float)q);
        }
    }
    return 0.0f;
}

__global__ void __launch_bounds__(256) b200_cpy_q_f32_kernel(b200_tensor s, b200_tensor d, int64_t total) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const Idx4 a = unravel(e, s.ne), b = unravel(e, d.ne);
    const uint8_t *row = (const uint8_t *)s.data + a.i1 * s.nb[1] + a.i2 * s.nb[2] + a.i3 * s.nb[3];
    *(float *)((char *)d.data + b.i0 * d.nb[0] + b.i1 * d.nb[1] + b.i2 * d.nb[2] + b.i3 * d.nb[3]) = dequant_elem(s.type, row, a.i0);
}

// same-type copy of quantised blocks between strided views (KV defrag: llama-context.cpp build_kv_self_defrag moves cache rows with
// ggml_cpy(view_src, view_dst)); a block is the element, 2-byte granules (q4_0 / q8_0 blocks are only 2-byte aligned)
__global__ void __launch_bounds__(256) b200_cpy_qblocks_kernel(b200_tensor s, b200_tensor d, int64_t nblocks, int be, int bb) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nblocks) return;
    int64_t sne[4] = {s.ne[0] / be, s.ne[1], s.ne[2], s.ne[3]}, dne[4] = {d.ne[0] / be, d.ne[1], d.ne[2], d.ne[3]};
    const Idx4 a = unravel(i, sne), b = unravel(i, dne);
    const unsigned short *sp = (const unsigned short *)((const char *)s.data + a.i0 * s.nb[0] + a.i1 * s.nb[1] + a.i2 * s.nb[2] + a.i3 * s.nb[3]);
    unsigned short *dp = (unsigned short *)((char *)d.data + b.i0 * d.nb[0] + b.i1 * d.nb[1] + b.i2 * d.nb[2] + b.i3 * d.nb[3]);
    for (int k = 0; k < bb / 2; k++) dp[k] = sp[k];
}

// get_rows: dst[:, i10, i11, i12] = src0[:, idx[i10,i11,i12], i11, i12]
__global__ void __launch_bounds__(256) b200_get_rows_kernel(b200_tensor s, b200_tensor idx, b200_tensor d, int64_t total) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const Idx4 i = unravel(e, d.ne);
    const int32_t r = *(const int32_t *)((const char *)idx.data + i.i1 * idx.nb[0] + i.i2 * idx.nb[1] + i.i3 * idx.nb[2]);
    const uint8_t *row = (const uint8_t *)s.data + (int64_t)r * s.nb[1] + i.i2 * s.nb[2] + i.i3 * s.nb[3];
    *(float *)((char *)d.data + i.i0 * d.nb[0] + i.i1 * d.nb[1] + i.i2 * d.nb[2] + i.i3 * d.nb[3]) = dequant_elem(s.type, row, i.i0);
}

// ---------------------------------------------------------------------------------------------- soft_max
// ggml_compute_forward_soft_max_f32 (ggml-cpu.c:10224-10320): w = x*scale + slope*mask; max; exp(w-max) summed in double
template <typename MT>
__global__ void __launch_bounds__(256) b200_soft_max_kernel(b200_tensor x, b200_tensor mask, b200_tensor y, float scale, float max_bias, int has_mask, int exact) {
    __shared__ double shd[8];
    __shared__ float shf[8];
    const int64_t row = blockIdx.x;
    const int64_t ne00 = x.ne[0], ne01 = x.ne[1], ne02 = x.ne[2];
    const int64_t i1 = row % ne01, i2 = (row / ne01) % ne02, i3 = row / (ne01 * ne02);
    const float *xp = (const float *)((const char *)x.data + i1 * x.nb[1] + i2 * x.nb[2] + i3 * x.nb[3]);
    float *yp = (float *)((char *)y.data + i1 * y.nb[1] + i2 * y.nb[2] + i3 * y.nb[3]);
    float slope = 1.0f;
    if (max_bias > 0.0f) {
        const uint32_t n_head = (uint32_t)ne02, h = (uint32_t)i2;
        const uint32_t n_head_log2 = 1u << (uint32_t)floorf(log2f((float)n_head));
        const float m0 = powf(2.0f, -(max_bias) / n_head_log2), m1 = powf(2.0f, -(max_bias / 2.0f) / n_head_log2);
        slope = h < n_head_log2 ? powf(m0, (float)(h + 1)) : powf(m1, (float)(2 * (h - n_head_log2) + 1));
    }
    const MT *mp = has_mask ? (const MT *)mask.data + (row % ne01) * ne00 : nullptr;   // CPU: (i1 % ne01)*ne00 with i1 = flat row
    float mx = -INFINITY;
    for (int64_t i = threadIdx.x; i < ne00; i += blockDim.x) {
        float w = __fmul_rn(xp[i], scale);
        if (has_mask) w = __fadd_rn(w, __fmul_rn(slope, (float)mp[i]));
        yp[i] = w;
        mx = fmaxf(mx, w);
    }
    mx = block_reduce_max_f(mx, shf);
    double s = 0.0;
    if (exact) {
        // cpu-exact mode: ggml_vec_soft_max_f32's AVX2 path (ggml-cpu.c:2261-2271, 2296-2300): ggml_v_expf on full groups of 8, each group
        // enters the double sum as the float ((v0+v4)+(v2+v6))+((v1+v5)+(v3+v7)), groups in order; leftovers through glibc's expf
        const int64_t n8 = ne00 & ~(int64_t)7;
        for (int64_t i = threadIdx.x; i < ne00; i += blockDim.x) {
            const float d = __fsub_rn(yp[i], mx);
            yp[i] = i < n8 ? ggml_v_expf_lane(d) : glibc_expf(d);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int64_t i = 0; i < n8; i += 8) {
                const float s8 = __fadd_rn(__fadd_rn(__fadd_rn(yp[i], yp[i + 4]), __fadd_rn(yp[i + 2], yp[i + 6])),
                                           __fadd_rn(__fadd_rn(yp[i + 1], yp[i + 5]), __fadd_rn(yp[i + 3], yp[i + 7])));
                t += (double)s8;
            }
            for (int64_t i = n8; i < ne00; i++) t += (double)yp[i];
            shd[0] = t;
        }
        __syncthreads();
        s = shd[0];
    } else {
        for (int64_t i = threadIdx.x; i < ne00; i += blockDim.x) {
            const float v = expf(__fsub_rn(yp[i], mx));
            yp[i] = v;
            s += (double)v;
        }
        s = block_reduce_sum_d(s, shd);
    }
    const float inv = (float)(1.0 / s);
    for (int64_t i = threadIdx.x; i < ne00; i += blockDim.x) yp[i] = __fmul_rn(yp[i], inv);
}

// ---------------------------------------------------------------------------------------------- argsort / sum_rows
// ARGMAX (ggml_vec_argmax_f32, ggml-cpu.c:2393-2401: `max = MAX(max, x[i]); if (max == x[i]) idx = i;` -> the LAST index holding the
// maximum).  Greedy sampling on the device: the host reads 4 bytes per sequence instead of the full-vocabulary logits row.
__global__ void __launch_bounds__(1024) b200_argmax_kernel(b200_tensor a, b200_tensor d) {
    __shared__ float sv[32];
    __shared__ int si[32];
    const int row = blockIdx.x, n = (int)a.ne[0];
    const float *x = (const float *)((const char *)a.data + (size_t)row * a.nb[1]);
    float best = -INFINITY; int bi = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) { const float v = x[i]; if (v >= best) { best = v; bi = i; } }
    auto merge = [](float &v, int &i, float ov, int oi) { if (ov > v || (ov == v && oi > i)) { v = ov; i = oi; } };
    for (int o = 16; o > 0; o >>= 1) merge(best, bi, __shfl_xor_sync(0xffffffffu, best, o), __shfl_xor_sync(0xffffffffu, bi, o));
    if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = best; si[threadIdx.x >> 5] = bi; }
    __syncthreads();
    if (threadIdx.x < 32) {
        best = sv[threadIdx.x]; bi = si[threadIdx.x];
        for (int o = 16; o > 0; o >>= 1) merge(best, bi, __shfl_xor_sync(0xffffffffu, best, o), __shfl_xor_sync(0xffffffffu, bi, o));
        if (threadIdx.x == 0) *(int32_t *)((char *)d.data + (size_t)row * d.nb[0]) = bi;
    }
}

// bitonic sort of one row (ncols <= 1024) in shared memory; ties keep the lower index first like a stable CPU sort
__global__ void b200_argsort_kernel(b200_tensor x, b200_tensor y, int ncols_pad, int desc) {
    extern __shared__ int sidx[];
    const int64_t row = blockIdx.x;
    const int64_t ne00 = x.ne[0];
    const float *xp = (const float *)((const char *)x.data + row * x.nb[1]);
    const int t = threadIdx.x;
    sidx[t] = t;
    __syncthreads();
    auto before = [&](int a, int b) {   // should a come before b ?
        if (a >= ne00) return false;
        if (b >= ne00) return true;
        const float va = xp[a], vb = xp[b];
        if (va == vb) return a < b;
        return desc ? va > vb : va < vb;
    };
    for (int k = 2; k <= ncols_pad; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            const int ixj = t ^ j;
            if (ixj > t) {
                const int a = sidx[t], b = sidx[ixj];
                const bool up = (t & k) == 0;
                if (up ? before(b, a) : before(a, b)) { sidx[t] = b; sidx[ixj] = a; }
            }
            __syncthreads();
        }
    if (t < ne00) ((int32_t *)((char *)y.data + row * y.nb[1]))[t] = sidx[t];
}

__global__ void __launch_bounds__(256) b200_sum_rows_kernel(b200_tensor x, b200_tensor y) {
    __shared__ double sh[8];
    const int64_t row = blockIdx.x;
    const int64_t i1 = row % x.ne[1], i2 = (row / x.ne[1]) % x.ne[2], i3 = row / (x.ne[1] * x.ne[2]);
    const float *xp = (const float *)((const char *)x.data + i1 * x.nb[1] + i2 * x.nb[2] + i3 * x.nb[3]);
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < x.ne[0]; i += blockDim.x) s += (double)xp[i];
    s = block_reduce_sum_d(s, sh);
    if (threadIdx.x == 0) *(float *)((char *)y.data + i1 * y.nb[1] + i2 * y.nb[2] + i3 * y.nb[3]) = (float)s;
}

// ---------------------------------------------------------------------------------------------- helpers
inline float f32_param(const b200_op *op, int i) { float f; memcpy(&f, &op->params[i], 4); return f; }
inline unsigned nblk(int64_t n, int bs) { return (unsigned)((n + bs - 1) / bs); }
inline bool same_shape(const b200_tensor &a, const b200_tensor &b) {
    return a.ne[0] == b.ne[0] && a.ne[1] == b.ne[1] && a.ne[2] == b.ne[2] && a.ne[3] == b.ne[3];
}
inline bool rows_f32_ok(const b200_tensor &t) { return t.type == B200_TYPE_F32 && t.nb[0] == 4; }

float yarn_corr_dim(int n_dims, int n_ctx_orig, float n_rot, float base) {
    return n_dims * logf(n_ctx_orig / (n_rot * 2 * (float)M_PI)) / (2 * logf(base));
}

template <int OP> int launch_bin(b200_ctx *ctx, const b200_op *op) {
    const b200_tensor &a = op->src[0], &b = op->src[1], &d = op->dst;
    const int64_t total = tensor_nelements(d);
    if (total == 0) return B200_OK;
    const bool contig = tensor_is_contiguous(a) && tensor_is_contiguous(b) && tensor_is_contiguous(d);
    const bool al = !(((uintptr_t)a.data | (uintptr_t)b.data | (uintptr_t)d.data) & 15);
    if (contig && al && a.ne[0] % 4 == 0) {
        int64_t brow4 = -1;
        if (same_shape(a, b)) brow4 = 0;
        else if (b.ne[0] == a.ne[0] && b.ne[1] == 1 && b.ne[2] == 1 && b.ne[3] == 1) brow4 = b.ne[0] / 4;
        if (brow4 >= 0) {
            b200_bin_fast_kernel<OP><<<nblk(total / 4, 256), 256, 0, ctx->stream>>>((const float4 *)a.data, (const float4 *)b.data,
                                                                              (float4 *)d.data, total / 4, brow4);
            ctx->launches++;
            CUDA_TRY(cudaGetLastError());
            return B200_OK;
        }
    }
    b200_bin_bcast_kernel<OP><<<nblk(total, 256), 256, 0, ctx->stream>>>(a, b, d, total);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return B200_OK;
}

template <int OP> int launch_unary(b200_ctx *ctx, const b200_op *op, float p) {
    const int64_t n = tensor_nelements(op->dst);
    if (n == 0) return B200_OK;
    b200_unary_kernel<OP><<<nblk(n, 256), 256, 0, ctx->stream>>>((const float *)op->src[0].data,
                                                            OP == UN_SWIGLU ? (const float *)op->src[1].data : nullptr,
                                                            (float *)op->dst.data, n, p);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return B200_OK;
}

bool cpy_pair_ok(int st, int dt) {
    if (st == B200_TYPE_F32) return dt == B200_TYPE_F32 || dt == B200_TYPE_F16 || dt == B200_TYPE_BF16 || dt == B200_TYPE_Q8_0 || dt == B200_TYPE_Q4_0;
    if (st == B200_TYPE_F16) return dt == B200_TYPE_F16 || dt == B200_TYPE_F32;
    if (st == B200_TYPE_BF16) return dt == B200_TYPE_F32;
    if (st == B200_TYPE_I32) return dt == B200_TYPE_I32;
    if (b200_type_is_quant(st)) return dt == B200_TYPE_F32 || dt == st;
    return false;
}

int launch_cpy(b200_ctx *ctx, const b200_tensor &s, const b200_tensor &d) {
    const int64_t total = tensor_nelements(s);
    if (total == 0) return B200_OK;
    const int st = s.type, dt = d.type;
#define CPY_CASE(TS, TD) b200_cpy_kernel<TS, TD><<<nblk(total, 256), 256, 0, ctx->stream>>>(s, d, total)
    if (st == B200_TYPE_F32 && dt == B200_TYPE_F32) CPY_CASE(float, float);
    else if (st == B200_TYPE_F32 && dt == B200_TYPE_F16) CPY_CASE(float, __half);
    else if (st == B200_TYPE_F32 && dt == B200_TYPE_BF16) CPY_CASE(float, __nv_bfloat16);
    else if (st == B200_TYPE_F16 && dt == B200_TYPE_F16) CPY_CASE(__half, __half);
    else if (st == B200_TYPE_F16 && dt == B200_TYPE_F32) CPY_CASE(__half, float);
    else if (st == B200_TYPE_BF16 && dt == B200_TYPE_F32) CPY_CASE(__nv_bfloat16, float);
    else if (st == B200_TYPE_I32 && dt == B200_TYPE_I32) CPY_CASE(int32_t, int32_t);
    else if (st == B200_TYPE_F32 && dt == B200_TYPE_Q8_0) b200_cpy_f32_q_kernel<B200_TYPE_Q8_0><<<nblk(total / 32, 128), 128, 0, ctx->stream>>>(s, d, total / 32);
    else if (st == B200_TYPE_F32 && dt == B200_TYPE_Q4_0) b200_cpy_f32_q_kernel<B200_TYPE_Q4_0><<<nblk(total / 32, 128), 128, 0, ctx->stream>>>(s, d, total / 32);
    else if (b200_type_is_quant(st) && dt == st) {
        const int be = b200_type_block_elems(st), bb = b200_type_block_bytes(st);
        b200_cpy_qblocks_kernel<<<nblk(total / be, 256), 256, 0, ctx->stream>>>(s, d, total / be, be, bb);
    }
    else if (b200_type_is_quant(st) && dt == B200_TYPE_F32) b200_cpy_q_f32_kernel<<<nblk(total, 256), 256, 0, ctx->stream>>>(s, d, total);
    else { b200_set_error("cpy %d -> %d", st, dt); return B200_ERR_UNSUPPORTED; }
#undef CPY_CASE
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return B200_OK;
}


// ---------------------------------------------------------------------------------------------- fused rope + KV store (decode)
// One launch replaces ROPE(q), ROPE(k), CPY(k -> cache), CPY(v -> cache) of a llama attention block
// (llama-graph.cpp:1375-1397 + llama-model.cpp:4133-4143).  Arithmetic is that of the unfused kernels above, in the
// same order: rope result rounded to f32, then the KV-store conversion (f16 RNE / quantize_row_q8_0 / quantize_row_q4_0_ref).
// grid = (H + 2*Hkv head slots, T tokens); block = 64 threads (one per rotated pair, D <= 128... looped for larger D)
template <int KVT>
__global__ void __launch_bounds__(64) b200_rope_store_kernel(const RopeStoreDesc d, RopeParams rp) {
    __shared__ float sh[512];
    if (d.use_pdl) { pdl_trigger(); pdl_wait(); }
    const int slot = blockIdx.x, t = blockIdx.y;
    const int D = d.D, H = d.H, Hkv = d.Hkv;
    const bool is_q = slot < H, is_k = !is_q && slot < H + Hkv;
    const int head = is_q ? slot : (is_k ? slot - H : slot - H - Hkv);
    const float *src = is_q ? d.q + ((size_t)t * H + head) * D : (is_k ? d.k : d.v) + ((size_t)t * Hkv + head) * D;
    if (is_q || is_k) {
        const int p = d.pos[t];
        const bool neox = (rp.mode & 2) != 0;
        float *qo = is_q ? (float *)((char *)d.q_out + (size_t)head * d.q_out_nb1 + (size_t)t * d.q_out_nb2) : sh;
        for (int ip = threadIdx.x; ip < D / 2; ip += blockDim.x) {
            const int i0 = 2 * ip;
            if (i0 < rp.n_dims) {
                float theta = (float)p;
                for (int k = 0; k < ip; k++) theta = __fmul_rn(theta, rp.theta_scale);
                const float f = d.freq_factors ? d.freq_factors[ip] : 1.0f;
                const float te = __fdiv_rn(theta, f);
                float ti = __fmul_rn(rp.freq_scale, te), th = ti, ms = rp.attn_factor;
                if (rp.ext_factor != 0.0f) {
                    const float yv = __fdiv_rn((float)(i0 / 2) - rp.corr0, fmaxf(0.001f, rp.corr1 - rp.corr0));
                    const float ramp = __fmul_rn(1.0f - fminf(1.0f, fmaxf(0.0f, yv)), rp.ext_factor);
                    th = __fadd_rn(__fmul_rn(ti, 1.0f - ramp), __fmul_rn(te, ramp));
                    ms = __fmul_rn(ms, 1.0f + 0.1f * logf(__fdiv_rn(1.0f, rp.freq_scale)));
                }
                float sn, cs;
                rope_sincos(th, rp.exact, sn, cs);
                const float c = __fmul_rn(cs, ms), s = __fmul_rn(sn, ms);
                const int ia = neox ? ip : i0, ib = neox ? ip + rp.n_dims / 2 : i0 + 1;
                const float x0 = src[ia], x1 = src[ib];
                qo[ia] = __fsub_rn(__fmul_rn(x0, c), __fmul_rn(x1, s));
                qo[ib] = __fadd_rn(__fmul_rn(x0, s), __fmul_rn(x1, c));
            } else {
                qo[i0] = src[i0];
                qo[i0 + 1] = src[i0 + 1];
            }
        }
        if (is_q) return;
    } else {
        for (int i = threadIdx.x; i < D; i += blockDim.x) sh[i] = src[i];
    }
    __syncthreads();
    // ---- KV store of the row sh[0..D) into the cache: token t, head `head` ----
    const void *base = is_k ? (d.k_dst_ind ? *d.k_dst_ind : d.k_dst) : (d.v_dst_ind ? *d.v_dst_ind : d.v_dst);
    if (KVT == B200_TYPE_F16) {
        __half *o = (__half *)base + ((size_t)t * Hkv + head) * D;
        for (int i = threadIdx.x; i < D; i += blockDim.x) o[i] = __float2half_rn(sh[i]);
    } else {
        constexpr int BB = KVT == B200_TYPE_Q8_0 ? 34 : 18;
        const int nb = D / 32;
        if (threadIdx.x < nb) {
            const float *v = sh + threadIdx.x * 32;
            uint8_t *o = (uint8_t *)base + (((size_t)t * Hkv + head) * nb + threadIdx.x) * BB;
            if (KVT == B200_TYPE_Q8_0) {
                float amax = 0.0f;
                for (int j = 0; j < 32; j++) amax = fmaxf(amax, fabsf(v[j]));
                const float dd = __fdiv_rn(amax, 127.0f);
                const float id = amax != 0.0f ? __fdiv_rn(127.0f, amax) : 0.0f;
                *(__half *)o = __float2half_rn(dd);
                for (int j = 0; j < 32; j++) o[2 + j] = (uint8_t)(int8_t)__float2int_rn(__fmul_rn(v[j], id));
            } else {
                float amax = 0.0f, mx = 0.0f;
                for (int j = 0; j < 32; j++) { const float a = fabsf(v[j]); if (a > amax) { amax = a; mx = v[j]; } }
                const float dd = __fdiv_rn(mx, -8.0f);
                const float id = dd != 0.0f ? __fdiv_rn(1.0f, dd) : 0.0f;
                *(__half *)o = __float2half_rn(dd);
                for (int j = 0; j < 16; j++) {
                    const float x0 = __fmul_rn(v[j], id), x1 = __fmul_rn(v[16 + j], id);
                    int a = (int)(int8_t)(int)__fadd_rn(x0, 8.5f), c = (int)(int8_t)(int)__fadd_rn(x1, 8.5f);
                    a = a > 15 ? 15 : a; c = c > 15 ? 15 : c;
                    o[2 + j] = (uint8_t)((a & 0xff) | (c << 4));
                }
            }
        }
    }
}

RopeParams make_rope_params_impl(const int32_t *params) {
    RopeParams rp;
    auto f = [&](int i) { float v; memcpy(&v, &params[i], 4); return v; };
    rp.n_dims = params[1]; rp.mode = params[2]; rp.n_ctx_orig = params[4];
    rp.freq_base = f(5); rp.freq_scale = f(6); rp.ext_factor = f(7);
    rp.attn_factor = f(8); rp.beta_fast = f(9); rp.beta_slow = f(10);
    rp.theta_scale = powf(rp.freq_base, -2.0f / rp.n_dims);
    float lo = floorf(yarn_corr_dim(rp.n_dims, rp.n_ctx_orig, rp.beta_fast, rp.freq_base));
    float hi = ceilf(yarn_corr_dim(rp.n_dims, rp.n_ctx_orig, rp.beta_slow, rp.freq_base));
    rp.corr0 = lo < 0 ? 0 : lo;
    rp.corr1 = hi > rp.n_dims - 1 ? (float)(rp.n_dims - 1) : hi;
    rp.exact = 0;
    return rp;
}

}  // namespace

int launch_rope_store(b200_ctx *ctx, const RopeStoreDesc &din) {
    RopeStoreDesc d = din;
    d.use_pdl = ctx->opt_pdl;
    RopeParams rp = make_rope_params_impl(d.rope_params);
    rp.exact = ctx->opt_cpu_exact;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(d.H + 2 * d.Hkv), (unsigned)d.T);
    cfg.blockDim = dim3(64);
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = d.use_pdl ? 1 : 0;
    switch (d.kv_type) {
        case B200_TYPE_F16:  CUDA_TRY(cudaLaunchKernelEx(&cfg, b200_rope_store_kernel<B200_TYPE_F16>, d, rp)); break;
        case B200_TYPE_Q8_0: CUDA_TRY(cudaLaunchKernelEx(&cfg, b200_rope_store_kernel<B200_TYPE_Q8_0>, d, rp)); break;
        case B200_TYPE_Q4_0: CUDA_TRY(cudaLaunchKernelEx(&cfg, b200_rope_store_kernel<B200_TYPE_Q4_0>, d, rp)); break;
        default: b200_set_error("rope_store: kv type %d", d.kv_type); return B200_ERR_UNSUPPORTED;
    }
    ctx->launches++;
    return B200_OK;
}

bool supports_glue(const b200_op *op) {
    const b200_tensor &a = op->src[0], &b = op->src[1], &d = op->dst;
    switch (op->op) {
        case B200_OP_RMS_NORM: return rows_f32_ok(a) && rows_f32_ok(d);
        case B200_OP_RMS_NORM_MUL: return rows_f32_ok(a) && rows_f32_ok(d) && rows_f32_ok(b);
        case B200_OP_ADD: case B200_OP_SUB: case B200_OP_MUL: case B200_OP_DIV:
            return a.type == B200_TYPE_F32 && b.type == B200_TYPE_F32 && d.type == B200_TYPE_F32;
        case B200_OP_SILU: case B200_OP_GELU: case B200_OP_RELU: case B200_OP_TANH: case B200_OP_SIGMOID: case B200_OP_SCALE:
            return a.type == B200_TYPE_F32 && d.type == B200_TYPE_F32 && tensor_is_contiguous(a) && tensor_is_contiguous(d);
        case B200_OP_SWIGLU_FUSED:
            return a.type == B200_TYPE_F32 && b.type == B200_TYPE_F32 && tensor_is_contiguous(a) && tensor_is_contiguous(b) &&
                   tensor_is_contiguous(d) && same_shape(a, b);
        case B200_OP_ROPE: {
            const int mode = op->params[2];
            if (mode != 0 && mode != 2) return false;     // norm / neox only (mrope, vision: out of scope)
            if (a.type != d.type || (a.type != B200_TYPE_F32 && a.type != B200_TYPE_F16)) return false;
            return a.nb[0] == (uint64_t)b200_type_block_bytes(a.type) && d.nb[0] == a.nb[0] && a.ne[0] % 2 == 0;
        }
        case B200_OP_CPY: case B200_OP_CONT: {
            if (!cpy_pair_ok(a.type, d.type)) return false;
            if (tensor_nelements(a) != tensor_nelements(d)) return false;
            if (b200_type_is_quant(a.type) && a.type == d.type)
                return a.ne[0] % b200_type_block_elems(a.type) == 0 && d.ne[0] % b200_type_block_elems(a.type) == 0 &&
                       a.nb[0] == (uint64_t)b200_type_block_bytes(a.type) && d.nb[0] == a.nb[0] && a.data != d.data;
            if (d.type == B200_TYPE_Q8_0 || d.type == B200_TYPE_Q4_0)
                return a.nb[0] == 4 && a.ne[0] % 32 == 0 && d.ne[0] % 32 == 0 && !((uintptr_t)a.data & 15) && !(a.nb[1] & 15) &&
                       !(a.nb[2] & 15) && !(a.nb[3] & 15);
            if (b200_type_is_quant(a.type)) return true;
            return true;
        }
        case B200_OP_GET_ROWS:
            return b.type == B200_TYPE_I32 && d.type == B200_TYPE_F32 &&
                   (a.type == B200_TYPE_F32 || a.type == B200_TYPE_F16 || a.type == B200_TYPE_BF16 || b200_type_is_quant(a.type));
        case B200_OP_SOFT_MAX:
            if (!rows_f32_ok(a) || !rows_f32_ok(d)) return false;
            if (op->n_src > 1 && b.data) return (b.type == B200_TYPE_F16 || b.type == B200_TYPE_F32) && tensor_is_contiguous(b);
            return true;
        case B200_OP_ARGSORT: return rows_f32_ok(a) && d.type == B200_TYPE_I32 && a.ne[0] <= 1024 && tensor_is_contiguous(a);
        case B200_OP_SUM_ROWS: return rows_f32_ok(a) && d.type == B200_TYPE_F32;
        case B200_OP_ARGMAX: return rows_f32_ok(a) && d.type == B200_TYPE_I32 && d.nb[0] == 4 && a.ne[2] == 1 && a.ne[3] == 1 && a.ne[0] < (1ll << 31);
        default: return false;
    }
}

int op_glue(b200_ctx *ctx, const b200_op *op) {
    const b200_tensor &a = op->src[0], &b = op->src[1], &d = op->dst;
    switch (op->op) {
        case B200_OP_RMS_NORM:
        case B200_OP_RMS_NORM_MUL: {
            const int64_t rows = tensor_nrows(a);
            if (rows == 0) return B200_OK;
            if (op->op == B200_OP_RMS_NORM) b200_rms_norm_kernel<false><<<(unsigned)rows, 256, 0, ctx->stream>>>(a, a, d, f32_param(op, 0));
            else b200_rms_norm_kernel<true><<<(unsigned)rows, 256, 0, ctx->stream>>>(a, b, d, f32_param(op, 0));
            ctx->launches++;
            CUDA_TRY(cudaGetLastError());
            return B200_OK;
        }
        case B200_OP_ADD: return launch_bin<BIN_ADD>(ctx, op);
        case B200_OP_SUB: return launch_bin<BIN_SUB>(ctx, op);
        case B200_OP_MUL: return launch_bin<BIN_MUL>(ctx, op);
        case B200_OP_DIV: return launch_bin<BIN_DIV>(ctx, op);
        case B200_OP_SILU: return launch_unary<UN_SILU>(ctx, op, 0.0f);
        case B200_OP_GELU: return launch_unary<UN_GELU>(ctx, op, 0.0f);
        case B200_OP_RELU: return launch_unary<UN_RELU>(ctx, op, 0.0f);
        case B200_OP_TANH: return launch_unary<UN_TANH>(ctx, op, 0.0f);
        case B200_OP_SIGMOID: return launch_unary<UN_SIGMOID>(ctx, op, 0.0f);
        case B200_OP_SCALE: return launch_unary<UN_SCALE>(ctx, op, f32_param(op, 0));
        case B200_OP_SWIGLU_FUSED: return launch_unary<UN_SWIGLU>(ctx, op, 0.0f);
        case B200_OP_ROPE: {
            RopeParams rp;
            rp.n_dims = op->params[1]; rp.mode = op->params[2]; rp.n_ctx_orig = op->params[4];
            rp.freq_base = f32_param(op, 5); rp.freq_scale = f32_param(op, 6); rp.ext_factor = f32_param(op, 7);
            rp.attn_factor = f32_param(op, 8); rp.beta_fast = f32_param(op, 9); rp.beta_slow = f32_param(op, 10);
            rp.theta_scale = powf(rp.freq_base, -2.0f / rp.n_dims);
            float lo = floorf(yarn_corr_dim(rp.n_dims, rp.n_ctx_orig, rp.beta_fast, rp.freq_base));
            float hi = ceilf(yarn_corr_dim(rp.n_dims, rp.n_ctx_orig, rp.beta_slow, rp.freq_base));
            rp.corr0 = lo < 0 ? 0 : lo;
            rp.corr1 = hi > rp.n_dims - 1 ? (float)(rp.n_dims - 1) : hi;
            rp.exact = ctx->opt_cpu_exact;
            const int has_ff = op->n_src > 2 && op->src[2].data != nullptr;
            if (a.ne[2] == 0 || a.ne[1] == 0) return B200_OK;
            const dim3 grid((unsigned)a.ne[2], (unsigned)a.ne[1], (unsigned)a.ne[3]);
            const int threads = a.ne[0] / 2 >= 128 ? 128 : (a.ne[0] / 2 >= 64 ? 64 : 32);
            if (a.type == B200_TYPE_F32) b200_rope_kernel<float><<<grid, threads, 0, ctx->stream>>>(a, b, op->src[2], d, rp, has_ff);
            else b200_rope_kernel<__half><<<grid, threads, 0, ctx->stream>>>(a, b, op->src[2], d, rp, has_ff);
            ctx->launches++;
            CUDA_TRY(cudaGetLastError());
            return B200_OK;
        }
        case B200_OP_CPY: case B200_OP_CONT: return launch_cpy(ctx, a, d);
        case B200_OP_GET_ROWS: {
            const int64_t total = tensor_nelements(d);
            if (total == 0) return B200_OK;
            b200_get_rows_kernel<<<nblk(total, 256), 256, 0, ctx->stream>>>(a, b, d, total);
            ctx->launches++;
            CUDA_TRY(cudaGetLastError());
            return B200_OK;
        }
        case B200_OP_SOFT_MAX: {
            const int64_t rows = tensor_nrows(a);
            if (rows == 0) return B200_OK;
            const int has_mask = op->n_src > 1 && b.data != nullptr;
            if (has_mask && b.type == B200_TYPE_F32)
                b200_soft_max_kernel<float><<<(unsigned)rows, 256, 0, ctx->stream>>>(a, b, d, f32_param(op, 0), f32_param(op, 1), 1, ctx->opt_cpu_exact);
            else
                b200_soft_max_kernel<__half><<<(unsigned)rows, 256, 0, ctx->stream>>>(a, b, d, f32_param(op, 0), f32_param(op, 1), has_mask, ctx->opt_cpu_exact);
            ctx->launches++;
            CUDA_TRY(cudaGetLastError());
            return B200_OK;
        }
        case B200_OP_ARGSORT: {
            const int64_t rows = tensor_nrows(a);
            if (rows == 0) return B200_OK;
            int pad = 1;
            while (pad < a.ne[0]) pad <<= 1;
            b200_argsort_kernel<<<(unsigned)rows, pad, pad * sizeof(int), ctx->stream>>>(a, d, pad, op->params[0]);
            ctx->launches++;
            CUDA_TRY(cudaGetLastError());
            return B200_OK;
        }
        case B200_OP_ARGMAX: {
            const int64_t rows = a.ne[1];
            if (rows == 0) return B200_OK;
            b200_argmax_kernel<<<(unsigned)rows, 1024, 0, ctx->stream>>>(a, d);
            ctx->launches++;
            CUDA_TRY(cudaGetLastError());
            return B200_OK;
        }
        case B200_OP_SUM_ROWS: {
            const int64_t rows = tensor_nrows(a);
            if (rows == 0) return B200_OK;
            b200_sum_rows_kernel<<<(unsigned)rows, 256, 0, ctx->stream>>>(a, d);
            ctx->launches++;
            CUDA_TRY(cudaGetLastError());
            return B200_OK;
        }
        default:
            b200_set_error("glue: op %d", op->op);
            return B200_ERR_UNSUPPORTED;
    }
}
