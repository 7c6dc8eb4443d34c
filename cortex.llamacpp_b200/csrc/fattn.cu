// fattn.cu -- FLASH_ATTN_EXT over f16 / q8_0 / q4_0 KV caches (decode and batched), split-KV.
//
// Replaces ggml_cuda_flash_attn_ext (fattn.cu:244-319), flash_attn_vec_ext_f32 (fattn-vec-f32.cuh:4-282), the
// combine kernel (fattn-common.cuh:609-650) and the "dequantise the whole cache to f16 first" path of the
// reference's mma kernel (fattn-common.cuh:720-746).  Semantics follow the CPU oracle
// (ggml_compute_forward_flash_attn_ext_f16, ggml-cpu.c:12221-12434):
//   * f16 K      : Q rows are rounded to f16, K.Q products are exact, accumulated in f32
//   * q8_0/q4_0 K: Q rows are quantised to q8_0 exactly like quantize_row_q8_0 (RNE, d=amax/127 as f16); the
//                  per-32 integer dots are EXACT (integers carried in f16 through the tensor core, |sum| < 2^24)
//                  and scaled by d_k*d_q in f32 like ggml_vec_dot_q8_0_q8_0 / q4_0_q8_0
//   * online softmax in f32, -inf mask cells contribute nothing, ALiBi slope and logit softcap as the CPU
//   * V: f16 as is; q8_0/q4_0 kept as exact integers with their scales folded into P (p*d_v in f32); the softmax
//     weights are fed to the tensor core as an f16 hi+lo pair (22 significant bits), so P.V is f32-accurate like the
//     CPU's f32 path for quantised V (the CPU's f16 accumulator for f16 V is LESS accurate than this; see tests)
// Design: one CTA = one KV head x one tile of 16 query rows (GQA heads of the same KV head and/or several
// query columns share every K/V byte) x one KV split.  The 4 warps of a CTA take alternating 32-position KV
// tiles; K/V tiles are staged in shared memory (cp.async for f16, convert-on-load for quantised), fed to
// mma.sync.m16n8k16 via ldmatrix.  32-position tiles whose mask is -inf for every query of the CTA are
// skipped before any K/V byte is requested (unified multi-slot KV cache).  Splits are merged by a small
// combine kernel (log-sum-exp).  A tcgen05 variant for long prefill is future work (DESIGN.md).
#include "common.cuh"
#include "fattn_tc.h"

namespace {

enum { KV_F16 = 0, KV_Q8_0 = 1, KV_Q4_0 = 2 };
constexpr int BK = 32;          // kv positions per warp tile
constexpr int NWARP = 4;
constexpr float PV_SCALE = 256.0f, PV_UNSCALE = 1.0f / 256.0f;

struct FaParams {
    const char *q; uint64_t q_nb1, q_nb2, q_nb3;
    const char *k; uint64_t k_nb1, k_nb2, k_nb3;
    const char *v; uint64_t v_nb1, v_nb2, v_nb3;
    const char *mask; uint64_t m_nb1;
    float *dst;
    float *part;                 // [tile][split][16][D + 2]
    const int *map; int map_stride;   // live-tile map [n_coltiles][1 + n_kv / 32]: count, then the indices of the 32-position tiles with any unmasked cell
    int n_q, n_kv, H, Hkv, gq, HG, QC, n_headtiles, n_coltiles, n_splits, kv_per_split;
    float scale, softcap, max_bias, m0, m1;
    int n_head_log2;
    int use_pdl;
};

__device__ __forceinline__ void ldsm_x4(uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3, const void *p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3, const void *p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async16(void *s, const void *g) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(s)), "l"(g));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
    const __half2 h = __floats2half2_rn(a, b);
    return *(const uint32_t *)&h;
}

// stage one 32 x D tile of K or V into shared memory as f16 [32][D+8]; quantised types are converted on load.
// RAWINT: keep the integer quants (K path: scales go to `sc`), else dequantise d*q (V path).
template <int D, int T, bool RAWINT>
__device__ __forceinline__ void stage_tile(__half *s, float *sc, const char *g, uint64_t nb1, int kv0, int lane, const uint8_t *rawbuf, float sc_mul) {
    constexpr int LD = D + 8;
    if (T == KV_F16) {
        constexpr int CH = D / 8;                      // 16-byte chunks per row
        for (int c = lane; c < BK * CH; c += 32) {
            const int r = c / CH, cc = c % CH;
            cp_async16(s + r * LD + cc * 8, g + (uint64_t)(kv0 + r) * nb1 + cc * 16);
        }
    } else {
        // quantised rows (q8_0: 34*D/32, q4_0: 18*D/32 bytes, 8-byte aligned) were fetched into `raw` by fetch_raw() with coalesced
        // 8-byte cp.async; one lane converts one row.  The quants become exact f16 integers without a float conversion: 0x6400 | u is
        // the half 1024 + u, so (byte ^ 0x80) -> 1024 + 128 + q and one HSUB2 by 1152 (q8_0), or nibble -> 1024 + n and HSUB2 by
        // 1032 (q4_0: n - 8); 8 halves leave in one 16-byte store
        static_assert(RAWINT, "quantised tiles are staged as raw integers; their scales go to `sc`");
        constexpr int BB = T == KV_Q8_0 ? 34 : 18;
        constexpr int RB = BB * (D / 32);
        const uint2 *src = (const uint2 *)(rawbuf + lane * RB);
        uint32_t raw[RB / 4 + 1];
#pragma unroll
        for (int i = 0; i < RB / 8; i++) { const uint2 v = src[i]; raw[2 * i] = v.x; raw[2 * i + 1] = v.y; }
        raw[RB / 4] = 0;
        __half *row = s + lane * LD;
        auto word_at = [&](int byte_off) -> uint32_t {      // 32 bits at a 2-byte aligned offset of the row (constant after unrolling)
            return (byte_off & 2) ? __funnelshift_r(raw[byte_off >> 2], raw[(byte_off >> 2) + 1], 16) : raw[byte_off >> 2];
        };
        auto h2 = [](uint32_t bytes, uint32_t sel, uint32_t bias) -> uint32_t {
            const uint32_t v = __byte_perm(bytes, 0x64646464u, sel);
            const __half2 r = __hsub2(*(const __half2 *)&v, *(const __half2 *)&bias);
            return *(const uint32_t *)&r;
        };
#pragma unroll
        for (int b = 0; b < D / 32; b++) {
            const uint32_t hd = word_at(b * BB);
            sc[lane * (D / 32) + b] = __half2float(__ushort_as_half((unsigned short)(hd & 0xffffu))) * sc_mul;
            if (T == KV_Q8_0) {
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                    const uint32_t w0 = word_at(b * BB + 2 + j) ^ 0x80808080u, w1 = word_at(b * BB + 6 + j) ^ 0x80808080u;
                    *(uint4 *)(row + b * 32 + j) = make_uint4(h2(w0, 0x4140, 0x64806480u), h2(w0, 0x4342, 0x64806480u), h2(w1, 0x4140, 0x64806480u), h2(w1, 0x4342, 0x64806480u));
                }
            } else {
#pragma unroll
                for (int j = 0; j < 16; j += 8) {
                    const uint32_t w0 = word_at(b * BB + 2 + j), w1 = word_at(b * BB + 6 + j);
                    const uint32_t l0 = w0 & 0x0f0f0f0fu, l1 = w1 & 0x0f0f0f0fu, u0 = (w0 >> 4) & 0x0f0f0f0fu, u1 = (w1 >> 4) & 0x0f0f0f0fu;
                    *(uint4 *)(row + b * 32 + j)      = make_uint4(h2(l0, 0x4140, 0x64086408u), h2(l0, 0x4342, 0x64086408u), h2(l1, 0x4140, 0x64086408u), h2(l1, 0x4342, 0x64086408u));
                    *(uint4 *)(row + b * 32 + 16 + j) = make_uint4(h2(u0, 0x4140, 0x64086408u), h2(u0, 0x4342, 0x64086408u), h2(u1, 0x4140, 0x64086408u), h2(u1, 0x4342, 0x64086408u));
                }
            }
        }
    }
}

// quantised K/V: the 32 raw rows of a tile -> shared memory, consecutive lanes on consecutive 8-byte pieces of a row (a lane-per-row
// global read touches 32 different lines per instruction and serialises in the L1 tag stage: 47 us per bs32 layer)
template <int D, int T>
__device__ __forceinline__ void fetch_raw(uint8_t *rawbuf, const char *g, uint64_t nb1, int kv0, int lane) {
    constexpr int RB = (T == KV_Q8_0 ? 34 : 18) * (D / 32);
    constexpr int PC = RB / 8;                  // 8-byte pieces per row; BK * PC / 32 = PC pieces per lane
    int r = lane / PC, cc = lane % PC;
    const uint32_t sbase = smem_u32(rawbuf);
    const char *gb = g + (uint64_t)kv0 * nb1;
#pragma unroll
    for (int i = 0; i < PC; i++) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sbase + (uint32_t)(r * RB + cc * 8)), "l"(gb + (uint64_t)r * nb1 + cc * 8));
        cc += 32 % PC; r += 32 / PC;
        if (cc >= PC) { cc -= PC; r++; }
    }
}

// merge the per-warp results of a CTA (cm / cl / co in shared memory, rows r of the tile; fixed warp order), then write the result or,
// with several KV splits, the split partial for the combine kernel.  Shared by the 16-row kernel and the few-row kernel.
template <int D>
__device__ __forceinline__ void fa_merge_store(const FaParams &p, uint8_t *fsm, int ht, int hk, int c0, int split) {
    float *cm = (float *)fsm;             // [NWARP][16] max
    float *cl = cm + NWARP * 16;          // [NWARP][16] sum
    float *co = cl + NWARP * 16;          // [NWARP][16][D]
    __syncthreads();
    const int tile_id = blockIdx.y;
    for (int e = threadIdx.x; e < 16 * D; e += NWARP * 32) {
        const int r = e / D, d = e % D;
        {   // rows of the 16-row tile that hold no query (a bs1 decode step fills 4 of 16): nothing to merge or store
            const int hin_ = ht * p.HG + r % p.HG, col_ = c0 + r / p.HG;
            if (!((r / p.HG) < p.QC && col_ < p.n_q && hin_ < p.gq)) continue;
        }
        float M = -INFINITY;
#pragma unroll
        for (int w = 0; w < NWARP; w++) M = fmaxf(M, cm[w * 16 + r]);
        float val = 0.0f, L = 0.0f;
        if (M != -INFINITY) {
#pragma unroll
            for (int w = 0; w < NWARP; w++) {
                const float mw = cm[w * 16 + r];
                const float f = mw == -INFINITY ? 0.0f : expf(mw - M);
                val += co[(w * 16 + r) * D + d] * f;
                L += cl[w * 16 + r] * f;
            }
        }
        const int hin = ht * p.HG + r % p.HG, col = c0 + r / p.HG;
        const bool valid = (r / p.HG) < p.QC && col < p.n_q && hin < p.gq;
        if (p.n_splits == 1) {
            if (valid) p.dst[((uint64_t)col * p.H + hk * p.gq + hin) * D + d] = val / L;
        } else {
            float *pp = p.part + (((uint64_t)tile_id * p.n_splits + split) * 16 + r) * (D + 2);
            pp[d] = val;
            if (d == 0) { pp[D] = M; pp[D + 1] = L; }
        }
    }
}

template <int D, int KT, int VT>
__global__ void __launch_bounds__(NWARP * 32, 2) b200_fattn_kernel(const FaParams p) {
    constexpr int LD = D + 8;
    constexpr int NKS = D / 16;                  // k-steps of the QK product
    constexpr int NDT = D / 8;                   // n-tiles of the PV product
    constexpr int NB = D / 32;                   // 32-element blocks per row
    constexpr bool KQ = KT != KV_F16;
    extern __shared__ __align__(128) uint8_t fsm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (p.use_pdl) { pdl_trigger(); pdl_wait(); }
    // per-warp staging: K tile, V tile, K scales
    constexpr int RAWK = KQ ? BK * (KT == KV_Q8_0 ? 34 : 18) * NB : 0, RAWV = VT != KV_F16 ? BK * (VT == KV_Q8_0 ? 34 : 18) * NB : 0;
    constexpr int WARP_BYTES = 2 * BK * LD * 2 + 2 * BK * NB * 4 + RAWK + RAWV;
    __half *sK = (__half *)(fsm + warp * WARP_BYTES);
    __half *sV = sK + BK * LD;
    float *sKs = (float *)(sV + BK * LD);
    float *sVs = sKs + BK * NB;
    uint8_t *rawK = (uint8_t *)(sVs + BK * NB), *rawV = rawK + RAWK;
    constexpr bool VQ = VT != KV_F16;

    const int split = blockIdx.x;
    int tile = blockIdx.y;
    const int ct = tile % p.n_coltiles; tile /= p.n_coltiles;
    const int ht = tile % p.n_headtiles;
    const int hk = tile / p.n_headtiles;
    const int c0 = ct * p.QC;

    // rows owned by this lane in the mma layouts: r_lo = lane/4, r_hi = r_lo + 8
    int rcol[2], rhead[2]; bool rvalid[2];
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int r = (lane >> 2) + 8 * i;
        const int hin = ht * p.HG + r % p.HG;
        rcol[i] = c0 + r / p.HG;
        rhead[i] = hk * p.gq + hin;
        rvalid[i] = (r / p.HG) < p.QC && rcol[i] < p.n_q && hin < p.gq;
    }

    // ---- Q fragments (A operand), converted like the CPU converts Q for K's vec_dot_type -------------------
    uint32_t qa[NKS][4];
    float dq[2][NB];                      // q8_0 scales of my two rows (quantised K only)
    {
        float qv[2][NKS][4];
#pragma unroll
        for (int i = 0; i < 2; i++) {
            const float *qp = (const float *)(p.q + (uint64_t)rcol[i] * p.q_nb1 + (uint64_t)rhead[i] * p.q_nb2);
#pragma unroll
            for (int ks = 0; ks < NKS; ks++) {
                const int kb = ks * 16 + (lane & 3) * 2;
                if (rvalid[i]) {
                    const float2 a = *(const float2 *)(qp + kb), b = *(const float2 *)(qp + kb + 8);
                    qv[i][ks][0] = a.x; qv[i][ks][1] = a.y; qv[i][ks][2] = b.x; qv[i][ks][3] = b.y;
                } else {
                    qv[i][ks][0] = qv[i][ks][1] = qv[i][ks][2] = qv[i][ks][3] = 0.0f;
                }
            }
            if (KQ) {
#pragma unroll
                for (int b = 0; b < NB; b++) {
                    float amax = 0.0f;
#pragma unroll
                    for (int e = 0; e < 4; e++) amax = fmaxf(amax, fmaxf(fabsf(qv[i][2 * b][e]), fabsf(qv[i][2 * b + 1][e])));
                    amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 1));
                    amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 2));
                    const float d = __fdiv_rn(amax, 127.0f);
                    const float id = amax != 0.0f ? __fdiv_rn(127.0f, amax) : 0.0f;
                    dq[i][b] = __half2float(__float2half_rn(d));
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        qv[i][2 * b][e] = (float)__float2int_rn(__fmul_rn(qv[i][2 * b][e], id));
                        qv[i][2 * b + 1][e] = (float)__float2int_rn(__fmul_rn(qv[i][2 * b + 1][e], id));
                    }
                }
            }
        }
#pragma unroll
        for (int ks = 0; ks < NKS; ks++) {
            qa[ks][0] = pack_h2(qv[0][ks][0], qv[0][ks][1]);
            qa[ks][1] = pack_h2(qv[1][ks][0], qv[1][ks][1]);
            qa[ks][2] = pack_h2(qv[0][ks][2], qv[0][ks][3]);
            qa[ks][3] = pack_h2(qv[1][ks][2], qv[1][ks][3]);
        }
    }

    float slope[2] = {1.0f, 1.0f};
    if (p.max_bias > 0.0f) {
#pragma unroll
        for (int i = 0; i < 2; i++) {
            const int h = rhead[i];
            slope[i] = h < p.n_head_log2 ? powf(p.m0, (float)(h + 1)) : powf(p.m1, (float)(2 * (h - p.n_head_log2) + 1));
        }
    }

    float o[NDT][4];
#pragma unroll
    for (int t = 0; t < NDT; t++) o[t][0] = o[t][1] = o[t][2] = o[t][3] = 0.0f;
    float mrow[2] = {-INFINITY, -INFINITY}, lrow[2] = {0.0f, 0.0f};

    const char *kbase = p.k + (uint64_t)hk * p.k_nb2;
    const char *vbase = p.v + (uint64_t)hk * p.v_nb2;
    const int kv_begin = split * p.kv_per_split;
    const int kv_end = min(p.n_kv, kv_begin + p.kv_per_split);

    // with a live-tile map the splits share the LIVE tiles of this column tile evenly (a unified multi-slot cache leaves a batched
    // step ~3 % of the cache per column tile, all of it inside one or two uniform splits); without, a uniform split of [0, n_kv)
    const int *mp = p.map ? p.map + (size_t)ct * p.map_stride : nullptr;
    int it_begin = kv_begin / BK, it_end = kv_end / BK;
    if (mp) { const int cnt = mp[0]; it_begin = (int)((long long)split * cnt / p.n_splits); it_end = (int)((long long)(split + 1) * cnt / p.n_splits); }
    // quantised caches with a live-tile map: the raw rows of the NEXT tile are in flight (cp.async) while this one is multiplied
    constexpr bool PREFETCH = KQ && VQ;
    if (PREFETCH && mp && it_begin + warp < it_end) {
        const int kvf = mp[1 + it_begin + warp] * BK;
        fetch_raw<D, KT>(rawK, kbase, p.k_nb1, kvf, lane);
        fetch_raw<D, VT>(rawV, vbase, p.v_nb1, kvf, lane);
    }
    for (int it = it_begin + warp; it < it_end; it += NWARP) {
        const int kv0 = (mp ? mp[1 + it] : it) * BK;
        // ---- skip tiles that are fully masked for every query column of this CTA -------------------------
        if (p.mask && !mp) {
            bool any = false;
            for (int c = 0; c < p.QC; c++) {
                const int col = c0 + c;
                if (col < p.n_q) {
                    const __half mv = *(const __half *)(p.mask + (uint64_t)col * p.m_nb1 + (uint64_t)(kv0 + lane) * 2);
                    any |= !(__hisinf(mv) && __half2float(mv) < 0.0f);
                }
            }
            if (!__any_sync(0xffffffffu, any)) continue;
        }
        __syncwarp();
        if (!(PREFETCH && mp)) {
            if (KQ) fetch_raw<D, KT>(rawK, kbase, p.k_nb1, kv0, lane);
            if (VQ) fetch_raw<D, VT>(rawV, vbase, p.v_nb1, kv0, lane);
        }
        if (KQ || VQ) { cp_async_wait_all(); __syncwarp(); }
        stage_tile<D, KT, true>(sK, sKs, kbase, p.k_nb1, kv0, lane, rawK, 1.0f);
        stage_tile<D, VT, true>(sV, sVs, vbase, p.v_nb1, kv0, lane, rawV, PV_SCALE);      // exact power of two, see below
        if (KT == KV_F16 || VT == KV_F16) cp_async_wait_all();
        __syncwarp();
        if (PREFETCH && mp && it + NWARP < it_end) {
            const int kvn = mp[1 + it + NWARP] * BK;
            fetch_raw<D, KT>(rawK, kbase, p.k_nb1, kvn, lane);
            fetch_raw<D, VT>(rawV, vbase, p.v_nb1, kvn, lane);
        }

        // ---- S = Q K^T  (16 x 32) ---------------------------------------------------------------------
        float s[4][4];
#pragma unroll
        for (int nt = 0; nt < 4; nt++) {
            s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.0f;
#pragma unroll
            for (int ks = 0; ks < NKS; ks += 2) {
                uint32_t b0, b1, b2, b3;
                ldsm_x4(b0, b1, b2, b3, sK + (nt * 8 + (lane & 7)) * LD + ks * 16 + (lane >> 3) * 8);
                if (KQ) {
                    float t[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                    mma16816(t, qa[ks], b0, b1);
                    mma16816(t, qa[ks + 1], b2, b3);
                    const int b = ks >> 1;
                    const int kvc = nt * 8 + (lane & 3) * 2;
                    const float dk0 = sKs[kvc * NB + b], dk1 = sKs[(kvc + 1) * NB + b];
                    s[nt][0] += t[0] * (dk0 * dq[0][b]); s[nt][1] += t[1] * (dk1 * dq[0][b]);
                    s[nt][2] += t[2] * (dk0 * dq[1][b]); s[nt][3] += t[3] * (dk1 * dq[1][b]);
                } else {
                    mma16816(s[nt], qa[ks], b0, b1);
                    mma16816(s[nt], qa[ks + 1], b2, b3);
                }
            }
        }
        // ---- scale, softcap, mask, online softmax ---------------------------------------------------------
        float tmax[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int nt = 0; nt < 4; nt++) {
            const int kvc = kv0 + nt * 8 + (lane & 3) * 2;
#pragma unroll
            for (int i = 0; i < 2; i++) {
                float v0 = s[nt][2 * i] * p.scale, v1 = s[nt][2 * i + 1] * p.scale;
                if (p.softcap != 0.0f) { v0 = p.softcap * tanhf(v0); v1 = p.softcap * tanhf(v1); }
                if (p.mask && rvalid[i]) {
                    const __half2 mv = *(const __half2 *)(p.mask + (uint64_t)rcol[i] * p.m_nb1 + (uint64_t)kvc * 2);
                    v0 += slope[i] * __low2float(mv);
                    v1 += slope[i] * __high2float(mv);
                }
                s[nt][2 * i] = v0; s[nt][2 * i + 1] = v1;
                tmax[i] = fmaxf(tmax[i], fmaxf(v0, v1));
            }
        }
        float corr[2], muse[2];
#pragma unroll
        for (int i = 0; i < 2; i++) {
            tmax[i] = fmaxf(tmax[i], __shfl_xor_sync(0xffffffffu, tmax[i], 1));
            tmax[i] = fmaxf(tmax[i], __shfl_xor_sync(0xffffffffu, tmax[i], 2));
            const float mnew = fmaxf(mrow[i], tmax[i]);
            muse[i] = mnew == -INFINITY ? 0.0f : mnew;
            corr[i] = mrow[i] == -INFINITY ? 0.0f : expf(mrow[i] - muse[i]);
            mrow[i] = mnew;
            lrow[i] *= corr[i];
        }
#pragma unroll
        for (int nt = 0; nt < 4; nt++)
#pragma unroll
            for (int i = 0; i < 2; i++) {
                const float p0 = expf(s[nt][2 * i] - muse[i]), p1 = expf(s[nt][2 * i + 1] - muse[i]);
                s[nt][2 * i] = p0; s[nt][2 * i + 1] = p1;
                lrow[i] += p0 + p1;
            }
        if (__any_sync(0xffffffffu, corr[0] != 1.0f || corr[1] != 1.0f)) {       // multiplying by 1 is the identity: skipping it changes nothing
#pragma unroll
            for (int t = 0; t < NDT; t++) { o[t][0] *= corr[0]; o[t][1] *= corr[0]; o[t][2] *= corr[1]; o[t][3] *= corr[1]; }
        }
        // ---- O += P V : P as f16 hi+lo (22 bits); quantised V stays integer, its scale is folded into P per dim block ----
#pragma unroll
        for (int kk = 0; kk < 2; kk++) {
            const float pv[8] = {s[2 * kk][0], s[2 * kk][1], s[2 * kk][2], s[2 * kk][3], s[2 * kk + 1][0], s[2 * kk + 1][1], s[2 * kk + 1][2], s[2 * kk + 1][3]};
            const int kvA = kk * 16 + (lane & 3) * 2;       // kv index (within the tile) of pv[0], pv[2]; +1 for pv[1], pv[3]; +8 for pv[4..7]
#pragma unroll
            for (int b = 0; b < (VQ ? NB : 1); b++) {
                float w[8];
                if (VQ) {
                    const float dA0 = sVs[kvA * NB + b], dA1 = sVs[(kvA + 1) * NB + b], dB0 = sVs[(kvA + 8) * NB + b], dB1 = sVs[(kvA + 9) * NB + b];
                    w[0] = pv[0] * dA0; w[1] = pv[1] * dA1; w[2] = pv[2] * dA0; w[3] = pv[3] * dA1;
                    w[4] = pv[4] * dB0; w[5] = pv[5] * dB1; w[6] = pv[6] * dB0; w[7] = pv[7] * dB1;
                } else {
#pragma unroll
                    for (int e = 0; e < 8; e++) w[e] = pv[e];
                }
                // exact power-of-two pre-scale: keeps the f16 hi/lo pair out of the f16 subnormal range for small
                // softmax weights (w ~ 1e-4 would otherwise lose its low half); undone when the accumulators are stored
                if (!VQ) {
#pragma unroll
                    for (int e = 0; e < 8; e++) w[e] *= PV_SCALE;         // (quantised V: folded into the staged block scales)
                }
                uint32_t ph[4], pl[4];
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const __half2 hi = __floats2half2_rn(w[2 * e], w[2 * e + 1]);
                    const float2 hf = __half22float2(hi);
                    ph[e] = *(const uint32_t *)&hi;
                    pl[e] = pack_h2(w[2 * e] - hf.x, w[2 * e + 1] - hf.y);
                }
                constexpr int DT0 = 0;
                const int dt_begin = VQ ? b * 4 : DT0, dt_end = VQ ? b * 4 + 4 : NDT;
#pragma unroll
                for (int dt = dt_begin; dt < dt_end; dt += 2) {
                    uint32_t b0, b1, b2, b3;
                    ldsm_x4_t(b0, b1, b2, b3, sV + (kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LD + dt * 8 + (lane >> 4) * 8);
                    mma16816(o[dt], ph, b0, b1);
                    mma16816(o[dt], pl, b0, b1);
                    mma16816(o[dt + 1], ph, b2, b3);
                    mma16816(o[dt + 1], pl, b2, b3);
                }
            }
        }
    }

    // ---- merge the 4 warps of the CTA (fixed warp order), then write the result or the split partial ----------
#pragma unroll
    for (int i = 0; i < 2; i++) {
        lrow[i] += __shfl_xor_sync(0xffffffffu, lrow[i], 1);
        lrow[i] += __shfl_xor_sync(0xffffffffu, lrow[i], 2);
    }
    __syncthreads();                      // staging buffers are dead from here on
    float *cm = (float *)fsm;             // [NWARP][16] max
    float *cl = cm + NWARP * 16;          // [NWARP][16] sum
    float *co = cl + NWARP * 16;          // [NWARP][16][D]
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int r = (lane >> 2) + 8 * i;
        if ((lane & 3) == 0) { cm[warp * 16 + r] = mrow[i]; cl[warp * 16 + r] = lrow[i]; }
#pragma unroll
        for (int t = 0; t < NDT; t++) {
            const int d = t * 8 + (lane & 3) * 2;
            *(float2 *)(co + (warp * 16 + r) * D + d) = make_float2(o[t][2 * i] * PV_UNSCALE, o[t][2 * i + 1] * PV_UNSCALE);
        }
    }
    fa_merge_store<D>(p, fsm, ht, hk, c0, split);
}

// ---------------------------------------------------------------------------------------------------------------------
// Few-row attention (decode, and continuous-batching steps where every KV tile is live for ONE query column): tile = one KV head x
// one query column, rows = the gq <= 8 heads of the GQA group.  The 16-row kernel above would run 16-row MMA tiles with 4 live
// rows; here the products are transposed so that the KV cells are the MMA M dimension and the (<= 8) heads the N = 8 dimension:
//     S^T [32 cells x 8]  = K [32 x D] . Q^T [D x 8]            2 x D/16 mma.m16n8k16  (16 for D = 128, instead of 32)
//     O^T [D x 8]        += V^T [D x 32] . P^T [32 x 8]         D/16 x 2             (16, instead of 64)
// P^T leaves the first product in the accumulator layout (cell = lane/4, head = 2*(lane%4)) and enters the second as a B operand
// (cell = 2*(lane%4), head = lane/4): one 512-byte trip through shared memory per tile.  Arithmetic as in the 16-row kernel: exact
// integer K.Q per 32-block for quantised K, f32 online softmax, P as an f16 hi+lo pair, quantised V kept integer with its block
// scales folded into P.  Same splits, live-tile map, partial layout and combine kernel (rows r < gq of a 16-row slot).
// ---------------------------------------------------------------------------------------------------------------------
template <int D, int KT, int VT>
__global__ void __launch_bounds__(NWARP * 32, 2) b200_fattn_rows8_kernel(const FaParams p) {
    constexpr int LD = D + 8;
    constexpr int NKS = D / 16, NB = D / 32, NMD = D / 16;
    constexpr bool KQ = KT != KV_F16, VQ = VT != KV_F16;
    constexpr int PLD = 40;                      // halves per head row of the P^T staging buffer
    extern __shared__ __align__(128) uint8_t fsm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (p.use_pdl) { pdl_trigger(); pdl_wait(); }
    constexpr int RAWK = KQ ? BK * (KT == KV_Q8_0 ? 34 : 18) * NB : 0, RAWV = VQ ? BK * (VT == KV_Q8_0 ? 34 : 18) * NB : 0;
    constexpr int WARP_BYTES = 2 * BK * LD * 2 + 2 * BK * NB * 4 + RAWK + RAWV + 2 * 8 * PLD * 2;
    __half *sK = (__half *)(fsm + warp * WARP_BYTES);
    __half *sV = sK + BK * LD;
    float *sKs = (float *)(sV + BK * LD);
    float *sVs = sKs + BK * NB;
    uint8_t *rawK = (uint8_t *)(sVs + BK * NB), *rawV = rawK + RAWK;
    __half *sPh = (__half *)(rawV + RAWV), *sPl = sPh + 8 * PLD;

    const int split = blockIdx.x;
    const int col = blockIdx.y % p.n_q, hk = blockIdx.y / p.n_q;       // tile = (kv head, query column); c0 = col, QC = 1, HG = gq
    const int n_b = lane >> 2, q4 = lane & 3;                           // B-operand layout: head n_b, k pair q4
    const int R = lane >> 2, n0 = 2 * (lane & 3);                       // accumulator layout: cell / dim row R (+8), heads n0, n0 + 1

    // ---- Q^T fragments (B operand), converted like the CPU converts Q for K's vec_dot_type ---------------------------------
    uint32_t qb[NKS][2];
    float dqc[2][NB];                          // q8_0 scales of heads n0, n0 + 1 (quantised K only)
    {
        float qv[NKS][4];
        const bool hv = n_b < p.gq;
        const float *qp = (const float *)(p.q + (uint64_t)col * p.q_nb1 + (uint64_t)(hk * p.gq + (hv ? n_b : 0)) * p.q_nb2);
#pragma unroll
        for (int ks = 0; ks < NKS; ks++) {
            const int kb = ks * 16 + q4 * 2;
            if (hv) { const float2 a = *(const float2 *)(qp + kb), b = *(const float2 *)(qp + kb + 8); qv[ks][0] = a.x; qv[ks][1] = a.y; qv[ks][2] = b.x; qv[ks][3] = b.y; }
            else qv[ks][0] = qv[ks][1] = qv[ks][2] = qv[ks][3] = 0.0f;
        }
        float dq[NB];
        if (KQ) {
#pragma unroll
            for (int b = 0; b < NB; b++) {
                float amax = 0.0f;
#pragma unroll
                for (int e = 0; e < 4; e++) amax = fmaxf(amax, fmaxf(fabsf(qv[2 * b][e]), fabsf(qv[2 * b + 1][e])));
                amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 1));
                amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 2));
                const float d = __fdiv_rn(amax, 127.0f);
                const float id = amax != 0.0f ? __fdiv_rn(127.0f, amax) : 0.0f;
                dq[b] = __half2float(__float2half_rn(d));
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    qv[2 * b][e] = (float)__float2int_rn(__fmul_rn(qv[2 * b][e], id));
                    qv[2 * b + 1][e] = (float)__float2int_rn(__fmul_rn(qv[2 * b + 1][e], id));
                }
            }
#pragma unroll
            for (int b = 0; b < NB; b++) { dqc[0][b] = __shfl_sync(0xffffffffu, dq[b], 4 * n0); dqc[1][b] = __shfl_sync(0xffffffffu, dq[b], 4 * (n0 + 1)); }
        }
#pragma unroll
        for (int ks = 0; ks < NKS; ks++) { qb[ks][0] = pack_h2(qv[ks][0], qv[ks][1]); qb[ks][1] = pack_h2(qv[ks][2], qv[ks][3]); }
    }
    float slope[2] = {1.0f, 1.0f};
    if (p.max_bias > 0.0f) {
#pragma unroll
        for (int i = 0; i < 2; i++) {
            const int h = hk * p.gq + n0 + i;
            slope[i] = h < p.n_head_log2 ? powf(p.m0, (float)(h + 1)) : powf(p.m1, (float)(2 * (h - p.n_head_log2) + 1));
        }
    }
    float o[NMD][4];
#pragma unroll
    for (int t = 0; t < NMD; t++) o[t][0] = o[t][1] = o[t][2] = o[t][3] = 0.0f;
    float mrow[2] = {-INFINITY, -INFINITY}, lrow[2] = {0.0f, 0.0f};

    const char *kbase = p.k + (uint64_t)hk * p.k_nb2;
    const char *vbase = p.v + (uint64_t)hk * p.v_nb2;
    const char *mrowp = p.mask ? p.mask + (uint64_t)col * p.m_nb1 : nullptr;
    const int kv_begin = split * p.kv_per_split, kv_end = min(p.n_kv, kv_begin + p.kv_per_split);
    const int *mp = p.map ? p.map + (size_t)col * p.map_stride : nullptr;
    int it_begin = kv_begin / BK, it_end = kv_end / BK;
    if (mp) { const int cnt = mp[0]; it_begin = (int)((long long)split * cnt / p.n_splits); it_end = (int)((long long)(split + 1) * cnt / p.n_splits); }
    constexpr bool PREFETCH = KQ && VQ;
    if (PREFETCH && mp && it_begin + warp < it_end) {
        const int kvf = mp[1 + it_begin + warp] * BK;
        fetch_raw<D, KT>(rawK, kbase, p.k_nb1, kvf, lane);
        fetch_raw<D, VT>(rawV, vbase, p.v_nb1, kvf, lane);
    }
    for (int it = it_begin + warp; it < it_end; it += NWARP) {
        const int kv0 = (mp ? mp[1 + it] : it) * BK;
        // no live-tile map (a decode step): the tile's cache rows are requested BEFORE the mask says whether the tile is live -- the mask
        // words and the rows then travel together (one L2 round trip instead of two on the token's critical path; a dead tile costs a
        // few KB of L2 traffic, and its copies are drained before the buffers are reused)
        __syncwarp();
        if (!(PREFETCH && mp)) {
            if (KQ) fetch_raw<D, KT>(rawK, kbase, p.k_nb1, kv0, lane);
            if (VQ) fetch_raw<D, VT>(rawV, vbase, p.v_nb1, kv0, lane);
        }
        if (KT == KV_F16) stage_tile<D, KT, true>(sK, sKs, kbase, p.k_nb1, kv0, lane, rawK, 1.0f);
        if (VT == KV_F16) stage_tile<D, VT, true>(sV, sVs, vbase, p.v_nb1, kv0, lane, rawV, PV_SCALE);
        if (mrowp && !mp) {                       // skip a tile that is fully masked for this column
            const __half mv = *(const __half *)(mrowp + (uint64_t)(kv0 + lane) * 2);
            if (!__any_sync(0xffffffffu, !(__hisinf(mv) && __half2float(mv) < 0.0f))) { cp_async_wait_all(); continue; }
        }
        if (KQ || VQ) { cp_async_wait_all(); __syncwarp(); }
        if (KT != KV_F16) stage_tile<D, KT, true>(sK, sKs, kbase, p.k_nb1, kv0, lane, rawK, 1.0f);
        if (VT != KV_F16) stage_tile<D, VT, true>(sV, sVs, vbase, p.v_nb1, kv0, lane, rawV, PV_SCALE);
        if (KT == KV_F16 || VT == KV_F16) cp_async_wait_all();
        __syncwarp();
        if (PREFETCH && mp && it + NWARP < it_end) {
            const int kvn = mp[1 + it + NWARP] * BK;
            fetch_raw<D, KT>(rawK, kbase, p.k_nb1, kvn, lane);
            fetch_raw<D, VT>(rawV, vbase, p.v_nb1, kvn, lane);
        }
        // ---- S^T = K Q^T: s[mt] = {cell R: heads n0, n0+1; cell R+8: heads n0, n0+1} of cells mt*16.. -------------------------
        float s[2][4];
#pragma unroll
        for (int mt = 0; mt < 2; mt++) {
            s[mt][0] = s[mt][1] = s[mt][2] = s[mt][3] = 0.0f;
#pragma unroll
            for (int b = 0; b < NB; b++) {
                float t[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
                for (int ks = 2 * b; ks < 2 * b + 2; ks++) {
                    uint32_t a[4];
                    ldsm_x4(a[0], a[1], a[2], a[3], sK + (mt * 16 + (lane & 15)) * LD + ks * 16 + (lane >> 4) * 8);
                    if (KQ) mma16816(t, a, qb[ks][0], qb[ks][1]); else mma16816(s[mt], a, qb[ks][0], qb[ks][1]);
                }
                if (KQ) {
                    const float dk0 = sKs[(mt * 16 + R) * NB + b], dk1 = sKs[(mt * 16 + R + 8) * NB + b];
                    s[mt][0] += t[0] * (dk0 * dqc[0][b]); s[mt][1] += t[1] * (dk0 * dqc[1][b]);
                    s[mt][2] += t[2] * (dk1 * dqc[0][b]); s[mt][3] += t[3] * (dk1 * dqc[1][b]);
                }
            }
        }
        // ---- scale, softcap, mask (one query column: the mask depends on the cell only), online softmax per head ------------------
        float tmax[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const float mv = mrowp ? __half2float(*(const __half *)(mrowp + (uint64_t)(kv0 + mt * 16 + R + 8 * h) * 2)) : 0.0f;
#pragma unroll
                for (int i = 0; i < 2; i++) {
                    float v = s[mt][2 * h + i] * p.scale;
                    if (p.softcap != 0.0f) v = p.softcap * tanhf(v);
                    if (mrowp) v += slope[i] * mv;
                    s[mt][2 * h + i] = v;
                    tmax[i] = fmaxf(tmax[i], v);
                }
            }
        float corr[2], muse[2];
#pragma unroll
        for (int i = 0; i < 2; i++) {
            tmax[i] = fmaxf(tmax[i], __shfl_xor_sync(0xffffffffu, tmax[i], 4));
            tmax[i] = fmaxf(tmax[i], __shfl_xor_sync(0xffffffffu, tmax[i], 8));
            tmax[i] = fmaxf(tmax[i], __shfl_xor_sync(0xffffffffu, tmax[i], 16));
            const float mnew = fmaxf(mrow[i], tmax[i]);
            muse[i] = mnew == -INFINITY ? 0.0f : mnew;
            corr[i] = mrow[i] == -INFINITY ? 0.0f : expf(mrow[i] - muse[i]);
            mrow[i] = mnew;
            lrow[i] *= corr[i];
        }
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
            for (int e = 0; e < 4; e++) { const float pe = expf(s[mt][e] - muse[e & 1]); s[mt][e] = pe; lrow[e & 1] += pe; }
        if (__any_sync(0xffffffffu, corr[0] != 1.0f || corr[1] != 1.0f)) {
#pragma unroll
            for (int t = 0; t < NMD; t++) { o[t][0] *= corr[0]; o[t][1] *= corr[1]; o[t][2] *= corr[0]; o[t][3] *= corr[1]; }
        }
        // ---- O^T += V^T P^T: P^T through shared memory into the B layout, f16 hi + lo; quantised V: block scale folded into P ----
#pragma unroll
        for (int b = 0; b < (VQ ? NB : 1); b++) {
            __syncwarp();
#pragma unroll
            for (int mt = 0; mt < 2; mt++)
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int cell = mt * 16 + R + 8 * h;
                    const float dv = VQ ? sVs[cell * NB + b] : PV_SCALE;       // (quantised V: PV_SCALE is folded into the staged scales)
#pragma unroll
                    for (int i = 0; i < 2; i++) {
                        const float w = s[mt][2 * h + i] * dv;
                        const __half hi = __float2half_rn(w);
                        sPh[(n0 + i) * PLD + cell] = hi;
                        sPl[(n0 + i) * PLD + cell] = __float2half_rn(w - __half2float(hi));
                    }
                }
            __syncwarp();
            uint32_t bh[2][2], bl[2][2];
#pragma unroll
            for (int kk = 0; kk < 2; kk++) {
                bh[kk][0] = *(const uint32_t *)(sPh + n_b * PLD + kk * 16 + q4 * 2); bh[kk][1] = *(const uint32_t *)(sPh + n_b * PLD + kk * 16 + 8 + q4 * 2);
                bl[kk][0] = *(const uint32_t *)(sPl + n_b * PLD + kk * 16 + q4 * 2); bl[kk][1] = *(const uint32_t *)(sPl + n_b * PLD + kk * 16 + 8 + q4 * 2);
            }
            const int md0 = VQ ? 2 * b : 0, md1 = VQ ? 2 * b + 2 : NMD;
#pragma unroll
            for (int md = md0; md < md1; md++)
#pragma unroll
                for (int kk = 0; kk < 2; kk++) {
                    uint32_t a[4];
                    ldsm_x4_t(a[0], a[1], a[2], a[3], sV + (kk * 16 + (lane & 7) + ((lane >> 4) & 1) * 8) * LD + md * 16 + ((lane >> 3) & 1) * 8);
                    mma16816(o[md], a, bh[kk][0], bh[kk][1]);
                    mma16816(o[md], a, bl[kk][0], bl[kk][1]);
                }
        }
    }
    // ---- hand the per-warp results to the common merge: rows r = head n of the 16-row slot ------------------------------------------
#pragma unroll
    for (int i = 0; i < 2; i++) {
        lrow[i] += __shfl_xor_sync(0xffffffffu, lrow[i], 4);
        lrow[i] += __shfl_xor_sync(0xffffffffu, lrow[i], 8);
        lrow[i] += __shfl_xor_sync(0xffffffffu, lrow[i], 16);
    }
    __syncthreads();                      // staging buffers are dead from here on
    float *cm = (float *)fsm, *cl = cm + NWARP * 16, *co = cl + NWARP * 16;
    if (lane < 4) {
#pragma unroll
        for (int i = 0; i < 2; i++) { cm[warp * 16 + n0 + i] = mrow[i]; cl[warp * 16 + n0 + i] = lrow[i]; }
    }
#pragma unroll
    for (int t = 0; t < NMD; t++)
#pragma unroll
        for (int e = 0; e < 4; e++) co[(warp * 16 + n0 + (e & 1)) * D + t * 16 + R + 8 * (e >> 1)] = o[t][e] * PV_UNSCALE;
    fa_merge_store<D>(p, fsm, 0, hk, col, split);
}

// ---------------------------------------------------------------------------------------------------------------------
// Live-tile map of the mask: for every column tile (QC query columns) the ascending list of 32-position KV tiles in which at least
// one cell is not -inf.  One CTA per column tile; built once per graph (the mask is shared by all layers).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int MAP_MAX_BATCH = 32;       // 4 warps x 32 batches x 32 tiles = 4096 tiles = 131072 KV positions
__global__ void __launch_bounds__(128) b200_fattn_maskmap_kernel(const char *mask, uint64_t m_nb1, int n_q, int n_kv, int QC, int *map, int map_stride, int use_pdl) {
    __shared__ uint32_t bal[4][MAP_MAX_BATCH];
    __shared__ int wcnt[4];
    if (use_pdl) { pdl_trigger(); pdl_wait(); }
    const int ct = blockIdx.x, c0 = ct * QC, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ntile = n_kv / BK;
    const int nbatch = (ntile + 127) / 128;             // batches of 32 tiles per warp; warp w owns tiles [w * nbatch * 32, (w + 1) * nbatch * 32)
    int cnt = 0;
    for (int b = 0; b < nbatch; b++) {
        const int t = (warp * nbatch + b) * 32 + lane;
        bool live = false;
        if (t < ntile)
            for (int c = 0; c < QC && c0 + c < n_q; c++) {
                const uint4 *mp = (const uint4 *)(mask + (uint64_t)(c0 + c) * m_nb1 + (uint64_t)t * (BK * 2));
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const uint4 v = mp[i];
                    live |= v.x != 0xFC00FC00u || v.y != 0xFC00FC00u || v.z != 0xFC00FC00u || v.w != 0xFC00FC00u;
                }
            }
        const uint32_t m = __ballot_sync(0xffffffffu, live);
        if (lane == 0) bal[warp][b] = m;
        cnt += __popc(m);
    }
    if (lane == 0) wcnt[warp] = cnt;
    __syncthreads();
    int off = 0;
    for (int w = 0; w < warp; w++) off += wcnt[w];
    int *out = map + (size_t)ct * map_stride;
    if (threadIdx.x == 0) out[0] = wcnt[0] + wcnt[1] + wcnt[2] + wcnt[3];
    for (int b = 0; b < nbatch; b++) {
        const uint32_t m = bal[warp][b];
        if (m & (1u << lane)) out[1 + off + __popc(m & ((1u << lane) - 1))] = (warp * nbatch + b) * 32 + lane;
        off += __popc(m);
    }
}

// merge of the KV splits: one WARP per (tile, query row); lanes first reduce the per-split (max, sum) pairs, then each lane
// owns D/32 output dims and walks the splits with independent loads (log-sum-exp merge, fixed split order => deterministic)
template <int D>
__global__ void __launch_bounds__(128) b200_fattn_combine_kernel(const FaParams p, int n_tiles) {
    if (p.use_pdl) { pdl_trigger(); pdl_wait(); }
    const int lane = threadIdx.x & 31;
    const int wid = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int tile_id = wid >> 4, r = wid & 15;
    if (tile_id >= n_tiles) return;
    int tile = tile_id;
    const int ct = tile % p.n_coltiles; tile /= p.n_coltiles;
    const int ht = tile % p.n_headtiles;
    const int hk = tile / p.n_headtiles;
    const int hin = ht * p.HG + r % p.HG, col = ct * p.QC + r / p.HG;
    if (!((r / p.HG) < p.QC && col < p.n_q && hin < p.gq)) return;
    const float *base = p.part + ((uint64_t)tile_id * p.n_splits * 16 + r) * (D + 2);
    const uint64_t sstride = (uint64_t)16 * (D + 2);
    constexpr int PER = D / 32;
    float acc[PER];
#pragma unroll
    for (int j = 0; j < PER; j++) acc[j] = 0.0f;
    float M = -INFINITY, L = 0.0f;
    if (p.n_splits <= 32) {
        // Same arithmetic in the same order as the general path below, but every load of a group of 8 splits is in flight before anything
        // is consumed: the merge costs ~2 L2 round trips instead of n_splits + 2 (a decode step runs this kernel once per layer, on the
        // token's critical path).  Lane s holds (m_s, l_s); the per-split factors come from shuffles instead of reloads.
        const float ms_l = lane < p.n_splits ? base[lane * sstride + D] : -INFINITY;
        const float ls_l = lane < p.n_splits ? base[lane * sstride + D + 1] : 0.0f;
        float v[8][PER];
        auto fetch = [&](int s0) {
#pragma unroll
            for (int u = 0; u < 8; u++)
                if (s0 + u < p.n_splits) {
#pragma unroll
                    for (int j = 0; j < PER; j++) v[u][j] = base[(s0 + u) * sstride + lane + 32 * j];
                }
        };
        fetch(0);
        M = warp_reduce_max(ms_l);
        L = warp_reduce_sum(ms_l == -INFINITY ? 0.0f : ls_l * expf(ms_l - M));
        for (int s0 = 0; s0 < p.n_splits; s0 += 8) {
            if (s0) fetch(s0);
#pragma unroll
            for (int u = 0; u < 8; u++)
                if (s0 + u < p.n_splits) {
                    const float ms = __shfl_sync(0xffffffffu, ms_l, s0 + u);
                    const float f = ms == -INFINITY ? 0.0f : expf(ms - M);
#pragma unroll
                    for (int j = 0; j < PER; j++) acc[j] += v[u][j] * f;
                }
        }
    } else {
        for (int s = lane; s < p.n_splits; s += 32) M = fmaxf(M, base[s * sstride + D]);
        M = warp_reduce_max(M);
        for (int s = lane; s < p.n_splits; s += 32) {
            const float ms = base[s * sstride + D];
            L += ms == -INFINITY ? 0.0f : base[s * sstride + D + 1] * expf(ms - M);
        }
        // fixed-order sum over lanes (xor tree is order-independent of scheduling)
        L = warp_reduce_sum(L);
        for (int s = 0; s < p.n_splits; s++) {
            const float *pp = base + s * sstride;
            const float ms = pp[D];
            const float f = ms == -INFINITY ? 0.0f : expf(ms - M);
#pragma unroll
            for (int j = 0; j < PER; j++) acc[j] += pp[lane + 32 * j] * f;
        }
    }
    float *o = p.dst + ((uint64_t)col * p.H + hk * p.gq + hin) * D;
#pragma unroll
    for (int j = 0; j < PER; j++) o[lane + 32 * j] = acc[j] / L;
}

// ---------------------------------------------------------------------------------------------------------------------
// "cpu-exact" mode for an f16 cache (option fa_exact / GGML_B200_FA_EXACT=1).  The reference CPU path accumulates f16 V rows
// in an FP16 accumulator, cell by cell, rounding after every step (VKQ16: ggml_vec_scale_f16 / ggml_vec_mad_f16,
// ggml-cpu.c:12376-12390) -- about 1e-2 of relative noise at a few hundred cells, which no f32 kernel can agree with.  This
// kernel restates that arithmetic: one warp per (query column, head), cells in order, masked cells skipped, K.Q with the
// accumulator layout of ggml_vec_dot_f16 on the AVX2 build (4 x 8 FMA lanes over 32-element steps, then the
// GGML_F32x8_REDUCE tree, ggml-cpu.c:671-689, 1565-1605), the running maximum / rescale logic of :12359-12395, and an
// accumulator that is rounded to fp16 after the rescale and after every fused multiply-add.  Only libm-vs-CUDA expf ulps
// remain (and those are removed too: exp_rn below).  It is a serial chain over n_kv, so it is the parity mode, not the fast mode (the default kernel above
// accumulates in f32 and is closer to exact attention: tests/test_gpu_fattn.py bounds both against f64).
// softmax weights through glibc's expf restated (common.cuh): the CPU backend's weights bit for bit.  One ulp of difference in
// a weight flips fp16 roundings of the accumulator (5e-4 each), and those flip q8 activation roundings in the next matmul.
__device__ __forceinline__ float exp_rn(float x) { return glibc_expf(x); }

template <int D, int KT>
__global__ void __launch_bounds__(128) b200_fattn_f16acc_kernel(const FaParams p) {
    constexpr int PER = D / 32;
    constexpr int NBQ = D / 32;
    constexpr bool QUANT = KT != KV_F16;
    constexpr int BB = KT == KV_Q8_0 ? 34 : 18;           // bytes per 32-element block of a quantised cache row
    __shared__ float sq[4][D];                            // f16-rounded Q (f16 K) ...
    __shared__ __align__(16) int8_t sqq[4][D];            // ... or Q quantised to q8_0 (quantised K): quants and fp16-rounded scales
    __shared__ float sdq[4][NBQ];
    if (p.use_pdl) { pdl_trigger(); pdl_wait(); }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wid = blockIdx.x * 4 + warp;
    if (wid >= p.n_q * p.H) return;
    const int col = wid / p.H, head = wid % p.H, hk = head / p.gq;
    const float *qp = (const float *)(p.q + (uint64_t)col * p.q_nb1 + (uint64_t)head * p.q_nb2);
    if (!QUANT) {
#pragma unroll
        for (int i = 0; i < PER; i++) sq[warp][lane + 32 * i] = __half2float(__float2half_rn(qp[lane + 32 * i]));
    } else {
        // quantize_row_q8_0 (AVX2 path, ggml-cpu-quants.c:808-845): block b = elements [32b, 32b+32), one element per lane
#pragma unroll
        for (int b = 0; b < NBQ; b++) {
            const float x = qp[32 * b + lane];
            const float amax = warp_reduce_max(fabsf(x));
            const float d = __fdiv_rn(amax, 127.0f);
            const float id = amax != 0.0f ? __fdiv_rn(127.0f, amax) : 0.0f;
            sqq[warp][32 * b + lane] = (int8_t)__float2int_rn(__fmul_rn(x, id));
            if (lane == 0) sdq[warp][b] = __half2float(__float2half_rn(d));
        }
    }
    __syncwarp();
    float slope = 1.0f;
    if (p.max_bias > 0.0f) slope = head < p.n_head_log2 ? powf(p.m0, (float)(head + 1)) : powf(p.m1, (float)(2 * (head - p.n_head_log2) + 1));
    const char *kbase = p.k + (uint64_t)hk * p.k_nb2;
    const char *vbase = p.v + (uint64_t)hk * p.v_nb2;
    const __half *mp = p.mask ? (const __half *)(p.mask + (uint64_t)col * p.m_nb1) : nullptr;
    float M = -INFINITY, S = 0.0f;
    float acc[PER];
#pragma unroll
    for (int i = 0; i < PER; i++) acc[i] = 0.0f;
    for (int c0 = 0; c0 < p.n_kv; c0 += 32) {
        const int ic = c0 + lane;
        float s = 0.0f;
        bool skip = ic >= p.n_kv;
        float mv = 0.0f;
        if (!skip && mp) { mv = __fmul_rn(slope, __half2float(mp[ic])); skip = mv == -INFINITY; }
        if (!skip) {
            if (!QUANT) {
                const uint4 *kr = (const uint4 *)(kbase + (uint64_t)ic * p.k_nb1);
                float sum[4][8];
#pragma unroll
                for (int j = 0; j < 4; j++)
#pragma unroll
                    for (int l = 0; l < 8; l++) sum[j][l] = 0.0f;
#pragma unroll
                for (int i = 0; i < D / 32; i++)
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const uint4 kv = kr[i * 4 + j];
                        const __half2 *h = (const __half2 *)&kv;
                        const float *qq = &sq[warp][i * 32 + j * 8];
#pragma unroll
                        for (int l = 0; l < 4; l++) {
                            const float2 kf = __half22float2(h[l]);
                            sum[j][2 * l] = __fmaf_rn(kf.x, qq[2 * l], sum[j][2 * l]);
                            sum[j][2 * l + 1] = __fmaf_rn(kf.y, qq[2 * l + 1], sum[j][2 * l + 1]);
                        }
                    }
                float x0[8];
#pragma unroll
                for (int l = 0; l < 8; l++) x0[l] = __fadd_rn(__fadd_rn(sum[0][l], sum[2][l]), __fadd_rn(sum[1][l], sum[3][l]));
                const float t0 = __fadd_rn(x0[0], x0[4]), t1 = __fadd_rn(x0[1], x0[5]), t2 = __fadd_rn(x0[2], x0[6]), t3 = __fadd_rn(x0[3], x0[7]);
                s = __fadd_rn(__fadd_rn(t0, t1), __fadd_rn(t2, t3));
            } else {
                // ggml_vec_dot_{q8_0,q4_0}_q8_0, AVX2 order (see exact.cu): 8 lane partials per block, one FMA per block, hsum_float_8
                const uint8_t *kr = (const uint8_t *)(kbase + (uint64_t)ic * p.k_nb1);
                float a8[8];
#pragma unroll
                for (int l = 0; l < 8; l++) a8[l] = 0.0f;
#pragma unroll
                for (int b = 0; b < NBQ; b++) {
                    const uint8_t *blk = kr + b * BB;
                    const float d = __fmul_rn(__half2float(__ushort_as_half((unsigned short)(blk[0] | (blk[1] << 8)))), sdq[warp][b]);
#pragma unroll
                    for (int l = 0; l < 8; l++) {
                        const uint32_t a = *(const uint32_t *)&sqq[warp][32 * b + 4 * l];
                        uint32_t w;
                        if (KT == KV_Q8_0) w = (uint32_t)blk[2 + 4 * l] | ((uint32_t)blk[3 + 4 * l] << 8) | ((uint32_t)blk[4 + 4 * l] << 16) | ((uint32_t)blk[5 + 4 * l] << 24);
                        else {
                            const int o = 2 + 4 * (l & 3);
                            const uint32_t raw = (uint32_t)blk[o] | ((uint32_t)blk[o + 1] << 8) | ((uint32_t)blk[o + 2] << 16) | ((uint32_t)blk[o + 3] << 24);
                            w = __vsub4(l < 4 ? (raw & 0x0f0f0f0fu) : ((raw >> 4) & 0x0f0f0f0fu), 0x08080808u);
                        }
                        a8[l] = __fmaf_rn(d, (float)__dp4a((int)w, (int)a, 0), a8[l]);
                    }
                }
                s = __fadd_rn(__fadd_rn(__fadd_rn(a8[0], a8[4]), __fadd_rn(a8[2], a8[6])), __fadd_rn(__fadd_rn(a8[1], a8[5]), __fadd_rn(a8[3], a8[7])));
            }
            s = __fmul_rn(s, p.scale);
            if (p.softcap != 0.0f) s = __fmul_rn(p.softcap, tanhf(s));
            s = __fadd_rn(s, mv);
        }
        const unsigned live = __ballot_sync(0xffffffffu, !skip);
        for (int t = 0; t < 32; t++) {
            if (!((live >> t) & 1u)) continue;
            const float sc = __shfl_sync(0xffffffffu, s, t);
            float vv[PER];
            if (!QUANT) {
                const __half *vr = (const __half *)(vbase + (uint64_t)(c0 + t) * p.v_nb1) + lane * PER;
                if (PER == 4) { const uint2 raw = *(const uint2 *)vr; const float2 a = __half22float2(*(const __half2 *)&raw.x), b = __half22float2(*(const __half2 *)&raw.y); vv[0] = a.x; vv[1] = a.y; vv[PER - 2] = b.x; vv[PER - 1] = b.y; }
                else { const float2 a = __half22float2(*(const __half2 *)vr); vv[0] = a.x; vv[1] = a.y; }
            } else {
                // dequantize_row_q8_0 / q4_0 (ggml-quants.c:349, 255): (float)q * d; lane owns elements [PER*lane, PER*lane + PER)
                const uint8_t *vr = (const uint8_t *)(vbase + (uint64_t)(c0 + t) * p.v_nb1);
#pragma unroll
                for (int i = 0; i < PER; i++) {
                    const int e = lane * PER + i, b = e >> 5, j = e & 31;
                    const uint8_t *blk = vr + b * BB;
                    const float d = __half2float(__ushort_as_half((unsigned short)(blk[0] | (blk[1] << 8))));
                    int q;
                    if (KT == KV_Q8_0) q = (int)(int8_t)blk[2 + j];
                    else q = (j < 16 ? (blk[2 + j] & 0x0f) : (blk[2 + j - 16] >> 4)) - 8;
                    vv[i] = __fmul_rn((float)q, d);
                }
            }
            float ms = 1.0f, vs = 1.0f;
            if (sc > M) {
                ms = exp_rn(M - sc);
                M = sc;
#pragma unroll
                for (int i = 0; i < PER; i++) acc[i] = QUANT ? __fmul_rn(acc[i], ms) : __half2float(__float2half_rn(__fmul_rn(acc[i], ms)));
            } else vs = exp_rn(sc - M);
#pragma unroll
            for (int i = 0; i < PER; i++) acc[i] = QUANT ? __fmaf_rn(vv[i], vs, acc[i]) : __half2float(__float2half_rn(__fmaf_rn(vv[i], vs, acc[i])));
            S = __fadd_rn(__fmul_rn(S, ms), vs);
        }
    }
    const float Sinv = __fdiv_rn(1.0f, S);
    float *o = p.dst + ((uint64_t)col * p.H + head) * D + lane * PER;
#pragma unroll
    for (int i = 0; i < PER; i++) o[i] = __fmul_rn(acc[i], Sinv);
}

int kv_kind(int type) { return type == B200_TYPE_F16 ? KV_F16 : type == B200_TYPE_Q8_0 ? KV_Q8_0 : type == B200_TYPE_Q4_0 ? KV_Q4_0 : -1; }

template <int D, int KT, int VT, bool ROWS8 = false>
int launch_fa(b200_ctx *ctx, const FaParams &p, int n_tiles) {
    constexpr int LD = D + 8;
    constexpr int RAWK = KT != KV_F16 ? BK * (KT == KV_Q8_0 ? 34 : 18) * (D / 32) : 0, RAWV = VT != KV_F16 ? BK * (VT == KV_Q8_0 ? 34 : 18) * (D / 32) : 0;
    constexpr int WARP_BYTES = 2 * BK * LD * 2 + 2 * BK * (D / 32) * 4 + RAWK + RAWV + (ROWS8 ? 2 * 8 * 40 * 2 : 0);
    constexpr int COMBINE_BYTES = (2 * NWARP * 16 + NWARP * 16 * D) * 4;      // warp merge area (fa_merge_store)
    constexpr int SMEM = NWARP * WARP_BYTES > COMBINE_BYTES ? NWARP * WARP_BYTES : COMBINE_BYTES;
    auto kern = ROWS8 ? b200_fattn_rows8_kernel<D, KT, VT> : b200_fattn_kernel<D, KT, VT>;
    static bool attr_set[16] = {false};
    if (!attr_set[ctx->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
        attr_set[ctx->device & 15] = true;
    }
    cudaLaunchAttribute attr[1];
    int na = 0;
    if (p.use_pdl) { attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization; attr[na].val.programmaticStreamSerializationAllowed = 1; na++; }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)p.n_splits, (unsigned)n_tiles);
    cfg.blockDim = dim3(NWARP * 32);
    cfg.dynamicSmemBytes = SMEM;
    cfg.stream = ctx->stream;
    cfg.attrs = attr;
    cfg.numAttrs = na;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, p));
    ctx->launches++;
    if (p.n_splits > 1) {
        cfg.gridDim = dim3((unsigned)((n_tiles * 16 + 3) / 4));
        cfg.blockDim = dim3(128);
        cfg.dynamicSmemBytes = 0;
        CUDA_TRY(cudaLaunchKernelEx(&cfg, b200_fattn_combine_kernel<D>, p, n_tiles));
        ctx->launches++;
    }
    return B200_OK;
}

template <int D>
int launch_fa_types(b200_ctx *ctx, const FaParams &p, int n_tiles, int kt, int vt, bool rows8) {
    if (kt == KV_F16 && vt == KV_F16) return rows8 ? launch_fa<D, KV_F16, KV_F16, true>(ctx, p, n_tiles) : launch_fa<D, KV_F16, KV_F16>(ctx, p, n_tiles);
    if (D == 128) {
        if constexpr (D == 128) {
            if (kt == KV_Q8_0 && vt == KV_Q8_0) return rows8 ? launch_fa<128, KV_Q8_0, KV_Q8_0, true>(ctx, p, n_tiles) : launch_fa<128, KV_Q8_0, KV_Q8_0>(ctx, p, n_tiles);
            if (kt == KV_Q4_0 && vt == KV_Q4_0) return rows8 ? launch_fa<128, KV_Q4_0, KV_Q4_0, true>(ctx, p, n_tiles) : launch_fa<128, KV_Q4_0, KV_Q4_0>(ctx, p, n_tiles);
        }
    }
    b200_set_error("flash_attn: K/V type combination not built");
    return B200_ERR_UNSUPPORTED;
}

}  // namespace

bool supports_flash_attn_ext(const b200_op *op) {
    const b200_tensor &q = op->src[0], &k = op->src[1], &v = op->src[2], &m = op->src[3], &d = op->dst;
    if (q.type != B200_TYPE_F32 || d.type != B200_TYPE_F32) return false;
    const int64_t D = q.ne[0];
    if (D != 64 && D != 128) return false;
    if (k.ne[0] != D || v.ne[0] != D) return false;
    const int kt = kv_kind(k.type), vt = kv_kind(v.type);
    if (kt < 0 || vt < 0 || kt != vt) return false;
    if (kt != KV_F16 && D != 128) return false;
    if (q.ne[3] != 1 || k.ne[3] != 1 || v.ne[3] != 1) return false;
    const int64_t H = q.ne[2], Hkv = k.ne[2], n_kv = k.ne[1];
    if (Hkv == 0 || H % Hkv || v.ne[2] != Hkv || v.ne[1] != n_kv) return false;
    if (n_kv % BK != 0 || n_kv == 0) return false;
    if (q.nb[0] != 4 || (q.nb[1] & 7) || (q.nb[2] & 7) || ((uintptr_t)q.data & 7)) return false;
    const uint64_t rowb = b200_row_bytes(k.type, D);
    if (k.nb[0] != (uint64_t)b200_type_block_bytes(k.type) || v.nb[0] != k.nb[0]) return false;
    const uint64_t al = kt == KV_F16 ? 15 : 7;
    if ((k.nb[1] & al) || (k.nb[2] & al) || (v.nb[1] & al) || (v.nb[2] & al) || ((uintptr_t)k.data & al) || ((uintptr_t)v.data & al)) return false;
    if (k.nb[1] < rowb || v.nb[1] < rowb) return false;
    if (!tensor_is_contiguous(d)) return false;
    if (op->n_src > 3 && m.data) {
        if (m.type != B200_TYPE_F16 || m.ne[0] != n_kv || m.ne[1] < q.ne[1] || m.nb[0] != 2 || (m.nb[1] & 3) || ((uintptr_t)m.data & 3)) return false;
    }
    return true;
}

int op_flash_attn_ext(b200_ctx *ctx, const b200_op *op) {
    const b200_tensor &q = op->src[0], &k = op->src[1], &v = op->src[2], &m = op->src[3], &d = op->dst;
    FaParams p = {};
    const int D = (int)q.ne[0];
    p.q = (const char *)q.data; p.q_nb1 = q.nb[1]; p.q_nb2 = q.nb[2]; p.q_nb3 = q.nb[3];
    p.k = (const char *)k.data; p.k_nb1 = k.nb[1]; p.k_nb2 = k.nb[2]; p.k_nb3 = k.nb[3];
    p.v = (const char *)v.data; p.v_nb1 = v.nb[1]; p.v_nb2 = v.nb[2]; p.v_nb3 = v.nb[3];
    const bool has_mask = op->n_src > 3 && m.data != nullptr;
    p.mask = has_mask ? (const char *)m.data : nullptr; p.m_nb1 = has_mask ? m.nb[1] : 0;
    p.dst = (float *)d.data;
    p.n_q = (int)q.ne[1]; p.n_kv = (int)k.ne[1]; p.H = (int)q.ne[2]; p.Hkv = (int)k.ne[2];
    p.gq = p.H / p.Hkv;
    p.HG = p.gq < 16 ? p.gq : 16;
    p.QC = 16 / p.HG;
    p.n_headtiles = (p.gq + p.HG - 1) / p.HG;
    p.n_coltiles = (p.n_q + p.QC - 1) / p.QC;
    memcpy(&p.scale, &op->params[0], 4);
    memcpy(&p.max_bias, &op->params[1], 4);
    memcpy(&p.softcap, &op->params[2], 4);
    if (p.softcap != 0.0f) p.scale /= p.softcap;
    p.n_head_log2 = 1 << (int)floorf(log2f((float)p.H));
    p.use_pdl = ctx->opt_pdl;
    p.m0 = powf(2.0f, -(p.max_bias) / p.n_head_log2);
    p.m1 = powf(2.0f, -(p.max_bias / 2.0f) / p.n_head_log2);
    // decode and continuous-batching steps: the few-row kernel (tile = one KV head x one column, the GQA group's heads as the MMA N = 8)
    static const int use_rows8 = getenv("GGML_B200_FA_ROWS8") ? atoi(getenv("GGML_B200_FA_ROWS8")) : 1;
    const bool rows8 = use_rows8 && !ctx->opt_cpu_exact && p.gq <= 8 && p.n_q <= 32 && kv_kind(k.type) == kv_kind(v.type) && kv_kind(k.type) >= 0;
    if (rows8) { p.HG = p.gq; p.QC = 1; p.n_headtiles = 1; p.n_coltiles = p.n_q; }
    const int n_tiles = p.Hkv * p.n_headtiles * p.n_coltiles;
    if (n_tiles == 0 || p.n_q == 0) return B200_OK;
    // parity mode: reproduce the CPU's fp16 V accumulator (see b200_fattn_f16acc_kernel)
    if (ctx->opt_cpu_exact && kv_kind(k.type) == kv_kind(v.type)) {
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)((p.n_q * p.H + 3) / 4));
        cfg.blockDim = dim3(128);
        cfg.stream = ctx->stream;
        cfg.attrs = attr;
        cfg.numAttrs = p.use_pdl ? 1 : 0;
        const int kt_ = kv_kind(k.type);
        if (D == 128 && kt_ == KV_F16) CUDA_TRY(cudaLaunchKernelEx(&cfg, b200_fattn_f16acc_kernel<128, KV_F16>, p));
        else if (D == 128 && kt_ == KV_Q8_0) CUDA_TRY(cudaLaunchKernelEx(&cfg, b200_fattn_f16acc_kernel<128, KV_Q8_0>, p));
        else if (D == 128 && kt_ == KV_Q4_0) CUDA_TRY(cudaLaunchKernelEx(&cfg, b200_fattn_f16acc_kernel<128, KV_Q4_0>, p));
        else CUDA_TRY(cudaLaunchKernelEx(&cfg, b200_fattn_f16acc_kernel<64, KV_F16>, p));
        ctx->launches++;
        return B200_OK;
    }
    // prompt-sized query blocks at head size 128: the tcgen05 kernel (fattn_tc.cu: 128 query rows of one head per CTA, S and the per-tile
    // P V in TMEM).  Soft-capping and ALiBi slopes stay on the mma.sync kernel below.
    static const int use_tc = getenv("GGML_B200_FA_TC") ? atoi(getenv("GGML_B200_FA_TC")) : 1;
    static const int tc_min_q = getenv("GGML_B200_FA_TC_MIN_Q") ? atoi(getenv("GGML_B200_FA_TC_MIN_Q")) : 64;
    if (use_tc && D == 128 && p.n_q >= tc_min_q && kv_kind(k.type) == kv_kind(v.type) && kv_kind(k.type) >= 0 && p.softcap == 0.0f && p.max_bias == 0.0f &&
        p.n_kv % 64 == 0 && !(((uintptr_t)q.data | q.nb[1] | q.nb[2] | (uintptr_t)d.data) & 15) && (!has_mask || !(((uintptr_t)m.data | m.nb[1]) & 15))) {
        FaTcArgs a = {};
        a.q = p.q; a.q_nb1 = p.q_nb1; a.q_nb2 = p.q_nb2; a.k = p.k; a.k_nb1 = p.k_nb1; a.k_nb2 = p.k_nb2; a.v = p.v; a.v_nb1 = p.v_nb1; a.v_nb2 = p.v_nb2;
        a.mask = p.mask; a.m_nb1 = p.m_nb1; a.dst = p.dst; a.n_q = p.n_q; a.n_kv = p.n_kv; a.H = p.H; a.gq = p.gq; a.scale = p.scale;
        return fattn_tc_launch(ctx, a, kv_kind(k.type));
    }
    // batched steps and prompt ubatches: live-tile map of the mask, shared by every layer of the graph
    static const int use_map = getenv("GGML_B200_FA_MAP") ? atoi(getenv("GGML_B200_FA_MAP")) : 1;
    if (use_map && has_mask && p.n_q > 1 && p.n_kv / BK <= 4 * MAP_MAX_BATCH * 32 && !((uintptr_t)m.data & 15) && !(m.nb[1] & 15)) {
        p.map_stride = p.n_kv / BK + 1;
        const size_t need = (size_t)p.n_coltiles * p.map_stride * sizeof(int);
        const bool grow = need > ctx->scratch_size[SCRATCH_FAMAP];
        int *map = (int *)ctx->get_scratch(SCRATCH_FAMAP, need);
        if (!map) return B200_ERR_ALLOC;
        const int64_t key[4] = {(int64_t)m.nb[1], p.n_kv, p.n_q, p.QC};
        if (grow || !ctx->fa_map_valid || ctx->fa_map_mask != (uintptr_t)m.data || memcmp(key, ctx->fa_map_key, sizeof(key)) != 0) {
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[0].val.programmaticStreamSerializationAllowed = 1;
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((unsigned)p.n_coltiles); cfg.blockDim = dim3(128); cfg.stream = ctx->stream;
            cfg.attrs = attr; cfg.numAttrs = p.use_pdl ? 1 : 0;
            CUDA_TRY(cudaLaunchKernelEx(&cfg, b200_fattn_maskmap_kernel, p.mask, p.m_nb1, p.n_q, p.n_kv, p.QC, map, p.map_stride, p.use_pdl));
            ctx->launches++;
            ctx->fa_map_valid = true; ctx->fa_map_mask = (uintptr_t)m.data; ctx->fa_map_mask_end = (uintptr_t)m.data + (size_t)m.nb[1] * (size_t)m.ne[1];
            memcpy(ctx->fa_map_key, key, sizeof(key));
        }
        p.map = map;
    }
    // split the KV range so the grid covers the machine ~2-3x; each split is a multiple of NWARP*BK positions
    const int unit = NWARP * BK;
    const int max_splits = (p.n_kv + unit - 1) / unit;
    int ns = (3 * ctx->sm_count + n_tiles - 1) / n_tiles;
    if (p.map) ns = (2 * ctx->sm_count) / n_tiles;
    if (rows8) ns = (2 * ctx->sm_count) / n_tiles;            // one wave of the 2 resident CTAs per SM; a full batch needs no split at all      // live tiles are shared evenly: one full wave of the 2 resident CTAs per SM (the per-warp
                                                        // set-up -- Q fragments, merge -- costs about as much as one KV tile)
    if (ns > max_splits) ns = max_splits;
    if (ns < 1) ns = 1;
    p.kv_per_split = ((p.n_kv + ns - 1) / ns + unit - 1) / unit * unit;
    ns = (p.n_kv + p.kv_per_split - 1) / p.kv_per_split;
    p.n_splits = ns;
    if (ns > 1) {
        // sized by its upper bound (n_tiles * ns <= 4 * sm_count + n_tiles) so that a growing n_kv never reallocates it under
        // captured graphs
        p.part = (float *)ctx->get_scratch(SCRATCH_FATTN, (size_t)(4 * ctx->sm_count + n_tiles) * 16 * (D + 2) * 4);
        if (!p.part) return B200_ERR_ALLOC;
    }
    const int kt = kv_kind(k.type), vt = kv_kind(v.type);
    if (D == 128) return launch_fa_types<128>(ctx, p, n_tiles, kt, vt, rows8);
    if (D == 64) return launch_fa_types<64>(ctx, p, n_tiles, kt, vt, rows8);
    b200_set_error("flash_attn: D=%d", D);
    return B200_ERR_UNSUPPORTED;
}
