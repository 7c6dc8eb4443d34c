// gemm_tc.cu -- K-quant matmul for token batches (continuous-batching decode steps up to prompt ubatches) on the 5th-generation
// tensor cores: tcgen05.mma kind::f16 with EXACT-INTEGER f16 operands, f32 accumulators in TMEM.
//
// Replaces mul_mat_q (ggml-cuda/mmq.cuh:2501-2657: mma.sync m16n8k32 on q8_1 activations, float fix-up per 32-k block) and, behind
// it, the CPU's ggml_vec_dot_q{4,5,6}_K_q8_K (ggml-cpu-quants.c) whose per-super-block integers it reproduces:
//   * activations: quantised once per matmul to q8_K exactly like quantize_row_q8_K_ref (quant_warp.cuh) by a pack kernel that writes
//     the int8 quants AS f16 INTEGERS into the tensor core's canonical K-major layout -- one contiguous image per (token tile,
//     super-block) = four 64-k operand stages + a 16-column tile of the per-16 quant sums (for the min term) -- and the block scale d;
//   * weights stay GGUF blocks in HBM.  The expander warps stage the raw blocks of 128 rows with 16-byte cp.async (completion on an
//     mbarrier), then turn every 4/5/6-bit quant times its 6-bit (Q4_K/Q5_K) or int8 (Q6_K) sub-block scale into ONE f16 operand
//     element w' = sc_j * q: <= 1953, exactly representable, built with the 0x6400 magic-number trick (PRMT + one HFMA2 per two
//     weights).  Q6_K's |sc * (q - 32)| reaches 4064 (12 bits), so it is written as two exact operand tiles
//     2*sc*((q >> 1) - 16) and sc*(q & 1) that accumulate into the same TMEM columns;
//   * per 256-k super-block the tensor core accumulates  P = sum_j sc_j sum_l q_jl a_jl  (16 MMAs of K = 16) and, for Q4_K/Q5_K,
//     the min term  Mn = sum_j m_j * bsum_j  as ONE extra K = 16 MMA (operand rows: the 6-bit mins twice, the per-16 activation
//     sums) into a second accumulator.  All values are integers below 2^24 in f32: the CPU's integers, bit for bit;
//   * the drain warps read both accumulators (tcgen05.ld), and fold  d_a * (d_w * P - dmin_w * Mn)  into f32 registers: three
//     flops per element per super-block, nothing else -- no hi/lo operand split, no dp2a, no int->float conversion.
// The round-1 kind::i8 kernel (measured slower and removed, DESIGN.md 8) needed two operand tiles + two accumulators + a 16-instruction
// drain per element; the mma.sync kernel (gemm_mma.cu) is bounded by the legacy IMMA pipe and its 4 IMAD per IMMA.
// Roofline: tensor pipe (f16: half the int8 rate) for prompt batches, HBM for <= 32 tokens.  Algorithmic work: 2*N*K*M.
#include "common.cuh"
#include "quant_warp.cuh"
#include "tc05.cuh"
#include "gemm_tc.h"

namespace {

constexpr int TM = 128;                 // weight rows per CTA tile (MMA M = TMEM lanes)
// k per operand stage: 128 (two stages per super-block) for Q4_K / Q5_K, 64 for Q6_K whose weights need two operand tiles per stage
__host__ __device__ constexpr int stage_k(bool q6) { return q6 ? 64 : 128; }
constexpr int N_EXP = 8, N_DRAIN = 8;   // expander / drain warps; warp 0: activation producer, warp 1: MMA issuer
constexpr int TC_THREADS = (2 + N_EXP + N_DRAIN) * 32;
__host__ __device__ constexpr uint32_t main_bytes(int ks) { return (uint32_t)(TM * ks * 2); }      // one f16 operand tile of 128 rows: 16 / 32 KB
constexpr uint32_t MIN_BYTES = TM * 16 * 2;             // the min-term tile of 128 rows: 4 KB
// canonical K-major no-swizzle layout: 8 rows x 16 bytes = one 128-byte core matrix; K-adjacent core matrices 128 bytes apart (LBO),
// 8-row groups (chunks per row) * 128 bytes apart (SBO)
constexpr uint32_t LBO = 128, SBO_MIN = 2 * 128;
__host__ __device__ constexpr uint32_t sbo_main(int ks) { return (uint32_t)(ks / 8) * 128u; }

// activation image of one (token tile, super-block): [stage 0: tn x 2 ks B][min tiles u1, u2: 2 x tn x 32 B][stage 1]..[stage 256 / ks - 1]
__host__ __device__ inline uint32_t img_bytes(int tn) { return (uint32_t)tn * 576u; }
__host__ __device__ inline uint32_t img_stage_off(int tn, int s, int ks) { return s == 0 ? 0u : (uint32_t)tn * (64u + 2u * (uint32_t)ks * (uint32_t)s); }

struct TcParams {
    const uint8_t *W; uint32_t rb; int N, K, M, Mpad, nsb;
    const uint8_t *img;                 // [token tile][nsb] images
    const float *Bd;                    // [nsb][Mpad] q8_K block scales
    float *dst; size_t dst_stride;      // dst[tok * dst_stride + row]
    int sb_per_split; float *part;      // split-K: blockIdx.z covers super-blocks [z * sb_per_split, ...), partials [z][M][N]
    int na, nb, rs;                     // weight-operand ring depth, activation-operand ring depth (64-k stages), raw ring depth (super-blocks)
    uint32_t a_slot, b_slot, rstride;
    int nbm;                            // activation-side min-tile ring depth (super-blocks)
    // grouped mode (MUL_MAT_ID prompt batches): token tile = chunk of <= 128 (token, slot) pairs of one expert; g_E = 0: dense
    const int32_t *g_off, *g_pairs; int g_E, g_n_used, g_b_ne1; size_t g_expert_stride, g_d_nb1, g_d_nb2;
    unsigned long long *prof;           // optional in-kernel timeline of CTA 0 (GGML_B200_TC_PROF=1): [3 roles][256] clock64 stamps
    int dbg;                            // timing experiments (GGML_B200_TC_DBG): 1 skip expansion, 2 skip MMAs, 4 skip drain math, 8 skip the proxy fence
};

// grouped mode: chunk -> (expert, first pair, pairs in the chunk); cnt = 0: the chunk does not exist (fewer pairs than the upper bound)
__device__ __forceinline__ void tc_g_lookup(const TcParams &p, int chunk, int &e, int &first, int &cnt) {
    cnt = 0; first = 0;
    for (e = 0; e < p.g_E; e++) {
        const int o0 = p.g_off[e], n = p.g_off[e + 1] - o0, nch = (n + 127) / 128;
        if (chunk < nch) { first = o0 + chunk * 128; cnt = min(128, n - chunk * 128); return; }
        chunk -= nch;
    }
}

// a hang on the GPU box costs a whole lease: every wait in this kernel gives up (trap -> launch failure) after ~1 s.  No printf: a
// kernel that can print pays for the FIFO set-up at every launch.
__device__ __forceinline__ void tc_wait(uint64_t *bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 24)) __trap();
    }
}

// one lane of a fully converged warp.  The single-thread roles run their loops WARP-UNIFORMLY and predicate only the issue on this: inside
// an `if (lane == 0)` region the compiler cannot prove the tcgen05 / bulk-copy operands uniform and wraps every instruction in an
// R2UR + ELECT + BRA.U.ANY waterfall -- ~170 dependent SASS instructions per operand stage, which bounded the whole kernel
// (profiles/r2_gemm_tc.md)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------------------------------------------------------- activation pack
// one warp per (token, super-block); lane owns 8 consecutive elements
__global__ void __launch_bounds__(256) b200_gemm_tc_pack_kernel(const float *__restrict__ x, size_t x_stride, int K, int M, int Mpad, int nsb, int tn, int ks,
                                                                uint8_t *__restrict__ img, float *__restrict__ Bd, const TcParams g) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (gw >= (int64_t)Mpad * nsb) return;
    const int b = (int)(gw % nsb), tok = (int)(gw / nsb), tile = tok / tn, n = tok % tn;
    float v[8];
    int64_t col = tok;                                 // source column of this token slot (dense: itself)
    bool live = tok < M;
    if (g.g_E) {                                       // grouped: slot n of chunk `tile` = a (token, slot) pair of the chunk's expert
        int e, first, cnt;
        tc_g_lookup(g, tile, e, first, cnt);
        live = n < cnt;
        if (live) { const int pair = g.g_pairs[first + n]; col = g.g_b_ne1 == 1 ? pair / g.g_n_used : pair; }
    }
    if (live) {
        const float *xp = (const float *)((const char *)x + (size_t)col * x_stride) + b * 256 + lane * 8;
        const float4 a = *(const float4 *)xp, c = *(const float4 *)(xp + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
    } else {
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = 0.0f;
    }
    uint2 qp; float d; int pair;
    warp_quant_q8k(v, lane, qp, d, pair);              // pair: valid in even lanes = bsum of the 16-group lane / 2
    uint8_t *im = img + ((size_t)tile * nsb + b) * img_bytes(tn);
    const int s = lane * 8 / ks, c = (lane * 8 % ks) >> 3;     // operand stage, 16-byte chunk inside the stage row
    const int8_t *q = (const int8_t *)&qp;
    __half2 h[4];
#pragma unroll
    for (int j = 0; j < 4; j++) h[j] = __halves2half2(__int2half_rn(q[2 * j]), __int2half_rn(q[2 * j + 1]));
    *(uint4 *)(im + img_stage_off(tn, s, ks) + (uint32_t)(n >> 3) * sbo_main(ks) + (uint32_t)c * LBO + (uint32_t)(n & 7) * 16) = *(const uint4 *)h;
    // min-term operand: u_j = d * bsum_j (per-32 sums) split into two tf32 parts whose product with the weight side stays exact
    const int s32 = pair + __shfl_down_sync(0xffffffffu, pair, 2);      // lanes 0, 4, 8, ..: sum of the 32-group lane / 4
    if ((lane & 3) == 0) {
        const int j = lane >> 2;
        const float u = __fmul_rn(d, (float)s32);
        const float u1 = __uint_as_float(__float_as_uint(u) & 0xffffe000u);
        const float u2 = __uint_as_float(__float_as_uint(__fsub_rn(u, u1)) & 0xffffe000u);
        uint8_t *mp = im + (uint32_t)tn * 2u * (uint32_t)ks + (uint32_t)(n >> 3) * SBO_MIN + (uint32_t)(j >> 2) * LBO + (uint32_t)(n & 7) * 16 + (uint32_t)(j & 3) * 4;
        *(float *)mp = u1;
        *(float *)(mp + (uint32_t)tn * 32u) = u2;
    }
    if (lane == 0) Bd[(size_t)b * Mpad + tok] = d;
}

// ---------------------------------------------------------------------------------------------------------------- weight expansion
__device__ __forceinline__ __half2 u32_h2(uint32_t u) { return *(const __half2 *)&u; }
__device__ __forceinline__ uint32_t h2_u32(__half2 h) { return *(const uint32_t *)&h; }
// bytes (2p, 2p+1) of `w` (each < 1024) -> half2 of the integers 1024 + byte
__device__ __forceinline__ __half2 magic_pair(uint32_t w, int p) { return u32_h2(__byte_perm(w, 0x64646464u, p ? 0x4342 : 0x4140)); }

// 8 words from a 2-byte aligned shared-memory address
__device__ __forceinline__ void lds8_unaligned(const uint8_t *p, uint32_t (&w)[8]) {
    const uint32_t *q = (const uint32_t *)((uintptr_t)p & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)((uintptr_t)p & 2) * 8;
    uint32_t t[9];
#pragma unroll
    for (int i = 0; i < 9; i++) t[i] = q[i];
#pragma unroll
    for (int i = 0; i < 8; i++) w[i] = __funnelshift_r(t[i], t[i + 1], sh);
}

struct KHeader { uint32_t sc_lo, sc_hi, m_lo, m_hi; float d, dmin; };      // Q4_K / Q5_K: 6-bit scales and mins as bytes (get_scale_min_k4, ggml-quants.c:631)
__device__ __forceinline__ KHeader read_kheader(const uint8_t *blk) {
    const uint4 h = *(const uint4 *)blk;                                   // d, dmin, scales[12]
    KHeader k;
    k.d = half_bits_to_float(h.x); k.dmin = half_bits_to_float(h.x >> 16);
    k.sc_lo = h.y & 0x3f3f3f3fu; k.m_lo = h.z & 0x3f3f3f3fu;
    k.sc_hi = (h.w & 0x0f0f0f0fu) | ((h.y >> 2) & 0x30303030u);
    k.m_hi = ((h.w >> 4) & 0x0f0f0f0fu) | ((h.z >> 2) & 0x30303030u);
    return k;
}

// min-term operand row: v_j = dmin * m_j (exact in f32: 11 x 6 bits) as two tf32 parts hi + lo (8 k-columns of 4 bytes each); the activation
// side holds u_j = d_a * bsum_j as u1 + u2: the tensor core accumulates hi*u1 + hi*u2 + lo*u1 (every product exact, 2^-21 of the term dropped)
__device__ __forceinline__ void write_min_row(const KHeader &k, int r, uint8_t *a_hi, uint8_t *a_lo) {
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const float v = __fmul_rn(k.dmin, (float)(((j < 4 ? k.m_lo : k.m_hi) >> (8 * (j & 3))) & 0xffu));
        hi[j] = __float_as_uint(v) & 0xffffe000u;
        lo[j] = __float_as_uint(__fsub_rn(v, __uint_as_float(hi[j])));
    }
    const uint32_t off = (uint32_t)(r >> 3) * SBO_MIN + (uint32_t)(r & 7) * 16;
    *(uint4 *)(a_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *(uint4 *)(a_hi + off + LBO) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
    *(uint4 *)(a_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    *(uint4 *)(a_lo + off + LBO) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
}

// Q4_K / Q5_K, 128-k stages: thread (row r, half h) expands the 32-byte quant group 2 s + h of stage s = sub-blocks j = 2 (2 s + h) (low
// nibbles) and j + 1 (high nibbles), 64 weights, into chunks 8 h .. 8 h + 7 of the operand row
template <bool Q5>
__device__ __forceinline__ void expand_k45(const uint8_t *blk, const KHeader &k, const uint32_t (&qh)[8], int s, int h, int r, uint8_t *a_main) {
    const int grp = 2 * s + h;
    const uint4 *qs = (const uint4 *)(blk + (Q5 ? 48 : 16) + 32 * grp);
    const uint4 q0 = qs[0], q1 = qs[1];
    const uint32_t w[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
    const uint32_t scw = s ? k.sc_hi : k.sc_lo;            // sub-blocks 4 s .. 4 s + 3 live in one scale word
    uint8_t *dst = a_main + (uint32_t)(r >> 3) * sbo_main(128) + (uint32_t)(8 * h) * LBO + (uint32_t)(r & 7) * 16;
#pragma unroll
    for (int nib = 0; nib < 2; nib++) {
        const int j = 2 * grp + nib;
        const __half sch = __int2half_rn((int)((scw >> (8 * (2 * h + nib))) & 0xffu));
        const __half2 sc2 = __half2half2(sch), nsc2 = __half2half2(__hmul(sch, __float2half_rn(-1024.0f)));
#pragma unroll
        for (int c = 0; c < 4; c++) {
            uint32_t o[4];
#pragma unroll
            for (int e = 0; e < 2; e++) {
                const int wi = 2 * c + e;
                uint32_t n4 = (nib ? w[wi] >> 4 : w[wi]) & 0x0f0f0f0fu;
                if (Q5) n4 |= ((qh[wi] >> j) & 0x01010101u) << 4;
                o[2 * e]     = h2_u32(__hfma2(magic_pair(n4, 0), sc2, nsc2));
                o[2 * e + 1] = h2_u32(__hfma2(magic_pair(n4, 1), sc2, nsc2));
            }
            *(uint4 *)(dst + (uint32_t)(4 * nib + c) * LBO) = make_uint4(o[0], o[1], o[2], o[3]);
        }
    }
}

// Q6_K: thread (r, h) expands quadrant t = 2 (s & 1) + h of half hf = s >> 1 (ggml-quants.c:1690-1719) into the two exact tiles
__device__ __forceinline__ void expand_q6k(const uint8_t *blk, int s, int h, int r, uint8_t *a_even, uint8_t *a_odd) {
    const int hf = s >> 1, t = 2 * (s & 1) + h;
    uint32_t ql[8], qh[8];
    lds8_unaligned(blk + 64 * hf + 32 * h, ql);
    lds8_unaligned(blk + 128 + 32 * hf, qh);
    const uint32_t scw = *(const unsigned short *)(blk + 192 + 8 * hf + 2 * t);
    const __half m1040 = __float2half_rn(-1040.0f), m1024 = __float2half_rn(-1024.0f);
    const __half2 o1040 = __half2half2(m1040), o1024 = __half2half2(m1024);
    const uint32_t off = (uint32_t)(r >> 3) * sbo_main(64) + (uint32_t)(4 * h) * LBO + (uint32_t)(r & 7) * 16;
#pragma unroll
    for (int c = 0; c < 4; c++) {
        const int sci = (int)(int8_t)(c < 2 ? (scw & 0xffu) : (scw >> 8));         // 16-element scale group of this chunk pair
        const __half sch = __int2half_rn(sci);
        const __half2 sc2 = __half2half2(sch), sc2x2 = __hadd2(sc2, sc2);
        uint32_t ev[4], od[4];
#pragma unroll
        for (int e = 0; e < 2; e++) {
            const int wi = 2 * c + e;
            const uint32_t q4 = ((ql[wi] >> (4 * (s & 1))) & 0x0f0f0f0fu) | (((qh[wi] >> (2 * t)) & 0x03030303u) << 4);     // 4 x (0..63)
            const uint32_t vh = (q4 >> 1) & 0x1f1f1f1fu, vl = q4 & 0x01010101u;
#pragma unroll
            for (int p = 0; p < 2; p++) {
                ev[2 * e + p] = h2_u32(__hmul2(__hadd2(magic_pair(vh, p), o1040), sc2x2));       // 2 sc ((q >> 1) - 16): |.| <= 4064, even
                od[2 * e + p] = h2_u32(__hmul2(__hadd2(magic_pair(vl, p), o1024), sc2));         // sc (q & 1)
            }
        }
        *(uint4 *)(a_even + off + (uint32_t)c * LBO) = make_uint4(ev[0], ev[1], ev[2], ev[3]);
        *(uint4 *)(a_odd + off + (uint32_t)c * LBO) = make_uint4(od[0], od[1], od[2], od[3]);
    }
}

// ---------------------------------------------------------------------------------------------------------------- the GEMM
struct TcBars {
    // operand stage g uses full[g & 15] / empty[g & 15] (phase (g >> 4) & 1) whatever the two operand rings' depths are: the expanders (8
    // arrivals) and the activation producer (1 arrival + the copies' bytes) complete `full`, ONE tcgen05.commit completes `empty`
    uint64_t raw_full[8], raw_empty[8], full[16], empty[16], acc_full[2], acc_empty[2];
    uint32_t tmem_base, pad[3];
};

template <int TYPE, int TN>
__global__ void __launch_bounds__(TC_THREADS, 1) b200_gemm_tc_kernel(const TcParams p) {
    constexpr bool Q6 = TYPE == B200_TYPE_Q6_K, Q5 = TYPE == B200_TYPE_Q5_K;
    constexpr int BLK = TYPE == B200_TYPE_Q4_K ? 144 : TYPE == B200_TYPE_Q5_K ? 176 : 210;
    constexpr int CPR = TYPE == B200_TYPE_Q4_K ? 9 : TYPE == B200_TYPE_Q5_K ? 11 : 14;       // 16-byte chunks per staged row piece (Q6_K: phase <= 14, + 210)
    constexpr int KS = stage_k(Q6), SPS = 256 / KS, LG_SPS = Q6 ? 2 : 1;                        // k per stage, stages per super-block
    constexpr uint32_t MAIN_BYTES = main_bytes(KS), SBO_MAIN = sbo_main(KS);
    constexpr int CH = TN / 2;                                                                // token columns per drain thread
    extern __shared__ __align__(1024) uint8_t tsm[];
    uint8_t *a_ring = tsm;
    uint8_t *b_ring = a_ring + (size_t)p.na * p.a_slot;
    uint8_t *raw = b_ring + (size_t)p.nb * p.b_slot;
    uint8_t *amin = raw + (size_t)p.rs * TM * p.rstride;                  // [hi | lo] tf32 tiles of the current super-block's mins (2 x 4 KB)
    uint8_t *bmin = amin + (Q6 ? 0 : 2 * MIN_BYTES);                      // [nbm][u1 | u2] (2 x TN x 32 B)
    float2 *meta = (float2 *)(bmin + (Q6 ? 0 : (size_t)p.nbm * TN * 64));       // [4][TM]: (d, dmin) of the row's super-block
    TcBars *S = (TcBars *)(meta + 4 * TM);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row0 = blockIdx.x * TM, tok0 = blockIdx.y * TN;
    int g_e = 0, g_first = 0, g_cnt = TN;
    if (p.g_E) {                                       // grouped: this token tile is a chunk of one expert's pairs (or does not exist)
        tc_g_lookup(p, blockIdx.y, g_e, g_first, g_cnt);
        if (g_cnt == 0) return;
    }
    const int sb0 = (int)blockIdx.z * p.sb_per_split;
    const int nsb = min(p.sb_per_split, p.nsb - sb0);
    const int na = p.na, nb = p.nb, rs = p.rs;

    if (threadIdx.x == 0) {
        for (int i = 0; i < 8; i++) { mbar_init(&S->raw_full[i], N_EXP * 32); mbar_init(&S->raw_empty[i], N_EXP); }
        for (int i = 0; i < 16; i++) { mbar_init(&S->full[i], N_EXP + 1); mbar_init(&S->empty[i], 1); }
        for (int i = 0; i < 2; i++) { mbar_init(&S->acc_full[i], 1); mbar_init(&S->acc_empty[i], N_DRAIN); }
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&S->tmem_base, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = S->tmem_base;
#define TPROF(role, idx) do { if (p.prof && lane == 0 && (blockIdx.x | blockIdx.y | blockIdx.z) == 0 && (idx) < 256) p.prof[(role) * 256 + (idx)] = (unsigned long long)clock64(); } while (0)

    if (warp == 0) {
        // ------------------------------------------------------------ activation producer: one bulk copy per operand stage
        {
            const uint8_t *src = p.img + ((size_t)blockIdx.y * p.nsb + sb0) * img_bytes(TN);
            int slot = 0, mslot = 0;                   // activation ring slot g % nb, min-tile ring slot b % nbm (kept incrementally: run-time depths)
            for (int g = 0; g < SPS * nsb; g++) {
                const int b = g >> LG_SPS, s = g & (SPS - 1);
                if (p.dbg & 32) break;
                if (g >= nb) tc_wait(&S->empty[(g - nb) & 15], ((g - nb) >> 4) & 1);
                const bool with_min = s == 0 && !Q6;
                if (elect_one()) {
                    uint64_t *bar = &S->full[g & 15];
                    mbar_arrive_expect_tx(bar, (uint32_t)TN * (2u * KS + (with_min ? 64u : 0u)));
                    const uint8_t *sp = src + (size_t)b * img_bytes(TN) + img_stage_off(TN, s, KS);
                    bulk_g2s(b_ring + (size_t)slot * p.b_slot, sp, (uint32_t)TN * 2u * KS, bar);
                    if (with_min) bulk_g2s(bmin + (size_t)mslot * TN * 64, sp + (size_t)TN * 2 * KS, (uint32_t)TN * 64u, bar);
                }
                __syncwarp();
                if (with_min && ++mslot == p.nbm) mslot = 0;
                if (++slot == nb) slot = 0;
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer (warp-uniform loop, one elected lane issues)
        {
            const uint32_t idesc = (1u << 4) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);      // f16 x f16 -> f32, K-major A and B
            const uint64_t dm = make_desc(0, LBO, SBO_MAIN), dn = make_desc(0, LBO, SBO_MIN);      // descriptors = these + (address >> 4)
            const uint32_t idesc32 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);      // tf32 x tf32 -> f32
            const uint32_t am = smem_u32(amin);
            int slot = 0, bslot = 0, mslot = 0;
            const int G = SPS * nsb;
            for (int g = 0; g < G; g++) {
                const int b = g >> LG_SPS, s = g & (SPS - 1), pr = b & 1;
                TPROF(0, 4 * g);
                if (s == 0 && b >= 2) tc_wait(&S->acc_empty[pr], ((b >> 1) - 1) & 1);
                if (!(p.dbg & 32)) tc_wait(&S->full[g & 15], (g >> 4) & 1);
                TPROF(0, 4 * g + 1);
                tc_fence_after();
                const uint32_t aa = smem_u32(a_ring + (size_t)slot * p.a_slot), bb = smem_u32(b_ring + (size_t)bslot * p.b_slot);
                const uint32_t d_main = tmem + (uint32_t)pr * TN, d_min = tmem + 2 * TN;
                constexpr int NK = KS / 16, NK0 = NK;
                if (elect_one() && !(p.dbg & 2)) {
#pragma unroll
                    for (int ks = 0; ks < NK0; ks++) {
                        const uint64_t bd = dm + ((bb + ks * 2 * LBO) >> 4);
                        mma_f16(d_main, dm + ((aa + ks * 2 * LBO) >> 4), bd, idesc, (s | ks) ? 1u : 0u);
                        if (Q6) mma_f16(d_main, dm + ((aa + MAIN_BYTES + ks * 2 * LBO) >> 4), bd, idesc, 1u);
                    }
                }
                __syncwarp();
                TPROF(0, 4 * g + 2);
                if (elect_one()) {
                    if (!(p.dbg & 2)) {
#pragma unroll
                        for (int ks = NK0; ks < NK; ks++) {
                            const uint64_t bd = dm + ((bb + ks * 2 * LBO) >> 4);
                            mma_f16(d_main, dm + ((aa + ks * 2 * LBO) >> 4), bd, idesc, (s | ks) ? 1u : 0u);
                            if (Q6) mma_f16(d_main, dm + ((aa + MAIN_BYTES + ks * 2 * LBO) >> 4), bd, idesc, 1u);
                        }
                        if (!Q6 && s == 0) {                   // min term, accumulated over ALL super-blocks: hi*u1 + hi*u2 + lo*u1
                            const uint32_t bm = smem_u32(bmin + (size_t)mslot * TN * 64);
                            mma_tf32(d_min, dn + (am >> 4), dn + (bm >> 4), idesc32, b ? 1u : 0u);
                            mma_tf32(d_min, dn + (am >> 4), dn + ((bm + TN * 32) >> 4), idesc32, 1u);
                            mma_tf32(d_min, dn + ((am + MIN_BYTES) >> 4), dn + (bm >> 4), idesc32, 1u);
                        }
                    }
                    tc_commit(&S->empty[g & 15]);              // operand slots free once these MMAs have read them
                    if (s == SPS - 1) tc_commit(&S->acc_full[pr]);   // the super-block's integers are complete
                }
                __syncwarp();
                if (!Q6 && s == 0 && ++mslot == p.nbm) mslot = 0;
                TPROF(0, 4 * g + 3);
                if (++slot == na) slot = 0;
                if (++bslot == nb) bslot = 0;
            }
        }
    } else if (warp < 2 + N_EXP) {
        // ------------------------------------------------------------ expanders: stage raw GGUF blocks (cp.async), write operand tiles
        const int et = threadIdx.x - 64, r = et & (TM - 1), h = et >> 7;
        const uint8_t *const Wt = p.W + (size_t)g_e * p.g_expert_stride + (size_t)row0 * p.rb + (size_t)sb0 * BLK;
        // staging: a thread owns chunks c = et + 256 i of a super-block's TM x CPR 16-byte chunks (consecutive lanes = consecutive chunks of
        // a row piece: whole sectors).  Row pointers and slot offsets are fixed for the launch; only the block offset moves.
        constexpr int NCP = (TM * CPR + N_EXP * 32 - 1) / (N_EXP * 32);
        const uint8_t *cp_row[NCP];
        uint32_t cp_dst[NCP], cp_ch[NCP];
#pragma unroll
        for (int i = 0; i < NCP; i++) {
            const int c = et + i * N_EXP * 32, rr = c / CPR, ch = c % CPR;
            cp_row[i] = Wt + (size_t)(rr < TM ? rr : 0) * p.rb;
            cp_ch[i] = (uint32_t)ch * 16u;
            cp_dst[i] = (uint32_t)rr * p.rstride + (uint32_t)ch * 16u;
        }
        int i_slot = 0, i_use = 0;                     // raw ring position of the next super-block to stage
        auto issue_raw = [&](int b) {
            if (p.dbg & 16) return;
            if (i_use > 0) tc_wait(&S->raw_empty[i_slot], (i_use - 1) & 1);
            const uint32_t slotp = smem_u32(raw) + (uint32_t)i_slot * (TM * p.rstride);
#pragma unroll
            for (int i = 0; i < NCP; i++) {
                if ((i + 1) * N_EXP * 32 <= TM * CPR || et + i * N_EXP * 32 < TM * CPR) {
                    const uint8_t *src = cp_row[i] + (size_t)b * BLK;
                    if (Q6) src -= (uintptr_t)src & 15;    // the piece keeps its 16-byte phase inside the slot row (Q4_K / Q5_K blocks are 16-byte aligned)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(slotp + cp_dst[i]), "l"(src + cp_ch[i]) : "memory");
                }
            }
            asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(&S->raw_full[i_slot])) : "memory");
            if (++i_slot == rs) { i_slot = 0; i_use++; }
        };
        for (int b = 0; b < rs - 1 && b < nsb; b++) issue_raw(b);
        const uint8_t *const myrow = Wt + (size_t)r * p.rb;
        int r_slot = 0, r_use = 0, slot = 0, g = 0;    // raw ring position of super-block b, weight-operand slot of stage g = SPS b + s
        for (int b = 0; b < nsb; b++) {
            if (b + rs - 1 < nsb) issue_raw(b + rs - 1);
            if (!(p.dbg & 16)) tc_wait(&S->raw_full[r_slot], r_use & 1);
            const uint8_t *blk = raw + ((size_t)r_slot * TM + r) * p.rstride + (Q6 ? (uint32_t)((uintptr_t)(myrow + (size_t)b * BLK) & 15) : 0u);
            KHeader kh = {};
            uint32_t qh[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            if (!Q6) {
                kh = read_kheader(blk);
                if (Q5) {
                    const uint4 h0 = *(const uint4 *)(blk + 16), h1 = *(const uint4 *)(blk + 32);
                    qh[0] = h0.x; qh[1] = h0.y; qh[2] = h0.z; qh[3] = h0.w; qh[4] = h1.x; qh[5] = h1.y; qh[6] = h1.z; qh[7] = h1.w;
                }
            }
#pragma unroll 1
            for (int s = 0; s < SPS; s++) {
                if (warp == 2) TPROF(1, 4 * (SPS * b + s));
                if (g >= na) tc_wait(&S->empty[(g - na) & 15], ((g - na) >> 4) & 1);
                if (warp == 2) TPROF(1, 4 * (SPS * b + s) + 1);
                uint8_t *as = a_ring + (size_t)slot * p.a_slot;
                if (p.dbg & 1) {}
                else if (Q6) expand_q6k(blk, s, h, r, as, as + MAIN_BYTES);
                else expand_k45<Q5>(blk, kh, qh, s, h, r, as);
                if (s == 0 && h == 0 && !(p.dbg & 128)) {
                    if (Q6) meta[(b & 3) * TM + r] = make_float2(half_bits_to_float(*(const unsigned short *)(blk + 208)), 0.0f);
                    else { write_min_row(kh, r, amin, amin + MIN_BYTES); meta[(b & 3) * TM + r] = make_float2(kh.d, kh.dmin); }
                }
                if (!(p.dbg & 8)) fence_proxy_async();     // generic-proxy stores -> visible to the tensor core's async proxy
                __syncwarp();
                if (lane == 0) mbar_arrive(&S->full[g & 15]);
                if (warp == 2) TPROF(1, 4 * (SPS * b + s) + 2);
                if (++slot == na) slot = 0;
                g++;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&S->raw_empty[r_slot]);
            if (++r_slot == rs) { r_slot = 0; r_use++; }
        }
    } else {
        // ------------------------------------------------------------ drain: TMEM -> registers, fold the block scales
        const int q = warp & 3, chalf = (warp - 2 - N_EXP) >> 2;          // TMEM lane quarter (fixed by the warp id), column half
        const int r = q * 32 + lane, c_base = chalf * CH;
        float out[CH];
#pragma unroll
        for (int c = 0; c < CH; c++) out[c] = 0.0f;
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        for (int b = 0; b < nsb; b++) {
            const int pr = b & 1;
            if (warp == 2 + N_EXP) TPROF(2, 4 * b);
            tc_wait(&S->acc_full[pr], (b >> 1) & 1);
            if (warp == 2 + N_EXP) TPROF(2, 4 * b + 1);
            tc_fence_after();
            const float2 mt = meta[(b & 3) * TM + r];
            const float4 *da4 = (const float4 *)(p.Bd + (size_t)(sb0 + b) * p.Mpad + tok0 + c_base);
            const uint32_t t_main = tmem + lane_addr + (uint32_t)pr * TN + (uint32_t)c_base;
#pragma unroll
            for (int c0 = 0; c0 < CH; c0 += 16) {
                uint32_t P[16];
                if (!(p.dbg & 64)) {
                    tmem_ld16(t_main + c0, P);
                    tmem_ld_wait();
                } else {
#pragma unroll
                    for (int j = 0; j < 16; j++) P[j] = 0;
                }
                if (c0 == CH - 16) {                       // every accumulator column of this warp is in registers: the tensor core may overwrite the buffer
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&S->acc_empty[pr]);
                    if (warp == 2 + N_EXP) TPROF(2, 4 * b + 2);
                }
                if (p.dbg & 4) continue;
#pragma unroll
                for (int j4 = 0; j4 < 4; j4++) {
                    const float4 d4 = __ldg(da4 + (c0 >> 2) + j4);
                    const float da[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
                    for (int j = 0; j < 4; j++) out[c0 + 4 * j4 + j] = fmaf(da[j] * mt.x, __uint_as_float(P[4 * j4 + j]), out[c0 + 4 * j4 + j]);
                }
            }
        }
        if (!Q6 && !(p.dbg & 64)) {
            // the min term of all super-blocks sits in its own accumulator (the last acc_full covers its MMAs too)
            const uint32_t t_min = tmem + lane_addr + 2 * TN + (uint32_t)c_base;
#pragma unroll
            for (int c0 = 0; c0 < CH; c0 += 16) {
                uint32_t Mn[16];
                tmem_ld16(t_min + c0, Mn);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; j++) out[c0 + j] -= __uint_as_float(Mn[j]);
            }
        }
        if (warp == 2 + N_EXP) TPROF(2, 255);
        float *const dstv = gridDim.z > 1 ? p.part + (size_t)blockIdx.z * p.M * p.N : p.dst;
        const size_t stride = gridDim.z > 1 ? (size_t)p.N : p.dst_stride;
        if (p.g_E) {
#pragma unroll
            for (int c = 0; c < CH; c++) {
                const int tl = c_base + c;
                if (tl < g_cnt) {
                    const int pair = p.g_pairs[g_first + tl];
                    p.dst[(size_t)(pair % p.g_n_used) * p.g_d_nb1 + (size_t)(pair / p.g_n_used) * p.g_d_nb2 + row0 + r] = out[c];
                }
            }
        } else {
#pragma unroll
            for (int c = 0; c < CH; c++) {
                const int tok = tok0 + c_base + c;
                if (tok < p.M) dstv[(size_t)tok * stride + row0 + r] = out[c];
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

// dst[tok][n] = sum over the K slices in slice order (deterministic)
__global__ void __launch_bounds__(256) b200_gemm_tc_reduce_kernel(const float *__restrict__ part, int ksplit, int N, int M, float *__restrict__ dst, size_t dst_stride) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)M * N) return;
    const int tok = (int)(i / N), n = (int)(i % N);
    float a = part[i];
    for (int z = 1; z < ksplit; z++) a += part[(size_t)z * M * N + i];
    dst[(size_t)tok * dst_stride + n] = a;
}

template <int TYPE, int TN>
int launch_tc_t(b200_ctx *ctx, const TcParams &p, dim3 grid, size_t smem) {
    auto kern = b200_gemm_tc_kernel<TYPE, TN>;
    static bool attr_set[16] = {false};
    if (!attr_set[ctx->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->smem_optin));
        attr_set[ctx->device & 15] = true;
    }
    kern<<<grid, TC_THREADS, smem, ctx->stream>>>(p);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return B200_OK;
}
template <int TYPE>
int launch_tc(b200_ctx *ctx, const TcParams &p, int tn, dim3 grid, size_t smem) {
    return tn == 32 ? launch_tc_t<TYPE, 32>(ctx, p, grid, smem) : tn == 64 ? launch_tc_t<TYPE, 64>(ctx, p, grid, smem) : launch_tc_t<TYPE, 128>(ctx, p, grid, smem);
}

}  // namespace

bool gemm_tc_supported(int type, int64_t N, int64_t K, int64_t M) {
    if (type != B200_TYPE_Q4_K && type != B200_TYPE_Q5_K && type != B200_TYPE_Q6_K) return false;
    static const bool off = getenv("GGML_B200_NO_GEMM_TC") != nullptr;
    return !off && N % TM == 0 && K % 256 == 0 && M >= 1;
}

// common host side: activation pack, shared-memory geometry, split-K, launch.  p: W, rb, N, K, M (dense) or the group fields (grouped; M = 0).
static int tc_go(b200_ctx *ctx, int type, TcParams &p, const float *x, size_t x_stride, int tn, int ntile, bool allow_split) {
    const int64_t N = p.N, K = p.K, M = p.M;
    const int Mpad = ntile * tn, nsb = (int)(K / 256);
    const size_t sz_img = (size_t)ntile * nsb * img_bytes(tn);
    uint8_t *scr = (uint8_t *)ctx->get_scratch(SCRATCH_ACT, sz_img + (size_t)nsb * Mpad * 4);
    if (!scr) return B200_ERR_ALLOC;
    p.Mpad = Mpad; p.nsb = nsb; p.img = scr; p.Bd = (const float *)(scr + sz_img);
    {
        const int64_t warps = (int64_t)Mpad * nsb;
        b200_gemm_tc_pack_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, ctx->stream>>>(x, x_stride, (int)K, (int)M, Mpad, nsb, tn, stage_k(type == B200_TYPE_Q6_K), scr, (float *)p.Bd, p);
        ctx->launches++;
        CUDA_TRY(cudaGetLastError());
    }
    const bool q6 = type == B200_TYPE_Q6_K;
    const int ks = stage_k(q6);
    p.a_slot = q6 ? 2 * main_bytes(ks) : main_bytes(ks);
    p.b_slot = (uint32_t)tn * 2u * (uint32_t)ks;
    p.rstride = type == B200_TYPE_Q4_K ? 144u : type == B200_TYPE_Q5_K ? 176u : 240u;        // odd multiples of 16: conflict-free 16-byte row reads
    // shared memory: the weight-operand ring is fed on chip (2-3 stages cover the expander -> MMA hand-off), the raw ring covers HBM latency
    // for 18-30 KB per super-block; everything else goes to the activation ring -- a 16-20 KB bulk copy out of L2 takes ~1.5 us and the
    // stages in flight bound the kernel (profiles/r2_gemm_tc.md)
    const size_t fixed = 4 * TM * sizeof(float2) + sizeof(TcBars) + 1024;
    static const int env_na = getenv("GGML_B200_TC_STAGES") ? atoi(getenv("GGML_B200_TC_STAGES")) : 0;
    static const int env_rs = getenv("GGML_B200_TC_RAW") ? atoi(getenv("GGML_B200_TC_RAW")) : 0;
    static const int env_dbg = getenv("GGML_B200_TC_DBG") ? atoi(getenv("GGML_B200_TC_DBG")) : 0;
    p.dbg = env_dbg;
    const size_t raw_sb = (size_t)TM * p.rstride;
    p.na = env_na >= 2 && env_na <= 4 ? env_na : 2;
    p.rs = env_rs >= 2 && env_rs <= 8 ? env_rs : (tn <= 32 ? 4 : tn <= 64 ? 3 : 2);
    // min-term tiles (Q4_K / Q5_K): one weight-side buffer (the operand ring is one super-block deep: na == stages per super-block) and a ring
    // of activation-side tiles as deep as the activation ring reaches in super-blocks
    const int sps = 256 / ks;
    if (!q6) p.na = sps;
    size_t left = ctx->smem_optin - fixed - (size_t)p.na * p.a_slot - (size_t)p.rs * raw_sb - (q6 ? 0 : 2 * MIN_BYTES);
    p.nb = 0; p.nbm = 0;
    for (int nb = 16; nb >= 2; nb--) {
        const int nbm = q6 ? 0 : (nb + sps - 1) / sps;
        if ((size_t)nb * p.b_slot + (size_t)nbm * tn * 64 <= left) { p.nb = nb; p.nbm = nbm; break; }
    }
    if (p.nb < 2) { b200_set_error("gemm_tc: shared memory"); return B200_ERR_FAILED; }
    const size_t smem = (size_t)p.na * p.a_slot + (size_t)p.nb * p.b_slot + (size_t)p.rs * raw_sb + (q6 ? 0 : 2 * MIN_BYTES + (size_t)p.nbm * tn * 64) +
                        4 * TM * sizeof(float2) + sizeof(TcBars);
    // split K when the (row tile x token tile) grid leaves most of the machine idle; slices of >= min_sb super-blocks, partials reduced in slice order
    static const int max_split = getenv("GGML_B200_TC_KSPLIT") ? atoi(getenv("GGML_B200_TC_KSPLIT")) : 8;
    const int min_sb = tn <= 32 ? 2 : 4;
    const int64_t ctas = (N / TM) * ntile;
    int ksplit = 1;
    while (allow_split && ksplit < max_split && ctas * ksplit * 2 <= ctx->sm_count && nsb / (ksplit * 2) >= min_sb) ksplit *= 2;
    p.sb_per_split = (nsb + ksplit - 1) / ksplit;
    ksplit = (nsb + p.sb_per_split - 1) / p.sb_per_split;
    if (ksplit > 1) {
        p.part = (float *)ctx->get_scratch(SCRATCH_MISC, (size_t)ksplit * M * N * 4);
        if (!p.part) return B200_ERR_ALLOC;
    }
    const dim3 grid((unsigned)(N / TM), (unsigned)ntile, (unsigned)ksplit);
    static const int env_prof = getenv("GGML_B200_TC_PROF") ? atoi(getenv("GGML_B200_TC_PROF")) : 0;
    static unsigned long long *prof_buf = nullptr;
    static int prof_left = 2;
    if (env_prof && prof_left > 0) {
        if (!prof_buf) cudaMalloc(&prof_buf, 3 * 256 * 8);
        cudaMemsetAsync(prof_buf, 0, 3 * 256 * 8, ctx->stream);
        p.prof = prof_buf;
    }
    int rc;
    switch (type) {
        case B200_TYPE_Q4_K: rc = launch_tc<B200_TYPE_Q4_K>(ctx, p, tn, grid, smem); break;
        case B200_TYPE_Q5_K: rc = launch_tc<B200_TYPE_Q5_K>(ctx, p, tn, grid, smem); break;
        default:             rc = launch_tc<B200_TYPE_Q6_K>(ctx, p, tn, grid, smem); break;
    }
    if (p.prof) {
        static unsigned long long hp[3 * 256];
        cudaStreamSynchronize(ctx->stream);
        cudaMemcpy(hp, prof_buf, sizeof(hp), cudaMemcpyDeviceToHost);
        unsigned long long t0 = ~0ull;
        for (int i = 0; i < 3 * 256; i++) if (hp[i] && hp[i] < t0) t0 = hp[i];
        fprintf(stderr, "gemm_tc timeline (clk after first stamp) type %d N %d K %d M %d tn %d na %d nb %d rs %d ksplit %d\n", type, (int)N, (int)K, (int)M, tn, p.na, p.nb, p.rs, ksplit);
        for (int g = 0; g < 64 && hp[4 * g]; g++) {
            fprintf(stderr, " g%2d mma: top %6lld a_full %6lld b_full %6lld issued %6lld | exp: top %6lld a_empty %6lld arrived %6lld", g, (long long)(hp[4 * g] - t0),
                    (long long)(hp[4 * g + 1] - t0), (long long)(hp[4 * g + 2] - t0), (long long)(hp[4 * g + 3] - t0), (long long)(hp[256 + 4 * g] - t0),
                    (long long)(hp[256 + 4 * g + 1] - t0), (long long)(hp[256 + 4 * g + 2] - t0));
            const int sps = 256 / ks;
            if (g % sps == sps - 1) {
                const int sb = g / sps;
                fprintf(stderr, " | drain sb%d: top %6lld acc_full %6lld loaded %6lld", sb, (long long)(hp[512 + 4 * sb] - t0), (long long)(hp[512 + 4 * sb + 1] - t0), (long long)(hp[512 + 4 * sb + 2] - t0));
            }
            fprintf(stderr, "\n");
        }
        fprintf(stderr, " drain done %lld\n", (long long)(hp[512 + 255] - t0));
        prof_left--;
    }
    if (rc || ksplit == 1) return rc;
    const int64_t total = M * N;
    b200_gemm_tc_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(p.part, ksplit, (int)N, (int)M, p.dst, p.dst_stride);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return B200_OK;
}

// dst[tok * dst_stride + n] = sum_k W[n, k] * x[k, tok]; x f32 with column stride x_stride bytes
int gemm_tc_run(b200_ctx *ctx, int type, const uint8_t *W, size_t rb, int64_t N, int64_t K, const float *x, size_t x_stride, int64_t M,
                float *dst, size_t dst_stride) {
    if (!gemm_tc_supported(type, N, K, M) || (type != B200_TYPE_Q6_K && (((uintptr_t)W | rb) & 15)) || ((uintptr_t)W & 1)) {
        b200_set_error("gemm_tc: unsupported shape");
        return B200_ERR_UNSUPPORTED;
    }
    const int tn = M <= 32 ? 32 : M <= 64 ? 64 : 128;
    TcParams p = {};
    p.W = W; p.rb = (uint32_t)rb; p.N = (int)N; p.K = (int)K; p.M = (int)M; p.dst = dst; p.dst_stride = dst_stride;
    return tc_go(ctx, type, p, x, x_stride, tn, (int)((M + tn - 1) / tn), true);
}

// MUL_MAT_ID for prompt batches: the (token, slot) pairs counting-sorted by expert on the device (mulmat.cu) become token tiles of <= 128 pairs
// per expert; every tile runs the same GEMM against its expert's matrix.  g.max_chunks: upper bound of sum_e ceil(count_e / 128).
int gemm_tc_run_grouped(b200_ctx *ctx, int type, const uint8_t *W, size_t rb, int64_t N, int64_t K, const float *x, size_t x_stride, const MmGroupDesc &g, float *dst) {
    if (!gemm_tc_supported(type, N, K, 128) || (type != B200_TYPE_Q6_K && (((uintptr_t)W | rb | g.expert_stride) & 15)) || (((uintptr_t)W | g.expert_stride) & 1)) {
        b200_set_error("gemm_tc: unsupported shape");
        return B200_ERR_UNSUPPORTED;
    }
    TcParams p = {};
    p.W = W; p.rb = (uint32_t)rb; p.N = (int)N; p.K = (int)K; p.M = 0; p.dst = dst;
    p.g_off = g.off; p.g_pairs = g.pairs; p.g_E = g.E; p.g_n_used = g.n_used; p.g_b_ne1 = g.b_ne1;
    p.g_expert_stride = g.expert_stride; p.g_d_nb1 = g.d_nb1; p.g_d_nb2 = g.d_nb2;
    return tc_go(ctx, type, p, x, x_stride, 128, g.max_chunks, false);
}
