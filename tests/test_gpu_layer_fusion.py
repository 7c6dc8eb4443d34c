"""The decode layer fusions of graph.cu fuse() held block by block against the oracle, at TinyLlama, Llama-3-8B and 70B shapes.

Each test builds the op list of one block the way llama_graph.build (= llama.cpp's graph) emits it, runs it at fusion 0, 1 and 2 and
checks every output the block makes observable:
- matmul + residual outputs: |got - (mm_ref + resid)| <= 3e-6 * max|mm_ref| (+ flips, see below) + 1 ulp of the sum; the bound is
  relative to the matmul term, so a large residual cannot hide an error;
- the FFN's down output: fusion_ref.flip_bound over h = silu(gate) * up, the intermediate the fused path never writes;
- the KV-cache rows at kv_head: fusion_ref.kv_bytes_ok; every other cell byte-identical to before the call;
- the roped q written for flash attention, against orc_rope of the reference q;
- the flash-attention output against exact_attention over the GPU's own cache bytes and roped q (NMSE <= 1e-10).
Intermediates normalised on the device (rms_norm(x) * w) are quantised like the reference's; their values agree to a few ulp, so the
activation rounding of an element within 3e-7 * |x_k| of a tie may flip: flip_bound admits exactly that.

Fusion 2 must launch fewer kernels than fusion 1 where the block fuses and the same number where it must decline (the liveness
cases at the end), and two fusion-2 runs must be bit-identical."""
import ctypes as C
import math

import numpy as np
import pytest

import fusion_ref as FR
import reflib as R
from test_gpu_fattn import exact_attention
from util import nmse, rand_quant_rows

pytestmark = pytest.mark.gpu

EPS = 1e-5
NORM_EPS = 3e-7                # relative difference of a device-normalised element (a few ulp of the two rounded multiplies)
MIX = "q4_k_m"                 # llama-quant's Q4_K_M: wv and down in Q6_K, the rest Q4_K
FORMATS = [R.Q4_K, R.Q5_K, R.Q6_K, R.Q4_0, R.Q8_0, MIX]


def wtype(fmt, role):
    if fmt == MIX:
        return R.Q6_K if role in ("v", "down") else R.Q4_K
    return fmt


def fname(fmt):
    return fmt if isinstance(fmt, str) else R.TYPE_NAMES[fmt]


@pytest.fixture
def opts(ctx):
    """every option these tests set, restored for the rest of the session"""
    ctx.set_option("pdl", 0); ctx.set_option("cuda_graphs", 0); ctx.set_option("ffn_pair", 1)
    try:
        yield ctx
    finally:
        ctx.set_option("fusion", 2); ctx.set_option("ffn_pair", 1); ctx.set_option("pdl", 0); ctx.set_option("cuda_graphs", 0)


class Dev:
    """device buffers (torch) with host views and b200 tensor descriptors"""

    def __init__(self, b200):
        import torch
        self.torch, self.b200, self.keep = torch, b200, []

    def f32(self, n, fill=np.nan):
        t = self.torch.full((int(n),), float(fill), dtype=self.torch.float32, device="cuda")
        self.keep.append(t)
        return t

    def put(self, arr):
        t = self.torch.from_numpy(np.ascontiguousarray(arr)).cuda()
        self.keep.append(t)
        return t

    def weight(self, t, N, K, rng):
        W = rand_quant_rows(t, N, K, rng)
        pad = self.b200.lib().b200_alloc_size(t, (C.c_int64 * 4)(K, N, 1, 1), W.size)
        d = self.torch.zeros(int(pad), dtype=self.torch.uint8, device="cuda")
        d[:W.size] = self.torch.from_numpy(W).cuda()
        self.keep.append(d)
        return W, self.b200.tensor(d.data_ptr(), t, [K, N], flags=self.b200.TENSOR_FLAG_WEIGHT)

    def t(self, buf, ne, off=0, type_=None, nb=None):
        return self.b200.tensor(buf.data_ptr() + off, self.b200.F32 if type_ is None else type_, ne, nb)


def act_columns(rng, T, E):
    """decode activations with the edges a norm prologue must get right, cycling over the columns: mean square comparable to eps
    (eps matters), ordinary, all zero, 1e3 dynamic range"""
    x = rng.standard_normal((T, E)).astype(np.float32)
    for c in range(T):
        kind = c % 4
        if kind == 0:
            x[c] *= math.sqrt(2 * EPS)
        elif kind == 2:
            x[c] = 0
        elif kind == 3:
            x[c] *= 10.0 ** rng.uniform(-1.5, 1.5, E)
    return x.astype(np.float32)


def sample_rows(rng, N):
    return np.unique(np.concatenate([np.arange(min(N, 16)), rng.integers(0, N, 24), np.arange(max(0, N - 8), N)]))


def run(ctx, ops, fusion, n_rep=1):
    ctx.set_option("fusion", fusion)
    n0 = ctx.launches()
    for _ in range(n_rep):
        ctx.compute(ops)
    ctx.sync()
    return (ctx.launches() - n0) // n_rep


def check_resid_out(got, mm_ref, resid, flip=0.0, what=""):
    """got, mm_ref, resid [T, n]; flip [T, n] or scalar: the extra tolerance of activation flips"""
    want = mm_ref.astype(np.float64) + resid.astype(np.float64)
    ulp = np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)
    tol = FR.REL * max(float(np.abs(mm_ref).max()), 1e-30) + flip + ulp
    err = np.abs(got.astype(np.float64) - want)
    assert np.isfinite(got).all(), what
    assert (err <= tol).all(), (what, float((err - tol).max()), np.unravel_index(int(np.argmax(err - tol)), err.shape))


def norm_stage(rng, T, E):
    x = act_columns(rng, T, E)
    nw = (1.0 + 0.02 * rng.standard_normal(E)).astype(np.float32)
    return x, nw, FR.norm_mul(x, nw, EPS)


# ----------------------------------------------------------------------------------------------------------- attention block
# (E, H, Hkv, D, rope base)
# flash attention takes quantised caches at head size 128 only: TinyLlama (D 64) runs over an f16 cache, the quantised caches are
# exercised at the D-128 layout of mid-d128 and Llama-3-8B
TINY_ATT = (2048, 32, 4, 64, 10000.0)
MID_ATT = (2048, 16, 4, 128, 10000.0)
L8B_ATT = (4096, 32, 8, 128, 500000.0)
KVS = [R.F16, R.Q8_0, R.Q4_0]
ATT_CASES = ([(TINY_ATT, f, T, R.F16, (i + j) % 2 == 1) for i, f in enumerate(FORMATS) for j, T in enumerate([1, 4, 17])] +
             [(MID_ATT, f, T, KVS[1 + (i + j) % 2], (i + j) % 2 == 0) for i, f in enumerate(FORMATS) for j, T in enumerate([1, 4, 17])] +
             [(MID_ATT, R.Q4_K, T, R.Q8_0, True) for T in (2, 3)] +
             [(L8B_ATT, f, T, KVS[j], j == 1) for f in (MIX, R.Q8_0) for j, T in enumerate([1, 5, 32])])


def att_id(c):
    return "E%d-D%d-%s-T%d-kv%s-%s" % (c[0][0], c[0][3], fname(c[1]), c[2], R.TYPE_NAMES[c[3]], "mask_in" if c[4] else "mask_before")


class AttBlock:
    """NORM MUL {MMq MMk MMv ROPEq ROPEk CPYk CPYv} FA over a cache of n_kv cells with the new rows at kv_head"""

    def __init__(self, b200, dev, rng, shape, fmt, T, kvt, mask_inside, extra_reader=False):
        E, H, Hkv, D, base = shape
        self.dev = dev                      # owns every device buffer the op list points at
        self.E, self.H, self.Hkv, self.D, self.T, self.kvt = E, H, Hkv, D, T, kvt
        self.kv_head, self.n_kv = 100 + T, 256
        t, F32 = dev.t, b200.F32
        self.x, self.nw, self.xn = norm_stage(rng, T, E)
        self.W = {}
        wt = {}
        for role, n in (("q", H * D), ("k", Hkv * D), ("v", Hkv * D)):
            self.W[role], wt[role] = dev.weight(wtype(fmt, role), n, E, rng)
        self.types = {r: wtype(fmt, r) for r in "qkv"}
        self.pos = np.arange(self.kv_head, self.kv_head + T, dtype=np.int32)
        Tp = (T + 63) // 64 * 64
        mask = np.full((Tp, self.n_kv), -np.inf, np.float32)
        for i in range(T):
            mask[i, :self.kv_head + i + 1] = 0
        self.mask16 = mask.astype(np.float16)
        self.rs_head, self.rs_row = R.row_size(kvt, D), R.row_size(kvt, Hkv * D)
        cells = rng.standard_normal((2, self.n_kv * Hkv, D)).astype(np.float32)
        self.cache0 = [cells[i].astype(np.float16).view(np.uint8).reshape(-1) if kvt == R.F16 else R.orc_quantize_act(kvt, cells[i]).reshape(-1)
                       for i in range(2)]
        xd, nwd = dev.put(self.x), dev.put(self.nw)
        self.kc, self.vc = dev.put(self.cache0[0]), dev.put(self.cache0[1])
        posd, m32, self.m16 = dev.put(self.pos), dev.put(mask), dev.f32(mask.size // 2, 0)
        cur, cur2 = dev.f32(E * T), dev.f32(E * T)
        q, k, v = dev.f32(H * D * T), dev.f32(Hkv * D * T), dev.f32(Hkv * D * T)
        self.qr, kr, self.att = dev.f32(H * D * T), dev.f32(Hkv * D * T), dev.f32(H * D * T)
        mk = b200.make_op
        rope_params = [0, D, 0, 0, 8192, float(base), 1.0, 0.0, 1.0, 32.0, 1.0]
        self.base = base
        mask_cpy = mk(b200.OP_CPY, t(self.m16, [self.n_kv, Tp], type_=b200.F16), [t(m32, [self.n_kv, Tp])])
        B = t(cur2, [E, T])
        ops = [] if mask_inside else [mask_cpy]
        ops += [mk(b200.OP_RMS_NORM, t(cur, [E, T]), [t(xd, [E, T])], [EPS]),
                mk(b200.OP_MUL, B, [t(cur, [E, T]), b200.tensor(nwd.data_ptr(), F32, [E], flags=b200.TENSOR_FLAG_WEIGHT)]),
                mk(b200.OP_MUL_MAT, t(q, [H * D, T]), [wt["q"], B]),
                mk(b200.OP_MUL_MAT, t(k, [Hkv * D, T]), [wt["k"], B]),
                mk(b200.OP_MUL_MAT, t(v, [Hkv * D, T]), [wt["v"], B])]
        post = t(posd, [T], type_=b200.I32)
        ops += [mk(b200.OP_ROPE, t(self.qr, [D, H, T]), [t(q, [D, H, T]), post, None], rope_params),
                mk(b200.OP_ROPE, t(kr, [D, Hkv, T]), [t(k, [D, Hkv, T]), post, None], rope_params)]
        off = self.rs_row * self.kv_head
        ops += [mk(b200.OP_CPY, t(self.kc, [Hkv * D * T], off, kvt), [t(kr, [D, Hkv, T])]),
                mk(b200.OP_CPY, t(self.vc, [Hkv * D * T], off, kvt), [t(v, [Hkv * D, T])])]
        if mask_inside:                     # llama.cpp schedules the conversion right before its first consumer
            ops.append(mask_cpy)
        bk = R.BLOCK[kvt][1]
        qv = t(self.qr, [D, T, H], nb=[4, D * H * 4, D * 4, D * H * T * 4])
        kvv = [t(c, [D, self.n_kv, Hkv], type_=kvt, nb=[bk, self.rs_row, self.rs_head, self.rs_row * self.n_kv]) for c in (self.kc, self.vc)]
        ops.append(mk(b200.OP_FLASH_ATTN_EXT, t(self.att, [D, H, T]), [qv, kvv[0], kvv[1], t(self.m16, [self.n_kv, Tp], type_=b200.F16)],
                      [1.0 / math.sqrt(D), 0.0, 0.0]))
        if extra_reader:                    # a parallel attention + FFN block reads the normed x again after FA
            self.probe = dev.f32(E * T)
            ops.append(mk(b200.OP_ADD, t(self.probe, [E, T]), [B, B]))
        self.ops = ops

    def reset(self):
        self.kc.copy_(self.torch_put(self.cache0[0])); self.vc.copy_(self.torch_put(self.cache0[1]))
        self.qr.fill_(float("nan")); self.att.fill_(float("nan"))

    def reference(self):
        E, H, Hkv, D, T = self.E, self.H, self.Hkv, self.D, self.T
        out = {}
        for r in "qkv":
            Wd = FR.dequant_rows(self.types[r], self.W[r], E)
            xa, _ = FR.quant_act(self.types[r], self.xn)
            mm = xa @ Wd.T
            flip = FR.flip_bound(self.xn, self.types[r], Wd, NORM_EPS, scale=0.0, per_element=True)
            out[r] = (mm, flip.max(1))
        self.q_ref, self.k_ref, self.v_ref = out["q"][0], out["k"][0], out["v"][0]
        self.flip = {r: out[r][1] for r in "qkv"}
        rope = lambda a, n: R.orc_rope(a.astype(np.float32).reshape(T, n, D), self.pos, D, 0, self.base)   # noqa: E731
        self.qr_ref, self.kr_ref = rope(self.q_ref, H), rope(self.k_ref, Hkv)

    def check(self, what):
        T, H, Hkv, D, kvt = self.T, self.H, self.Hkv, self.D, self.kvt
        qr = self.qr.cpu().numpy().reshape(T, H, D)
        # a rotation mixes the errors of a pair: |e0| + |e1| per output element
        tol_q = 2 * (FR.REL * np.abs(self.q_ref).max(1) + self.flip["q"]) + 1e-30
        err_q = np.abs(qr - self.qr_ref).reshape(T, -1).max(1)
        assert np.isfinite(qr).all() and (err_q <= tol_q).all(), (what, "roped q", err_q / np.maximum(tol_q, 1e-30))
        caches = []
        for c, c0, xr, r in ((self.kc, self.cache0[0], self.kr_ref, "k"), (self.vc, self.cache0[1], self.v_ref, "v")):
            got = c.cpu().numpy()
            lo, hi = self.rs_row * self.kv_head, self.rs_row * (self.kv_head + T)
            assert np.array_equal(got[:lo], c0[:lo]) and np.array_equal(got[hi:], c0[hi:]), (what, r, "cells outside the new rows changed")
            xt = np.asarray(xr, np.float64).reshape(T, Hkv * D)
            delta = 2 * (FR.REL * np.abs(xt).max(1) + self.flip[r])
            ok = FR.kv_bytes_ok(got[lo:hi].reshape(T * Hkv, self.rs_head), xt.reshape(T * Hkv, D), kvt, np.repeat(delta, Hkv))
            assert ok.all(), (what, r, "cache rows", int((~ok).sum()))
            caches.append(got.reshape(self.n_kv, Hkv, self.rs_head).transpose(1, 0, 2).copy())
        att = self.att.cpu().numpy().reshape(T, H, D)
        exact = exact_attention(qr.transpose(1, 0, 2).copy(), caches[0], caches[1], self.mask16, D, self.n_kv, Hkv, kvt, 1.0 / math.sqrt(D))
        assert np.isfinite(att).all() and nmse(att, exact) <= 1e-10, (what, nmse(att, exact))
        return qr, att, caches

    def torch_put(self, arr):
        import torch
        return torch.from_numpy(arr).cuda()


@pytest.mark.parametrize("case", ATT_CASES, ids=att_id)
def test_attention_block(b200, opts, case):
    ctx = opts
    shape, fmt, T, kvt, mask_inside = case
    rng = np.random.default_rng(1000 + 7 * T + shape[0] + kvt + (0 if isinstance(fmt, str) else fmt))
    blk = AttBlock(b200, Dev(b200), rng, shape, fmt, T, kvt, mask_inside)
    blk.reference()
    launches, outs = {}, {}
    for fusion in (0, 1, 2):
        blk.reset()
        launches[fusion] = run(ctx, blk.ops, fusion)
        outs[fusion] = blk.check("fusion %d" % fusion)
    assert launches[2] < launches[1], launches
    blk.reset()
    run(ctx, blk.ops, 2)
    again = blk.check("fusion 2, again")
    for a, b in zip(outs[2], again):
        assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8)), "fusion 2 is not deterministic"


# ----------------------------------------------------------------------------------------------------------------- FFN block
class FfnBlock:
    """NORM MUL {MMup MMgate SILU MUL MMdown} ADD(down, ffn_inp)"""

    def __init__(self, b200, dev, rng, E, FF, fmt, T):
        self.E, self.FF, self.T = E, FF, T
        self.dev = dev
        t = dev.t
        self.x, self.nw, self.xn = norm_stage(rng, T, E)
        self.types = {r: wtype(fmt, r) for r in ("gate", "up", "down")}
        self.W, wt = {}, {}
        for role, N, K in (("gate", FF, E), ("up", FF, E), ("down", E, FF)):
            self.W[role], wt[role] = dev.weight(self.types[role], N, K, rng)
        xd, nwd = dev.put(self.x), dev.put(self.nw)
        cur, cur2, g, u, gu, tmp = dev.f32(E * T), dev.f32(E * T), dev.f32(FF * T), dev.f32(FF * T), dev.f32(FF * T), dev.f32(E * T)
        self.g = g
        self.out = dev.f32(E * T)
        mk = b200.make_op
        B = t(cur2, [E, T])
        self.ops = [mk(b200.OP_RMS_NORM, t(cur, [E, T]), [t(xd, [E, T])], [EPS]),
                    mk(b200.OP_MUL, B, [t(cur, [E, T]), b200.tensor(nwd.data_ptr(), b200.F32, [E], flags=b200.TENSOR_FLAG_WEIGHT)]),
                    mk(b200.OP_MUL_MAT, t(u, [FF, T]), [wt["up"], B]),
                    mk(b200.OP_MUL_MAT, t(g, [FF, T]), [wt["gate"], B]),
                    mk(b200.OP_SILU, t(gu, [FF, T]), [t(g, [FF, T])]),
                    mk(b200.OP_MUL, t(gu, [FF, T]), [t(gu, [FF, T]), t(u, [FF, T])]),
                    mk(b200.OP_MUL_MAT, t(tmp, [E, T]), [wt["down"], t(gu, [FF, T])]),
                    mk(b200.OP_ADD, t(self.out, [E, T]), [t(tmp, [E, T]), t(xd, [E, T])])]

    def reference(self, rng):
        g = FR.mm_f64(self.types["gate"], self.W["gate"], self.xn, self.E).astype(np.float32)
        u = FR.mm_f64(self.types["up"], self.W["up"], self.xn, self.E).astype(np.float32)
        self.h = R.orc_silu_mul(g, u)
        self.rows = sample_rows(rng, self.E)
        td = self.types["down"]
        rb = R.row_size(td, self.FF)
        Wsub = self.W["down"].reshape(self.E, rb)[self.rows].reshape(-1)
        self.mm_ref = R.orc_mul_mat(td, Wsub, self.h, len(self.rows), self.FF)
        Wd = FR.dequant_rows(td, Wsub, self.FF)
        # the device's h differs from h_ref by the summation order of gate and up (the GEMV's 3e-6 bound)
        self.flip = FR.flip_bound(self.h, td, Wd, FR.REL, scale=0.0)

    def check(self, what):
        got = self.out.cpu().numpy().reshape(self.T, self.E)
        check_resid_out(got[:, self.rows], self.mm_ref, self.x[:, self.rows], self.flip, what)
        return got


L8B_FFN, L70B_FFN, TINY_FFN = (4096, 14336), (8192, 28672), (2048, 5632)
FFN_CASES = ([(TINY_FFN, f, [1, 4, 17]) for f in FORMATS] + [(TINY_FFN, R.Q4_K, [2, 3, 5, 32])] +
             [(s, f, [1, 5, 32]) for s in (L8B_FFN, L70B_FFN) for f in (MIX, R.Q8_0)])


@pytest.mark.parametrize("shape,fmt,Ts", FFN_CASES, ids=["E%d-FF%d-%s-T%s" % (c[0][0], c[0][1], fname(c[1]), "_".join(map(str, c[2]))) for c in FFN_CASES])
def test_ffn_block(b200, opts, shape, fmt, Ts):
    """the fused gate|up GEMV (norm prologue; pair epilogue at T = 1) and the down GEMV (swiglu prologue, residual epilogue);
    at T = 1 the ffn_pair options 0 and 1 must agree bit for bit (at FF >= 8192 option 0 takes the 4-CTA cluster swiglu prologue)"""
    ctx = opts
    E, FF = shape
    for T in Ts:
        rng = np.random.default_rng(2000 + T + E + (0 if isinstance(fmt, str) else fmt))
        blk = FfnBlock(b200, Dev(b200), rng, E, FF, fmt, T)
        blk.reference(rng)
        launches, outs = {}, {}
        for fusion in (0, 1, 2):
            blk.out.fill_(float("nan"))
            launches[fusion] = run(ctx, blk.ops, fusion)
            outs[fusion] = blk.check("T %d fusion %d" % (T, fusion))
        assert launches[2] < launches[1], (T, launches)
        run(ctx, blk.ops, 2)
        assert np.array_equal(outs[2], blk.check("T %d again" % T)), "fusion 2 is not deterministic"
        if T == 1:
            ctx.set_option("ffn_pair", 0)
            run(ctx, blk.ops, 2)
            ctx.set_option("ffn_pair", 1)
            assert np.array_equal(outs[2], blk.check("ffn_pair 0")), "ffn_pair 0 and 1 differ"


# ----------------------------------------------------------------------------------------------------- wo + residual (mm_add)
MM_ADD_CASES = ([(2048, 2048, f, [1, 4, 17]) for f in FORMATS] + [(4096, 4096, f, [1, 5, 32]) for f in (R.Q4_K, R.Q8_0)] +
                [(4096, 4100, f, [7]) for f in (R.Q4_K, R.Q6_K, R.Q8_0)])     # N % 16 != 0: gemv.cu in chunks of 4 columns


@pytest.mark.parametrize("K,N,fmt,Ts", MM_ADD_CASES, ids=["K%d-N%d-%s-T%s" % (c[0], c[1], fname(c[2]), "_".join(map(str, c[3]))) for c in MM_ADD_CASES])
def test_mm_add_block(b200, opts, K, N, fmt, Ts):
    ctx = opts
    for T in Ts:
        rng = np.random.default_rng(3000 + T + K + N)
        dev = Dev(b200)
        t = wtype(fmt, "o")
        W, wt = dev.weight(t, N, K, rng)
        a = rng.standard_normal((T, K)).astype(np.float32)
        resid = (rng.standard_normal((T, N)) * 30).astype(np.float32)
        ad, rd, tmp, out = dev.put(a), dev.put(resid), dev.f32(N * T), dev.f32(N * T)
        ops = [b200.make_op(b200.OP_MUL_MAT, dev.t(tmp, [N, T]), [wt, dev.t(ad, [K, T])]),
               b200.make_op(b200.OP_ADD, dev.t(out, [N, T]), [dev.t(tmp, [N, T]), dev.t(rd, [N, T])])]
        rows = sample_rows(rng, N)
        rb = R.row_size(t, K)
        mm_ref = R.orc_mul_mat(t, W.reshape(N, rb)[rows].reshape(-1), a, len(rows), K)
        launches, outs = {}, {}
        for fusion in (0, 1, 2):
            out.fill_(float("nan"))
            launches[fusion] = run(ctx, ops, fusion)
            outs[fusion] = out.cpu().numpy().reshape(T, N)
            check_resid_out(outs[fusion][:, rows], mm_ref, resid[:, rows], 0.0, "T %d fusion %d" % (T, fusion))
        assert launches[2] < launches[1], (T, launches)
        run(ctx, ops, 2)
        assert np.array_equal(outs[2], out.cpu().numpy().reshape(T, N))


# ------------------------------------------------------------------------------------------ final norm + output projection
NORM_MM_CASES = ([(16384, 512, f, [1, 4]) for f in (R.Q4_K, R.Q6_K, R.Q8_0)] +         # K > 15872: the streaming norm prologue
                 [(4096, 32000, f, [1, 4, 17]) for f in (R.Q6_K, R.Q4_0)] + [(4096, 32003, R.Q6_K, [1, 7, 17])])


@pytest.mark.parametrize("K,N,fmt,Ts", NORM_MM_CASES, ids=["K%d-N%d-%s-T%s" % (c[0], c[1], fname(c[2]), "_".join(map(str, c[3]))) for c in NORM_MM_CASES])
def test_norm_mm_block(b200, opts, K, N, fmt, Ts):
    ctx = opts
    for T in Ts:
        rng = np.random.default_rng(4000 + T + K + N)
        dev = Dev(b200)
        W, wt = dev.weight(fmt, N, K, rng)
        x, nw, xn = norm_stage(rng, T, K)
        xd, nwd, cur, cur2, out = dev.put(x), dev.put(nw), dev.f32(K * T), dev.f32(K * T), dev.f32(N * T)
        ops = [b200.make_op(b200.OP_RMS_NORM, dev.t(cur, [K, T]), [dev.t(xd, [K, T])], [EPS]),
               b200.make_op(b200.OP_MUL, dev.t(cur2, [K, T]), [dev.t(cur, [K, T]), b200.tensor(nwd.data_ptr(), b200.F32, [K], flags=1)]),
               b200.make_op(b200.OP_MUL_MAT, dev.t(out, [N, T]), [wt, dev.t(cur2, [K, T])])]
        rows = sample_rows(rng, N)
        Wsub = W.reshape(N, R.row_size(fmt, K))[rows].reshape(-1)
        mm_ref = R.orc_mul_mat(fmt, Wsub, xn, len(rows), K)
        flip = FR.flip_bound(xn, fmt, FR.dequant_rows(fmt, Wsub, K), NORM_EPS, scale=0.0, per_element=True)
        launches, outs = {}, {}
        for fusion in (0, 1, 2):
            out.fill_(float("nan"))
            launches[fusion] = run(ctx, ops, fusion)
            outs[fusion] = out.cpu().numpy().reshape(T, N)
            check_resid_out(outs[fusion][:, rows], mm_ref, np.zeros_like(mm_ref), flip, "T %d fusion %d" % (T, fusion))
        assert launches[2] < launches[1], (T, launches)


# ------------------------------------------------------------------------------------------------- liveness and declines
def test_decline_normed_x_read_after_fa(b200, opts):
    """a parallel attention + FFN block reads the normed x after FA: no attention fusion, the unfused answer"""
    ctx = opts
    rng = np.random.default_rng(5)
    blk = AttBlock(b200, Dev(b200), rng, MID_ATT, R.Q4_K, 2, R.Q8_0, False, extra_reader=True)
    blk.reference()
    res = {}
    for fusion in (1, 2):
        blk.reset(); blk.probe.fill_(float("nan"))
        n = run(ctx, blk.ops, fusion)
        res[fusion] = (n, blk.check("fusion %d" % fusion), blk.probe.cpu().numpy().reshape(2, -1).copy())
    assert res[1][0] == res[2][0], "must decline"
    assert np.array_equal(res[1][2], res[2][2])
    assert np.abs(res[2][2] - 2 * blk.xn).max() <= 2 * NORM_EPS * np.abs(blk.xn).max()


def _mm_add_ops(b200, dev, rng, K, N, T, t=R.Q4_K, layout="plain"):
    """MUL_MAT(mm = W a) ADD(dst = mm + resid) + optional reader; returns ops, outputs to compare and the device buffers"""
    W, wt = dev.weight(t, N, K, rng)
    a = rng.standard_normal((T, K)).astype(np.float32)
    resid = rng.standard_normal((T, N)).astype(np.float32)
    ad, rd = dev.put(a), dev.put(resid)
    mk, tt = b200.make_op, dev.t
    mmbuf = dev.f32(N * (T + 1), 0)
    mm, dst, extra = tt(mmbuf, [N, T]), None, []
    if layout == "wo_read_after_add":               # the wo output is read again after its ADD
        outb = dev.f32(N * T); dst = tt(outb, [N, T]); probe = dev.f32(N * T)
        extra = [mk(b200.OP_ADD, tt(probe, [N, T]), [mm, mm])]
        watch = [outb, probe]
    elif layout == "dst_overlaps_x":                # ADD writes over the matmul's x
        dst = tt(ad, [N, T]); watch = [ad]
        assert N == K
    elif layout == "inplace_resid":                 # add.dst == residual: must still fuse
        dst = tt(rd, [N, T]); watch = [rd]
    elif layout == "dst_one_column_on":             # add.dst = mm.dst shifted by one column; mm's first column read later
        # (ADD's column 1 reads what its column 0 writes: only the columns no write races with are compared)
        dst = tt(mmbuf, [N, T], off=N * 4); probe = dev.f32(N)
        extra = [mk(b200.OP_ADD, tt(probe, [N]), [tt(mmbuf, [N]), tt(mmbuf, [N])])]
        watch = [mmbuf[:2 * N], probe]
    ops = [mk(b200.OP_MUL_MAT, mm, [wt, tt(ad, [K, T])]), mk(b200.OP_ADD, dst, [mm, tt(rd, [N, T])])] + extra
    state = [(b, b.clone()) for b in (ad, rd, mmbuf)]
    return ops, watch, state, (W, a, resid)


@pytest.mark.parametrize("layout,fuses", [("wo_read_after_add", False), ("dst_overlaps_x", False), ("inplace_resid", True),
                                          ("dst_one_column_on", False)])
def test_mm_add_liveness(b200, opts, layout, fuses):
    """the unfused answer whatever the layout; fused only where no later op needs the matmul's own output"""
    ctx = opts
    K = N = 2048
    T = 2
    rng = np.random.default_rng(6)
    dev = Dev(b200)
    ops, watch, state, (W, a, resid) = _mm_add_ops(b200, dev, rng, K, N, T, layout=layout)
    res = {}
    for fusion in (1, 2):
        for b, b0 in state:
            b.copy_(b0)
        n = run(ctx, ops, fusion)
        res[fusion] = (n, [w.cpu().numpy().copy() for w in watch])
    assert (res[2][0] < res[1][0]) == fuses, (layout, res[1][0], res[2][0])
    for g1, g2 in zip(res[1][1], res[2][1]):
        if fuses:
            mm_ref = R.orc_mul_mat(R.Q4_K, W, a, N, K)
            check_resid_out(g2.reshape(T, N), mm_ref, resid, 0.0, layout)
        else:
            assert np.array_equal(g1, g2), layout


def test_ffn_dst_inside_gate_buffer(b200, opts):
    """ADD's destination starts inside gate's [FF, T] buffer and a later op reads gate's head: the gate values must be there, as in
    op-by-op execution (only a destination that covers an intermediate makes it dead)"""
    import torch
    ctx = opts
    E, FF, T = 2048, 5632, 1
    rng = np.random.default_rng(8)
    dev = Dev(b200)
    blk = FfnBlock(b200, dev, rng, E, FF, R.Q4_K, T)
    gbuf = dev.f32(FF * T + E * T, 0)
    shift = (FF * T - E * T // 2)                  # ADD's [E, T] starts in gate's second half and runs past its end
    # re-point gate, silu's source and the ADD destination into the shared buffer
    t, mk = dev.t, b200.make_op
    ops = list(blk.ops)
    ops[3] = mk(b200.OP_MUL_MAT, t(gbuf, [FF, T]), [ops[3].src[0], ops[3].src[1]])
    ops[4] = mk(b200.OP_SILU, ops[4].dst, [t(gbuf, [FF, T])])
    ops[7] = mk(b200.OP_ADD, t(gbuf, [E, T], off=shift * 4), [ops[7].src[0], ops[7].src[1]])
    probe = dev.f32(256)
    ops.append(mk(b200.OP_ADD, t(probe, [256]), [t(gbuf, [256]), t(gbuf, [256])]))
    res = {}
    for fusion in (1, 2):
        gbuf.zero_(); probe.fill_(float("nan")); torch.cuda.synchronize()
        n = run(ctx, ops, fusion)
        res[fusion] = (n, probe.cpu().numpy().copy(), gbuf.cpu().numpy()[:shift].copy())
    # the FFN fusion must decline (it would save 4 launches); down + ADD alone may still fuse, it leaves gate in place
    assert res[2][0] >= res[1][0] - 1, ("the FFN must not fuse: a later op reads gate", res[1][0], res[2][0])
    assert np.array_equal(res[1][1], res[2][1]) and np.array_equal(res[1][2], res[2][2])
    rows = np.arange(256)
    Wg = FR.dequant_rows(R.Q4_K, blk.W["gate"], E, rows)
    xa, _ = FR.quant_act(R.Q4_K, blk.xn)
    gate_ref = (xa @ Wg.T)[0]
    flip = FR.flip_bound(blk.xn, R.Q4_K, Wg, NORM_EPS, scale=0.0, per_element=True)[0]
    tol = 2 * (FR.REL * np.abs(gate_ref).max() + flip)
    assert (np.abs(res[2][1] - 2 * gate_ref) <= tol).all(), "gate's head was not written"


def test_decline_f16_weight_norm_mm(b200, opts):
    """an F16 weight after RMS_NORM MUL: no layer fusion, the same launches and the same answer as fusion 1"""
    import torch
    ctx = opts
    rng = np.random.default_rng(9)
    dev = Dev(b200)
    K, N, T = 2048, 512, 1
    x, nw, xn = norm_stage(rng, T, K)
    w = (rng.standard_normal((N, K)) * 0.05).astype(np.float16)
    wd = dev.put(w.view(np.uint8).reshape(-1))
    xd, nwd, cur, cur2, out = dev.put(x), dev.put(nw), dev.f32(K * T), dev.f32(K * T), dev.f32(N * T)
    ops = [b200.make_op(b200.OP_RMS_NORM, dev.t(cur, [K, T]), [dev.t(xd, [K, T])], [EPS]),
           b200.make_op(b200.OP_MUL, dev.t(cur2, [K, T]), [dev.t(cur, [K, T]), b200.tensor(nwd.data_ptr(), b200.F32, [K], flags=1)]),
           b200.make_op(b200.OP_MUL_MAT, dev.t(out, [N, T]), [b200.tensor(wd.data_ptr(), b200.F16, [K, N], flags=1), dev.t(cur2, [K, T])])]
    res = {}
    for fusion in (1, 2):
        out.fill_(float("nan")); torch.cuda.synchronize()
        res[fusion] = (run(ctx, ops, fusion), out.cpu().numpy().copy())
    assert res[1][0] == res[2][0]
    assert np.array_equal(res[1][1], res[2][1])
    want = R.orc_mul_mat(R.F16, w.view(np.uint8).reshape(-1), xn, N, K)
    assert np.abs(res[2][1].reshape(T, N) - want).max() <= 1e-5 * np.abs(want).max()
