"""F16 / BF16 MoE expert matmuls (MUL_MAT_ID) on the grouped tensor-core kernels: the (token, slot) pairs are counting-sorted by expert on
the device, then < 32 pairs per expert on average go through the grouped weight-streaming kernel (gemv_f16.cu), more through the grouped
tcgen05 GEMM (gemm_f16_tc.cu).  Results against the oracle's MUL_MAT_ID (F16), tests/bf16_moe_ref.py (BF16) and a float64 matmul of the
rounded operands; the dst layout; the fallbacks that keep the float kernel; the dispatch; determinism; whole MoE ubatches and CUDA-graph
replay of a BF16 MoE decode step."""
import os
import sys

import numpy as np
import pytest

import bf16_moe_ref as BM
import bf16_ref as B
import reflib as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

TYPES = [R.F16, B.BF16]
SHAPES = [(160, 1024), (333, 4104), (1024, 4096), (4096, 14336)]
N_TOKS = [1, 2, 4, 5, 16, 40, 97, 200, 512]
N_EXPERT, N_USED = 8, 2
SKEW = np.array([10, 4, 2, 1, 1, 0.5, 0.5, 0.0])     # expert 7 idle, expert 0 > 32 pairs from 40 tokens on, > 128 from 200 on
BOUND = 1e-5                    # max |got - want| <= BOUND * max |want|, as in test_gpu_float_weights.py
# K = 14336 on the tcgen05 GEMM: one f32 accumulation chain of 896 MMAs per output.  The dense GEMM measures 1.6-1.9e-5 on the same
# 4096 x 14336 matrix at M = 512 (profiles/float_weights.jsonl), the grouped GEMM the same (profiles/moe_float_weights.jsonl)
BOUND_LONG_K = 3e-5


def bound(K, n_tok):
    return BOUND_LONG_K if K > 8192 and n_tok * N_USED >= 32 * N_EXPERT else BOUND


@pytest.fixture(scope="module")
def torch():
    import torch as T
    return T


def tdtype(torch, t):
    return torch.float16 if t == R.F16 else torch.bfloat16


def rand_experts(torch, t, N, K, seed, dtype=None):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return ((torch.rand(N_EXPERT, N, K, device="cuda", generator=g) * 2 - 1) * 0.05).to(dtype or tdtype(torch, t))


def routing(rng, n_tok, skew=True):
    """[n_tok, n_expert] rows of an "argsort" (the first N_USED are the chosen experts), as build_moe_ffn's top-k view reads them"""
    p = SKEW / SKEW.sum() if skew else None
    return np.stack([np.concatenate([c := rng.choice(N_EXPERT, N_USED, replace=False, p=p), np.setdiff1d(np.arange(N_EXPERT), c)])
                     for _ in range(n_tok)]).astype(np.int32)


def moe_op(b200, t, A, b, sel, dst, N, K, b_ne1, d_nb1=None, b_nb1=None, es=2):
    n_tok = sel.shape[0]
    d_nb1 = d_nb1 or N * 4
    b_nb1 = b_nb1 or K * 4
    return b200.make_op(b200.OP_MUL_MAT_ID, b200.tensor(dst.data_ptr(), R.F32, [N, N_USED, n_tok], [4, d_nb1, d_nb1 * N_USED, d_nb1 * N_USED * n_tok]),
                        [b200.tensor(A.data_ptr(), t, [K, N, N_EXPERT], nb=[es, K * es, K * es * N, K * es * N * N_EXPERT], flags=1),
                         b200.tensor(b.data_ptr(), R.F32, [K, b_ne1, n_tok], [4, b_nb1, b_nb1 * b_ne1, b_nb1 * b_ne1 * n_tok]),
                         b200.tensor(sel.data_ptr(), R.I32, [N_USED, n_tok], [4, N_EXPERT * 4, N_EXPERT * 4 * n_tok, N_EXPERT * 4 * n_tok])])


def want_f64(torch, A, xr, ids, b_ne1):
    """float64 [n_tok, n_used, N] of the rounded operands"""
    n_tok = ids.shape[0]
    out = torch.zeros(n_tok, N_USED, A.shape[1], dtype=torch.float64, device="cuda")
    idt = torch.from_numpy(ids).cuda().long()
    Ad = A.double()
    for s in range(N_USED):
        xs = xr[:, s % b_ne1]
        for e in range(N_EXPERT):
            m = idt[:, s] == e
            if bool(m.any()):
                out[m, s] = xs[m] @ Ad[e].T
    return out


def run(b200, ctx, torch, op):
    assert b200.supports(op)
    torch.cuda.synchronize()
    l0 = ctx.launches()
    ctx.compute_op(op)
    ctx.sync()
    return ctx.launches() - l0


def check_close(got, want, bnd=BOUND):
    got = got.double()
    assert bool(torch_isfinite(got)), "non-finite output"
    err, scale = float((got - want).abs().max()), float(want.abs().max())
    assert err <= bnd * scale, "max err %.3g of max |want| %.3g (rel %.3g)" % (err, scale, err / scale)


def torch_isfinite(t):
    import torch as T
    return T.isfinite(t).all()


def expert_rows_bytes(torch, A, rows):
    """raw bytes of [N_EXPERT, len(rows), K] (the oracle's As layout) for a subset of every expert's rows"""
    return A[:, torch.from_numpy(rows).cuda()].contiguous().cpu().view(torch.int16).numpy().view(np.uint8).reshape(-1)


@pytest.mark.parametrize("n_tok", N_TOKS)
@pytest.mark.parametrize("N,K", SHAPES)
@pytest.mark.parametrize("b_ne1", [1, N_USED])
@pytest.mark.parametrize("t", TYPES)
def test_moe_float_experts_vs_reference(b200, ctx, torch, t, b_ne1, N, K, n_tok):
    seed = N * 7 + K + n_tok * 13 + t + b_ne1
    rng = np.random.default_rng(seed)
    A = rand_experts(torch, t, N, K, seed)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    b = torch.randn(n_tok, b_ne1, K, device="cuda", generator=g)
    sel = routing(rng, n_tok)
    ids = np.ascontiguousarray(sel[:, :N_USED])
    out = torch.full((n_tok, N_USED, N), float("nan"), dtype=torch.float32, device="cuda")
    launches = run(b200, ctx, torch, moe_op(b200, t, A, b, torch.from_numpy(sel).cuda(), out, N, K, b_ne1))
    npairs = n_tok * N_USED
    # group + stream (+ split-K reduce), or group + pack + GEMM (+ reduce), whatever the routing
    assert launches <= (3 if npairs < 32 * N_EXPERT else 4), launches
    check_close(out, want_f64(torch, A, b.to(tdtype(torch, t)).double(), ids, b_ne1), bound(K, n_tok))
    # the CPU backend's arithmetic on a row subset of every expert (and the first tokens of the biggest cases)
    rows = np.unique(np.concatenate([np.arange(min(N, 8)), rng.integers(0, N, 8), [N - 1]]))
    nt = n_tok if N * K * n_tok <= (1 << 31) else 16
    As = expert_rows_bytes(torch, A, rows)
    bn = b[:nt].cpu().numpy()
    ref = R.orc_mul_mat_id(t, As, bn, ids[:nt], len(rows), K, N_EXPERT) if t == R.F16 else BM.mul_mat_id_bf16(As, bn, ids[:nt], len(rows), K, N_EXPERT)
    got = out[:nt].cpu().numpy()[:, :, rows]
    assert np.abs(got - ref).max() <= bound(K, n_tok) * max(np.abs(ref).max(), 1e-30)


@pytest.mark.parametrize("n_tok", [3, 200])
@pytest.mark.parametrize("t", TYPES)
def test_dst_slot_stride_larger_than_n(b200, ctx, torch, t, n_tok):
    N, K, P = 200, 1024, 232
    rng = np.random.default_rng(60 + n_tok)
    A = rand_experts(torch, t, N, K, 61 + n_tok)
    b = torch.randn(n_tok, 1, K, device="cuda")
    sel = routing(rng, n_tok)
    out = torch.full((n_tok, N_USED, P), -7.0, dtype=torch.float32, device="cuda")
    run(b200, ctx, torch, moe_op(b200, t, A, b, torch.from_numpy(sel).cuda(), out, N, K, 1, d_nb1=P * 4))
    check_close(out[:, :, :N], want_f64(torch, A, b.to(tdtype(torch, t)).double(), np.ascontiguousarray(sel[:, :N_USED]), 1))
    assert bool((out[:, :, N:] == -7.0).all()), "wrote past the N rows of a dst column"


@pytest.mark.parametrize("case", ["k_not_multiple_of_8", "b_column_stride_unaligned", "f32_experts", "cpu_exact"])
@pytest.mark.parametrize("n_tok", [2, 200])
def test_fallbacks_stay_correct(b200, ctx, torch, case, n_tok):
    t, N, K = R.F16, 48, 256
    if case == "k_not_multiple_of_8":
        K = 100
    rng = np.random.default_rng(70 + n_tok)
    A = rand_experts(torch, t, N, K, 71)
    es = 2
    if case == "f32_experts":
        t, A, es = R.F32, A.float().contiguous(), 4
    bs = K + 1 if case == "b_column_stride_unaligned" else K
    bbuf = torch.randn(n_tok, N_USED, bs, device="cuda")
    sel = routing(rng, n_tok)
    out = torch.full((n_tok, N_USED, N), float("nan"), dtype=torch.float32, device="cuda")
    op = moe_op(b200, t, A, bbuf, torch.from_numpy(sel).cuda(), out, N, K, N_USED, b_nb1=bs * 4, es=es)
    if case == "cpu_exact":
        ctx.set_option("cpu_exact", 1)
    try:
        run(b200, ctx, torch, op)
    finally:
        ctx.set_option("cpu_exact", 0)
    xr = bbuf[:, :, :K].double() if t == R.F32 else bbuf[:, :, :K].to(tdtype(torch, t)).double()
    check_close(out, want_f64(torch, A, xr, np.ascontiguousarray(sel[:, :N_USED]), N_USED))


def dispatch_trace(t, n_toks):
    """per token count: launches of one MUL_MAT_ID and the kernel names of its profiler trace.  Runs in a fresh process (see
    test_dispatch_reaches_grouped_kernels): after earlier profiler sessions in a long test process, CUDA kernel records can go missing."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from __graft_entry__ import load_package
    b200 = load_package()
    ctx = b200.Context(0)
    N, K = 1024, 4096
    A = rand_experts(torch, t, N, K, 81)
    res = []
    for n_tok in n_toks:
        b = torch.randn(n_tok, 1, K, device="cuda")
        sel = torch.from_numpy(routing(np.random.default_rng(n_tok), n_tok, skew=False)).cuda()
        out = torch.empty(n_tok, N_USED, N, dtype=torch.float32, device="cuda")
        op = moe_op(b200, t, A, b, sel, out, N, K, 1)
        launches = run(b200, ctx, torch, op)               # also the warm-up outside the trace (module load, scratch growth)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ctx.compute_op(op)
            ctx.sync()
        res.append((launches, [e.name for e in prof.events()]))
    ctx.close()
    return res


@pytest.mark.parametrize("n_toks,kernel", [((1,), "b200_gemv_f16_grouped_kernel"), ((4, 16, 100), "b200_gemv_f16_grouped_kernel"),
                                           ((128, 512), "b200_gemm_f16_tc_grouped_kernel")])
@pytest.mark.parametrize("t", TYPES)
def test_dispatch_reaches_grouped_kernels(t, n_toks, kernel):
    import json
    import subprocess
    code = "import json, sys; sys.path[:0] = [%r, %r]; import test_gpu_moe_float_weights as T; print(json.dumps(T.dispatch_trace(%d, %r)))" % (
        os.path.dirname(os.path.abspath(__file__)), ROOT, t, list(n_toks))
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    res = json.loads(p.stdout.strip().splitlines()[-1])
    for launches, names in res:
        assert any(kernel in n for n in names), names
        assert any("b200_moe_group_kernel" in n for n in names), names
        assert not any("b200_mul_mat_id_float_kernel" in n or "b200_mul_mat_float_kernel" in n for n in names), names
    counts = [launches for launches, _ in res]
    assert len(set(counts)) == 1, "launches per op depend on the number of tokens: %s" % counts


@pytest.mark.parametrize("n_tok,N,K", [(1, 4096, 14336), (16, 1024, 14336), (200, 333, 4104), (512, 4096, 14336)])
@pytest.mark.parametrize("t", TYPES)
def test_bitwise_deterministic(b200, ctx, torch, t, n_tok, N, K):
    A = rand_experts(torch, t, N, K, 91)
    b = torch.randn(n_tok, 1, K, device="cuda")
    sel = torch.from_numpy(routing(np.random.default_rng(92), n_tok)).cuda()
    res = []
    for _ in range(2):
        out = torch.full((n_tok, N_USED, N), float("nan"), dtype=torch.float32, device="cuda")
        run(b200, ctx, torch, moe_op(b200, t, A, b, sel, out, N, K, 1))
        res.append(out)
    assert torch.equal(res[0].view(torch.int32), res[1].view(torch.int32))


# 1-, 2-, 4-, 5-, 32- and 128-token ubatches; tiny-moe has 4 experts: 64 pairs stream, 256 pairs take the grouped GEMM
SCHEDULE = [(5, 0), (1, 5), (2, 6), (4, 8), (32, 12), (128, 44)]
FAST_MODE_BOUND = 4e-2          # the fast-mode envelope of test_gpu_llama_step.py


@pytest.mark.parametrize("kv", ["f16", "q8_0"])
@pytest.mark.parametrize("ftype", ["f16", "bf16"])
def test_moe_ubatches_16bit_experts(b200, ctx, torch, monkeypatch, ftype, kv):
    """test_moe_steps_fast_mode's checks for a 16-bit MoE model: rows whose router decision is a near-tie in the oracle are exempt"""
    BM.with_bf16_moe(monkeypatch)              # the oracle forward multiplies BF16 weights and experts through the test-side reference
    import llama_forward as OF
    from __graft_entry__ import load_llama_graph
    g = load_llama_graph().LlamaGraph(b200, model="tiny-moe", ftype=ftype, kv=kv, n_ctx=256, max_tokens=128)
    wants, margins = [], []
    try:
        for fusion in (0, 2):
            ctx.set_option("fusion", fusion)
            for lw in g.layers:
                lw["k_cache"].zero_(); lw["v_cache"].zero_()
            rng = np.random.default_rng(5)
            caches, checked = None, 0
            for i, (T, kv_head) in enumerate(SCHEDULE):
                emb, pos, mask = g.set_inputs_host(T, kv_head, 256, rng)
                g.inp_embd[:T * g.E] = torch.from_numpy(emb.reshape(-1)).cuda()
                g.pos[:T] = torch.from_numpy(pos).cuda()
                g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).cuda()
                torch.cuda.synchronize()
                if len(wants) <= i:
                    OF.ROUTER_MARGINS.clear()
                    want, caches = OF.forward(g, emb, pos, mask, kv_head, 256, caches=caches)
                    wants.append(want)
                    margins.append(np.minimum.reduce(list(OF.ROUTER_MARGINS)) < 0.02)
                ctx.compute(g.build(T, kv_head, 256))
                ctx.sync()
                got = g.logits[:T * g.V].cpu().numpy().reshape(T, g.V)
                assert np.isfinite(got).all()
                for r in range(T):
                    if margins[i][r]:
                        continue
                    rel = float(np.abs(got[r] - wants[i][r]).max() / np.abs(wants[i][r]).max())
                    assert rel <= FAST_MODE_BOUND, (fusion, T, r, rel)
                    checked += 1
            assert checked >= 50, "too many routing near-ties to say anything"
    finally:
        ctx.set_option("fusion", 2)


def test_bf16_moe_decode_step_graph_replay(b200, ctx, torch):
    from __graft_entry__ import load_llama_graph
    g = load_llama_graph().LlamaGraph(b200, model="tiny-moe", ftype="bf16", kv="q8_0", n_ctx=256, max_tokens=1)
    rng = np.random.default_rng(3)
    emb, pos, mask = g.set_inputs_host(1, 7, 256, rng)
    g.inp_embd[:g.E] = torch.from_numpy(emb.reshape(-1)).cuda()
    g.pos[:1] = torch.from_numpy(pos).cuda()
    g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).cuda()
    torch.cuda.synchronize()
    ops = g.build(1, 7, 256)
    try:
        ctx.set_option("fusion", 2)
        ctx.set_option("cuda_graphs", 0)
        ctx.compute(ops)
        ctx.sync()
        eager = g.logits[:g.V].cpu().numpy().copy()
        ctx.set_option("cuda_graphs", 1)
        for _ in range(2):                       # first sighting runs eagerly, the second captures
            ctx.compute(ops)
            ctx.sync()
        for _ in range(3):
            g.logits.zero_()
            torch.cuda.synchronize()
            n0 = ctx.launches()
            ctx.compute(ops)
            ctx.sync()
            assert ctx.launches() - n0 == 1, "the BF16 MoE decode step was not replayed as one graph"
            assert np.array_equal(g.logits[:g.V].cpu().numpy(), eager)
    finally:
        ctx.set_option("cuda_graphs", 0)
