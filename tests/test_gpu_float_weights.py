"""F16 / BF16 weight MUL_MAT on the tensor-core kernels (gemv_f16.cu for <= 32 token columns, gemm_f16_tc.cu above): results against
the oracle and a float64 matmul of the rounded operands, batch layouts, the fallbacks that keep the float kernel, the dispatch itself,
determinism, whole llama ubatches and CUDA-graph replay of an F16 decode step."""
import os
import sys

import numpy as np
import pytest

import bf16_ref as B
import reflib as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

TYPES = [R.F16, B.BF16]
SHAPES = [(16, 256), (17, 512), (333, 2048), (1024, 4096), (4097, 4104), (300, 14336), (4096, 4096)]
MS = [1, 2, 3, 4, 5, 8, 16, 17, 32, 33, 64, 200, 512]
BOUND = 1e-5                    # max |got - want| <= BOUND * max |want|, as the float-weight test of test_gpu_mulmat.py


@pytest.fixture(scope="module")
def torch():
    import torch as T
    return T


def tdtype(torch, t):
    return torch.float16 if t == R.F16 else torch.bfloat16


def rand_weights(torch, t, N, K, seed, rows_stride=None):
    """device weights of type t ([N, rows_stride] 16-bit, the first K of a row used) and their values as float64"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    rs = rows_stride or K
    w = ((torch.rand(N, rs, device="cuda", generator=g) * 2 - 1) * 0.05).to(tdtype(torch, t))
    return w, w[:, :K].double()


def rounded_x(torch, t, x):
    return x.to(tdtype(torch, t)).double()


def mm_op(b200, t, w, K, N, x, dst, w_ne2=1, w_nb1=None, x_nb1=None, d_nb1=None, M=None, batch=1, flags=0):
    M = M if M is not None else x.shape[-2]
    es = 4 if t == R.F32 else 2
    w_nb1 = w_nb1 or K * es
    x_nb1 = x_nb1 or K * 4
    d_nb1 = d_nb1 or N * 4
    wt = b200.tensor(w.data_ptr(), t, [K, N, w_ne2], nb=[es, w_nb1, w_nb1 * N, w_nb1 * N * w_ne2], flags=flags)
    xt = b200.tensor(x.data_ptr(), R.F32, [K, M, batch], nb=[4, x_nb1, x_nb1 * M, x_nb1 * M * batch])
    dt = b200.tensor(dst.data_ptr(), R.F32, [N, M, batch], nb=[4, d_nb1, d_nb1 * M, d_nb1 * M * batch])
    return b200.make_op(b200.OP_MUL_MAT, dt, [wt, xt])


def run_mm(b200, ctx, torch, t, w, K, N, x, **kw):
    M = x.shape[0]
    out = torch.full((M, N), float("nan"), dtype=torch.float32, device="cuda")
    op = mm_op(b200, t, w, K, N, x, out, **kw)
    assert b200.supports(op)
    torch.cuda.synchronize()
    ctx.compute_op(op)
    ctx.sync()
    return out


def check_close(got, want):
    got = got.double()
    err = float((got - want).abs().max())
    scale = float(want.abs().max())
    assert bool(torch_isfinite(got)), "non-finite output"
    assert err <= BOUND * scale, "max err %.3g of max |want| %.3g (rel %.3g)" % (err, scale, err / scale)


def torch_isfinite(t):
    import torch as T
    return T.isfinite(t).all()


@pytest.mark.parametrize("M", MS)
@pytest.mark.parametrize("N,K", SHAPES)
@pytest.mark.parametrize("t", TYPES)
def test_float_weight_vs_reference(b200, ctx, torch, t, N, K, M):
    seed = N * 7 + K + M * 13 + t
    w, wd = rand_weights(torch, t, N, K, seed)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    x = torch.randn(M, K, device="cuda", generator=g)
    got = run_mm(b200, ctx, torch, t, w, K, N, x)
    want = rounded_x(torch, t, x) @ wd.T
    check_close(got, want)
    # the CPU backend's arithmetic on a row subset: the C oracle (F16), tests/bf16_ref.py (BF16)
    rng = np.random.default_rng(seed)
    rows = np.unique(np.concatenate([np.arange(min(N, 16)), rng.integers(0, N, 16), [N - 1]]))
    if N * K * M > (1 << 26):
        rows = rows[:12]
    wsub = w[torch.from_numpy(rows).cuda()].contiguous().cpu().view(torch.int16).numpy().view(np.uint8).reshape(-1)
    ref = R.orc_mul_mat(t, wsub, x.cpu().numpy(), len(rows), K) if t == R.F16 else B.mul_mat_bf16(wsub, x.cpu().numpy(), len(rows), K)
    g_sub = got.cpu().numpy()[:, rows]
    assert np.abs(g_sub - ref).max() <= BOUND * max(np.abs(ref).max(), 1e-30)


@pytest.mark.parametrize("M", [3, 40])
@pytest.mark.parametrize("t", TYPES)
def test_weight_broadcast_over_batch(b200, ctx, torch, t, M):
    N, K, B, WB = 96, 512, 8, 2
    w, _ = rand_weights(torch, t, N * WB, K, 11 + M)
    g = torch.Generator(device="cuda").manual_seed(12)
    x = torch.randn(B, M, K, device="cuda", generator=g)
    out = torch.full((B, M, N), float("nan"), dtype=torch.float32, device="cuda")
    op = mm_op(b200, t, w, K, N, x, out, w_ne2=WB, M=M, batch=B)
    assert b200.supports(op)
    torch.cuda.synchronize()
    ctx.compute_op(op)
    ctx.sync()
    wd = w.double().reshape(WB, N, K)
    for i2 in range(B):
        check_close(out[i2], rounded_x(torch, t, x[i2]) @ wd[i2 // (B // WB)].T)


@pytest.mark.parametrize("M", [5, 100])
@pytest.mark.parametrize("t", TYPES)
def test_dst_column_stride_larger_than_n(b200, ctx, torch, t, M):
    N, K, P = 200, 1024, 232
    w, wd = rand_weights(torch, t, N, K, 21 + M)
    g = torch.Generator(device="cuda").manual_seed(22)
    x = torch.randn(M, K, device="cuda", generator=g)
    out = torch.full((M, P), -7.0, dtype=torch.float32, device="cuda")
    op = mm_op(b200, t, w, K, N, x, out, d_nb1=P * 4)
    torch.cuda.synchronize()
    ctx.compute_op(op)
    ctx.sync()
    check_close(out[:, :N], rounded_x(torch, t, x) @ wd.T)
    assert bool((out[:, N:] == -7.0).all()), "wrote past the N rows of a dst column"


@pytest.mark.parametrize("case", ["k_not_multiple_of_8", "x_column_stride_unaligned", "strided_weight_view", "f32_weights", "cpu_exact"])
@pytest.mark.parametrize("M", [2, 40])
def test_fallbacks_stay_correct(b200, ctx, torch, case, M):
    t, N, K = R.F16, 48, 256
    kw = {}
    if case == "k_not_multiple_of_8":
        K = 100
    w, wd = rand_weights(torch, t, N, K, 31, rows_stride=K + 8 if case == "strided_weight_view" else None)
    if case == "strided_weight_view":
        kw["w_nb1"] = (K + 8) * 2
    g = torch.Generator(device="cuda").manual_seed(32)
    xs = K + 1 if case == "x_column_stride_unaligned" else K
    xbuf = torch.randn(M, xs, device="cuda", generator=g)
    x = xbuf[:, :K]
    kw["x_nb1"] = xs * 4
    if case == "f32_weights":
        t, w = R.F32, wd.float().contiguous()
    out = torch.full((M, N), float("nan"), dtype=torch.float32, device="cuda")
    op = mm_op(b200, t, w, K, N, xbuf, out, M=M, **kw)
    assert b200.supports(op)
    torch.cuda.synchronize()
    if case == "cpu_exact":
        ctx.set_option("cpu_exact", 1)
    try:
        ctx.compute_op(op)
        ctx.sync()
    finally:
        ctx.set_option("cpu_exact", 0)
    xr = x.double() if t == R.F32 else rounded_x(torch, t, x)
    check_close(out, xr @ wd.T)


def kernel_names(torch, fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events()]


@pytest.mark.parametrize("M,kernel", [(8, "b200_gemv_f16_kernel"), (128, "b200_gemm_f16_tc_kernel")])
@pytest.mark.parametrize("t", TYPES)
def test_dispatch_reaches_new_kernels(b200, ctx, torch, t, M, kernel):
    N, K = 1024, 4096
    w, _ = rand_weights(torch, t, N, K, 41)
    x = torch.randn(M, K, device="cuda")
    out = torch.empty(M, N, dtype=torch.float32, device="cuda")
    op = mm_op(b200, t, w, K, N, x, out)
    ctx.compute_op(op)                   # warm-up outside the trace (module load, scratch growth)
    ctx.sync()
    names = kernel_names(torch, lambda: (ctx.compute_op(op), ctx.sync()))
    assert any(kernel in n for n in names), names
    assert not any("b200_mul_mat_float_kernel" in n for n in names), names


@pytest.mark.parametrize("M", [1, 64])
@pytest.mark.parametrize("t", TYPES)
def test_split_k_bitwise_deterministic(b200, ctx, torch, t, M):
    N, K = 1024, 14336
    w, _ = rand_weights(torch, t, N, K, 51)
    x = torch.randn(M, K, device="cuda")
    a = run_mm(b200, ctx, torch, t, w, K, N, x)
    b = run_mm(b200, ctx, torch, t, w, K, N, x)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))


SCHEDULE = [(5, 0), (1, 5), (2, 6), (4, 8), (1, 12), (3, 13), (32, 16), (128, 48)]   # prompt chunk, 1..4-token steps, a 32-token step, a 128-token ubatch
FAST_MODE_BOUND = 4e-2          # the fast-mode envelope of test_gpu_llama_step.py


def run_steps(torch, ctx, g, fusion, wants):
    """device logits of every SCHEDULE ubatch; the oracle's are computed into `wants` on the first call (they do not depend on fusion)"""
    import llama_forward as OF
    ctx.set_option("fusion", fusion)
    rng = np.random.default_rng(5)
    caches = None
    outs = []
    for i, (T, kv_head) in enumerate(SCHEDULE):
        n_kv = 256
        emb, pos, mask = g.set_inputs_host(T, kv_head, n_kv, rng)
        g.inp_embd[:T * g.E] = torch.from_numpy(emb.reshape(-1)).cuda()
        g.pos[:T] = torch.from_numpy(pos).cuda()
        g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).cuda()
        torch.cuda.synchronize()
        if len(wants) <= i:
            want, caches = OF.forward(g, emb, pos, mask, kv_head, n_kv, caches=caches)
            wants.append(want)
        ctx.compute(g.build(T, kv_head, n_kv))
        ctx.sync()
        outs.append((g.logits[:T * g.V].cpu().numpy().reshape(T, g.V).copy(), wants[i]))
    return outs


def margin(row):
    part = np.partition(row, row.size - 2)
    return (part[-1] - part[-2]) / np.abs(row).max()


@pytest.mark.parametrize("kv", ["f16", "q8_0"])
@pytest.mark.parametrize("ftype", ["f16", "bf16"])
@pytest.mark.parametrize("model", ["tiny-d128", "mid-d128"])
def test_llama_ubatches_16bit_weights(b200, ctx, torch, monkeypatch, model, ftype, kv):
    B.with_bf16(monkeypatch)                 # the oracle forward multiplies BF16 weights through the test-side reference
    from __graft_entry__ import load_llama_graph
    g = load_llama_graph().LlamaGraph(b200, model=model, ftype=ftype, kv=kv, n_ctx=256, max_tokens=128)
    worst, wants = (0.0, None), []
    try:
        for fusion in (0, 2):
            for lw in g.layers:
                lw["k_cache"].zero_(); lw["v_cache"].zero_()
            for (got, want), (T, _) in zip(run_steps(torch, ctx, g, fusion, wants), SCHEDULE):
                assert np.isfinite(got).all()
                for r in range(T):
                    rel = float(np.abs(got[r] - want[r]).max() / np.abs(want[r]).max())
                    if rel > worst[0]:
                        worst = (rel, (fusion, T, r))
                    assert rel <= FAST_MODE_BOUND, (fusion, T, r, rel)
                    if got[r].argmax() != want[r].argmax():
                        assert margin(want[r]) <= 2 * rel, (fusion, T, r, rel, margin(want[r]))
    finally:
        ctx.set_option("fusion", 2)
    print("%s %s kv %s: worst row %.3g of the largest logit at (fusion, T, row) %s" % (model, ftype, kv, worst[0], worst[1]))


def test_f16_decode_step_graph_replay(b200, ctx, torch):
    from __graft_entry__ import load_llama_graph
    g = load_llama_graph().LlamaGraph(b200, model="tiny-d128", ftype="f16", kv="q8_0", n_ctx=256, max_tokens=1)
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
            n0 = ctx.launches()
            ctx.compute(ops)
            ctx.sync()
            assert ctx.launches() - n0 == 1, "the F16 decode step was not replayed as one graph"
            assert np.array_equal(g.logits[:g.V].cpu().numpy(), eager)
    finally:
        ctx.set_option("cuda_graphs", 0)
