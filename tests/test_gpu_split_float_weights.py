"""Row-split F16 / BF16 weight MUL_MAT (B200_TENSOR_FLAG_SPLIT, what the plugin's split buffer type emits for MOSTLY_F16 /
MOSTLY_BF16 files under --split-mode row) and the one-process-per-GPU (Megatron) form in bf16.

Every shard runs the one-GPU dispatch on its own device (gemv_f16 up to 32 token columns, gemm_f16_tc above, the float kernel for
layouts those refuse).  Both tensor-core kernels choose their K slices from the shard's row count, so a split result equals the
unsplit one up to f32 summation order (not bit for bit, as the quantised split does), and a repeated split gives the same bits.
op_mul_mat_split runs a shard that lives on the calling context's device on that context, so the whole split path runs on one GPU
with every shard on device 0; the cases that need shards on other devices skip below two GPUs."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SPLIT = 2                       # B200_TENSOR_FLAG_SPLIT
BOUND = 1e-5                    # max |got - want| <= BOUND * max |want|, as test_gpu_float_weights.py
FAST_MODE_BOUND = 4e-2          # the fast-mode logit envelope of test_gpu_float_weights.py / test_gpu_llama_step.py
MS = [1, 5, 32, 33, 200]
KS = [4096, 8192, 1004]         # 1004: K % 8 != 0, every shard takes the float kernel
# (N, row_low) of the one-GPU splits
SPLITS = {
    "two_at_768": (1536, [0, 768, 1536]),
    "three_uneven_one_empty": (1536, [0, 640, 640, 1536]),
    "last_not_multiple_of_128": (1100, [0, 1024, 1100]),
}


class Split(C.Structure):
    """b200_split of include/ggml_b200.h"""
    _fields_ = [("n_dev", C.c_int32), ("device", C.c_int32 * 16), ("shard", C.c_void_p * 16), ("row_low", C.c_int64 * 17)]


@pytest.fixture(scope="module")
def torch():
    import torch as T
    return T


def tdtype(torch, b200, t):
    return torch.float16 if t == b200.F16 else torch.bfloat16


def rand_weights(torch, b200, t, N, K, seed):
    """[N, K] weights of 16-bit type t on device 0 and their values as float64"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    w = ((torch.rand(N, K, device="cuda", generator=g) * 2 - 1) * 0.05).to(tdtype(torch, b200, t))
    return w, w.double()


def shard_table(torch, w, row_low, devices):
    """b200_split over w's rows: shard i = rows [row_low[i], row_low[i + 1]) as a dense matrix on devices[i], with the plugin's 512
    bytes of slack; returns the table and the shard tensors (kept alive by the caller)"""
    N, K = w.shape
    sp, keep = Split(), []
    sp.n_dev = len(devices)
    for i, dev in enumerate(devices):
        sp.device[i], sp.row_low[i] = dev, row_low[i]
        nr = row_low[i + 1] - row_low[i]
        if nr > 0:
            s = torch.zeros(nr * K + 256, dtype=w.dtype, device="cuda:%d" % dev)
            s[:nr * K] = w[row_low[i]:row_low[i + 1]].reshape(-1).to(s.device)
            keep.append(s)
            sp.shard[i] = s.data_ptr()
    sp.row_low[len(devices)] = N
    return sp, keep


def mm_op(b200, t, w_ptr, K, N, x, dst, flags, d_nb1=None):
    M = x.shape[0]
    d_nb1 = d_nb1 or N * 4
    wt = b200.tensor(w_ptr, t, [K, N], flags=b200.TENSOR_FLAG_WEIGHT | flags)
    dt = b200.tensor(dst.data_ptr(), b200.F32, [N, M], nb=[4, d_nb1, d_nb1 * M, d_nb1 * M])
    return b200.make_op(b200.OP_MUL_MAT, dt, [wt, b200.tensor(x.data_ptr(), b200.F32, [K, M])])


def run(torch, ctx, op):
    torch.cuda.synchronize()
    ctx.compute_op(op)
    ctx.sync()


def max_err(got, want):
    assert bool(got.isfinite().all()), "non-finite output"
    return float((got.double() - want).abs().max())


def check_split(b200, ctx, torch, t, N, K, M, row_low, devices, seed):
    """split result against float64 and against the unsplit op; a second run, into a dst with padded columns, gives the same bits
    and leaves the padding alone"""
    w, wd = rand_weights(torch, b200, t, N, K, seed)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    x = torch.randn(M, K, device="cuda", generator=g)
    want = x.to(w.dtype).double() @ wd.T
    scale = float(want.abs().max())
    sp, keep = shard_table(torch, w, row_low, devices)
    got = torch.full((M, N), float("nan"), dtype=torch.float32, device="cuda")
    op = mm_op(b200, t, C.addressof(sp), K, N, x, got, SPLIT)
    assert b200.supports(op)
    run(torch, ctx, op)
    err = max_err(got, want)
    assert err <= BOUND * scale, "vs float64: rel %.3g" % (err / scale)
    one = torch.full((M, N), float("nan"), dtype=torch.float32, device="cuda")
    run(torch, ctx, mm_op(b200, t, w.data_ptr(), K, N, x, one, 0))
    d1 = float((got - one).abs().max())
    assert d1 <= 2 * BOUND * scale, "vs the unsplit op: rel %.3g" % (d1 / scale)
    P = 24
    padded = torch.full((M, N + P), -7.0, dtype=torch.float32, device="cuda")
    run(torch, ctx, mm_op(b200, t, C.addressof(sp), K, N, x, padded, SPLIT, d_nb1=(N + P) * 4))
    assert torch.equal(padded[:, :N].contiguous().view(torch.int32), got.view(torch.int32)), "two runs of one split differ"
    assert bool((padded[:, N:] == -7.0).all()), "a shard wrote outside its rows"
    del keep


@pytest.mark.parametrize("split", list(SPLITS))
@pytest.mark.parametrize("K", KS)
@pytest.mark.parametrize("M", MS)
@pytest.mark.parametrize("tname", ["F16", "BF16"])
def test_split_on_one_gpu(b200, ctx, torch, tname, M, K, split):
    N, row_low = SPLITS[split]
    t = getattr(b200, tname)
    check_split(b200, ctx, torch, t, N, K, M, row_low, [0] * (len(row_low) - 1), seed=M * 131 + K + len(split) + t)


def profiled_split(b200, ctx, torch, t, M, K=4096):
    """kernel names in the profiler trace of one split over two shards on device 0, and its error against float64"""
    from torch.profiler import ProfilerActivity, profile
    N, row_low = SPLITS["two_at_768"]
    w, wd = rand_weights(torch, b200, t, N, K, 61 + M)
    x = torch.randn(M, K, device="cuda")
    sp, keep = shard_table(torch, w, row_low, [0, 0])
    out = torch.empty(M, N, dtype=torch.float32, device="cuda")
    op = mm_op(b200, t, C.addressof(sp), K, N, x, out, SPLIT)
    run(torch, ctx, op)                       # warm-up outside the trace (module load, scratch growth)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.compute_op(op)
        ctx.sync()
    want = x.to(w.dtype).double() @ wd.T
    return [e.name for e in prof.events()], max_err(out, want) / float(want.abs().max())


def split_traces():
    """profiled_split of every dispatch case, in a fresh process: after earlier profiler sessions in a long test process, CUDA kernel
    records can go missing (as in test_gpu_moe_float_weights.py)"""
    import torch
    from __graft_entry__ import load_package
    b200 = load_package()
    ctx = b200.Context(0)
    res = {}
    for tname in ("F16", "BF16"):
        for M in (1, 200):
            res["%s-%d" % (tname, M)] = profiled_split(b200, ctx, torch, getattr(b200, tname), M)
    ctx.set_option("cpu_exact", 1)
    for M in (1, 40):
        res["cpu_exact-%d" % M] = profiled_split(b200, ctx, torch, b200.F16, M)
    ctx.close()
    return res


@pytest.fixture(scope="module")
def traces():
    import json
    import subprocess
    code = "import json, sys; sys.path[:0] = [%r, %r]; import test_gpu_split_float_weights as T; print(json.dumps(T.split_traces()))" % (
        os.path.dirname(os.path.abspath(__file__)), ROOT)
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    return json.loads(p.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("M,kernel", [(1, "b200_gemv_f16_kernel"), (200, "b200_gemm_f16_tc_kernel")])
@pytest.mark.parametrize("tname", ["F16", "BF16"])
def test_split_reaches_tensor_core_kernels(traces, tname, M, kernel):
    names, rel = traces["%s-%d" % (tname, M)]
    assert rel <= BOUND, rel
    assert sum(kernel in n for n in names) >= 2, names          # one launch per shard
    assert not any("b200_mul_mat_float_kernel" in n for n in names), names


@pytest.mark.parametrize("M", [1, 40])
def test_split_cpu_exact_uses_float_kernel(traces, M):
    names, rel = traces["cpu_exact-%d" % M]
    assert rel <= BOUND, rel
    assert sum("b200_mul_mat_float_kernel" in n for n in names) >= 2, names
    assert not any("b200_gemv_f16_kernel" in n or "b200_gemm_f16_tc_kernel" in n for n in names), names


def need_gpus(torch, n=2):
    if torch.cuda.device_count() < n:
        pytest.skip("needs %d GPUs" % n)


@pytest.mark.parametrize("K", [4096, 1004])
@pytest.mark.parametrize("M", MS)
@pytest.mark.parametrize("tname", ["F16", "BF16"])
def test_split_over_all_gpus(b200, ctx, torch, tname, M, K):
    need_gpus(torch)
    n = torch.cuda.device_count()
    N = 1100 + 128 * n                  # the last shard's row count is not a multiple of 128
    row_low = [0] + [N * d // n // 128 * 128 for d in range(1, n)] + [N]      # the plugin's split_rows at equal fractions
    for rep in range(2):                # the second pass reuses the peer contexts
        check_split(b200, ctx, torch, getattr(b200, tname), N, K, M, row_low, list(range(n)), seed=71 + M + K + rep)


# ---------------------------------------------------------------------------------------------------------- Megatron form, bf16
MEGATRON_SCHEDULE = [(40, 0), (1, 40), (3, 41)]      # a prompt ubatch (gemm_f16_tc), then decode steps (gemv_f16)


def megatron_graph(b200, rank, world, device=0):
    from __graft_entry__ import load_llama_graph
    return load_llama_graph().LlamaGraph(b200, model="llama3-8b", ftype="bf16", kv="f16", n_ctx=256, layers=2, max_tokens=40,
                                         device=device, tp_rank=rank, tp_world=world)


def upload(torch, g, emb, pos, mask, T):
    g.inp_embd[:T * g.E] = torch.from_numpy(emb.reshape(-1)).to(g.dev)
    g.pos[:T] = torch.from_numpy(pos).to(g.dev)
    g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).to(g.dev)
    torch.cuda.synchronize(g.dev)


def f32_at(torch, g, ptr, n):
    """the n floats at device address ptr inside one of g's f32 buffers"""
    for b in g.keep:
        if b.dtype == torch.float32 and b.data_ptr() <= ptr < b.data_ptr() + 4 * b.numel():
            o = (ptr - b.data_ptr()) // 4
            return b[o:o + n]
    raise AssertionError("no buffer at 0x%x" % ptr)


def test_megatron_bf16_shards_on_one_gpu(b200, ctx, torch):
    """Both ranks of a TP=2 bf16 model on one GPU, op by op, with each B200_OP_ALLREDUCE done by torch in the kernel's order (rank 0 +
    rank 1, then the residual): the row- and K-split 16-bit shards must give the TP=1 logits within the fast-mode envelope."""
    ranks = [megatron_graph(b200, r, 2) for r in range(2)]
    ref = megatron_graph(b200, 0, 1)
    rng = np.random.default_rng(13)
    worst = 0.0
    for T, kv_head in MEGATRON_SCHEDULE:
        emb, pos, mask = ref.set_inputs_host(T, kv_head, 256, rng)
        for g in ranks + [ref]:
            upload(torch, g, emb, pos, mask, T)
        ctx.compute(ref.build(T, kv_head, 256))
        ctx.sync()
        for ops in zip(*[g.build(T, kv_head, 256) for g in ranks]):
            if ops[0].op != b200.OP_ALLREDUCE:
                for op in ops:
                    ctx.compute_op(op)
                continue
            ctx.sync()
            n = ops[0].src[0].ne[0] * ops[0].src[0].ne[1]
            total = f32_at(torch, ranks[0], ops[0].src[0].data, n) + f32_at(torch, ranks[1], ops[1].src[0].data, n)
            for g, op in zip(ranks, ops):
                f32_at(torch, g, op.dst.data, n).copy_(total + f32_at(torch, g, op.src[1].data, n))
            torch.cuda.synchronize()
        ctx.sync()
        got = [g.logits[:T * g.V].cpu().numpy().reshape(T, g.V) for g in ranks]
        want = ref.logits[:T * ref.V].cpu().numpy().reshape(T, ref.V)
        assert np.isfinite(got[0]).all() and np.array_equal(got[0], got[1])
        rel = float((np.abs(got[0] - want).max(axis=1) / np.abs(want).max(axis=1)).max())
        worst = max(worst, rel)
        assert rel <= FAST_MODE_BOUND, (T, rel)
    print("bf16 TP=2 on one GPU vs TP=1: worst row %.3g of the largest logit" % worst)


def _megatron_worker(rank, world, port, q):
    try:
        sys.path.insert(0, ROOT)
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import torch
        import torch.distributed as dist
        from __graft_entry__ import load_package
        torch.cuda.set_device(rank)
        dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
        b200 = load_package()
        ctx = b200.Context(rank)

        def exchange(blob):
            out = [None] * world
            dist.all_gather_object(out, blob)
            return out
        ctx.comm_init(rank, world, exchange)
        g = megatron_graph(b200, rank, world, device=rank)
        ref = megatron_graph(b200, 0, 1, device=rank) if rank == 0 else None
        ctx1 = b200.Context(rank) if rank == 0 else None
        rng = np.random.default_rng(11)
        worst, same_ranks = 0.0, True
        for T, kv_head in MEGATRON_SCHEDULE:
            emb, pos, mask = g.set_inputs_host(T, kv_head, 256, rng)
            for m in (g, ref):
                if m is not None:
                    upload(torch, m, emb, pos, mask, T)
            ctx.compute(g.build(T, kv_head, 256))
            ctx.sync()
            got = g.logits[:T * g.V].cpu()
            both = [torch.empty_like(got) for _ in range(world)]
            dist.all_gather(both, got)
            same_ranks &= all(torch.equal(both[0], b) for b in both)
            if rank == 0:
                ctx1.compute(ref.build(T, kv_head, 256))
                ctx1.sync()
                want = ref.logits[:T * ref.V].cpu().numpy().reshape(T, ref.V)
                gotn = got.numpy().reshape(T, g.V)
                worst = max(worst, float((np.abs(gotn - want).max(axis=1) / np.abs(want).max(axis=1)).max()))
        dist.barrier()
        ctx.close()
        if ctx1 is not None:
            ctx1.close()
        dist.destroy_process_group()
        q.put((rank, "ok", worst, same_ranks))
    except Exception as ex:      # surface the failure in the parent instead of a hang
        import traceback
        q.put((rank, "error: %s\n%s" % (ex, traceback.format_exc()), 0.0, False))


def test_megatron_bf16_tp2_matches_tp1(torch):
    need_gpus(torch)
    import torch.multiprocessing as mp
    mpc = mp.get_context("spawn")
    q = mpc.Queue()
    port = 29600 + (os.getpid() + 517) % 2000
    ps = [mpc.Process(target=_megatron_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = sorted(q.get(timeout=600) for _ in ps)
    for p in ps:
        p.join(60)
    for r in res:
        assert r[1] == "ok", r[1]
        assert r[3], "logits differ between ranks"
    assert res[0][2] <= FAST_MODE_BOUND, "TP=2 vs TP=1 logits: rel %.3g" % res[0][2]


# ---------------------------------------------------------------------------------------------------------- through llama.cpp
def test_split_mode_row_bf16_through_llama_cpp(torch):
    """llama.cpp's --split-mode row on a bf16 GGUF allocates the 16-bit weights in the plugin's split buffer type; the logits stay
    within the fast-mode envelope of the one-GPU run."""
    need_gpus(torch)
    import test_gpu_reference_parity as P
    P.need_tools()
    gguf = P.gguf_for("llama3-8b", "bf16", 2)
    row, _, err = P.dump(gguf, "split_bf16_row", 99, 32, 24, "f16", False, 10, {"LOGITS_DUMP_SPLIT_MODE": "row"})
    assert "_Split" in err, "llama.cpp did not allocate the weights in the split buffer type:\n" + err[-1500:]
    one, _, _ = P.dump(gguf, "split_bf16_one", 99, 32, 24, "f16", False, 10, {"LOGITS_DUMP_SPLIT_MODE": "none"})
    assert np.isfinite(row).all() and row.shape == one.shape
    rel = P.rel_err(one, row)
    print("bf16 split-mode row vs none: max rel %.3g" % float(rel.max()))
    assert rel.max() <= FAST_MODE_BOUND
