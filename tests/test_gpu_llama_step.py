"""GPU parity of whole llama ubatches through b200_graph_compute (the op list the ggml backend forwards) against the CPU
oracle forward (oracle/llama_forward.py), with and without the decode layer fusions, for every KV-cache type.
Two modes: cpu-exact (bit-identical logits, hence identical greedy tokens) and the default fast mode (bounded by the reference's
own cross-build reproducibility); see FAST_MODE_BOUND."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def run_steps(b200, ctx, g, schedule, rng, fusion, graphs=0):
    import torch
    import llama_forward as OF
    ctx.set_option("fusion", fusion)
    ctx.set_option("cuda_graphs", graphs)
    caches = None
    outs = []
    for T, kv_head in schedule:
        n_kv = 256
        emb, pos, mask = g.set_inputs_host(T, kv_head, n_kv, rng)
        g.inp_embd[:T * g.E] = torch.from_numpy(emb.reshape(-1)).cuda()
        g.pos[:T] = torch.from_numpy(pos).cuda()
        g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).cuda()
        torch.cuda.synchronize()
        want, caches = OF.forward(g, emb, pos, mask, kv_head, n_kv, caches=caches)
        n0 = ctx.launches()
        ctx.compute(g.build(T, kv_head, n_kv))
        ctx.sync()
        got = g.logits[:T * g.V].cpu().numpy().reshape(T, g.V).copy()
        outs.append((got, want, ctx.launches() - n0))
    return outs


CASES = [("tiny-d128", f, k) for f in ["q4_k_m", "q4_0", "q5_k_m", "q8_0"] for k in ["f16", "q8_0", "q4_0"]] + [("mid-d128", "q4_k_m", "q8_0"), ("mid-d128", "q4_k_m", "f16")]
MOE_CASES = [("tiny-moe", "q4_k_m", "q8_0"), ("tiny-moe", "q4_0", "f16"), ("tiny-moe", "q5_k_m", "q4_0")]   # Mixtral-shaped: 4 experts, 2 used
SCHEDULE = [(5, 0), (1, 5), (2, 6), (4, 8), (1, 12), (3, 13)]        # prompt chunk, then decode-sized ubatches (1..4 tokens)
# Fast-mode bound.  The fast kernels compute the CPU's integers exactly but add the per-block float terms in their own order; the
# reference pipeline is chaotic at that level (a 1e-7 difference flips a q8 rounding in the next matmul, each flip is 1/127 of a
# block maximum, the error grows ~sqrt per matmul and saturates): two builds of the REFERENCE ITSELF (AVX2 vs SSE4.2, same
# sources, same host) differ by max 1.6e-2 (2 layers) .. 3.7e-2 (22 layers) of the largest logit, mean 0.9e-2 .. 2.8e-2
# (profiles/r2_reference_cross_build.md, tools/ref_cross_build.sh).  The fast mode is held to that same envelope; the strict
# check is the cpu-exact mode below, which must reproduce the oracle (= the reference, tests/test_oracle_pin.py) bit for bit.
FAST_MODE_BOUND = 4e-2


def margin(row):
    part = np.partition(row, row.size - 2)
    return (part[-1] - part[-2]) / np.abs(row).max()


@pytest.mark.parametrize("model,ftype,kv", CASES + MOE_CASES)
def test_llama_steps_cpu_exact_mode_bit_identical_to_oracle(b200, ctx, model, ftype, kv):
    """option cpu_exact: whole ubatches (prompt chunk + decode steps, every weight format and KV type) must equal the CPU oracle
    forward BIT FOR BIT -- logits identical, hence greedy tokens identical -- because every float sum follows the reference
    build's order (exact.cu, fattn.cu b200_fattn_f16acc_kernel, restated glibc sinf/cosf/expf and ggml_v_expf)."""
    from __graft_entry__ import load_llama_graph
    lg = load_llama_graph()
    g = lg.LlamaGraph(b200, model=model, ftype=ftype, kv=kv, n_ctx=256, max_tokens=5)
    ctx.set_option("cpu_exact", 1)
    try:
        outs = run_steps(b200, ctx, g, SCHEDULE, np.random.default_rng(5), 2)
    finally:
        ctx.set_option("cpu_exact", 0)
    for (got, want, _), (T, _) in zip(outs, SCHEDULE):
        assert np.isfinite(got).all()
        assert np.array_equal(got, want), (T, float(np.abs(got - want).max() / np.abs(want).max()))
        assert (got.argmax(1) == want.argmax(1)).all()


@pytest.mark.parametrize("model,ftype,kv", CASES)
def test_llama_steps_fast_mode_fused_and_unfused(b200, ctx, model, ftype, kv):
    """default (fast) mode, with and without the decode layer fusions: logits inside the reference's own cross-build envelope
    (see FAST_MODE_BOUND), greedy token identical wherever the oracle's top-1/top-2 margin exceeds twice the row's difference,
    fused path really fewer launches"""
    from __graft_entry__ import load_llama_graph
    lg = load_llama_graph()
    g = lg.LlamaGraph(b200, model=model, ftype=ftype, kv=kv, n_ctx=256, max_tokens=5)
    res = {}
    for fusion in (0, 2):
        for lw in g.layers:
            lw["k_cache"].zero_(); lw["v_cache"].zero_()
        res[fusion] = run_steps(b200, ctx, g, SCHEDULE, np.random.default_rng(5), fusion)
    worst = 0.0
    for fusion in (0, 2):
        for (got, want, _), (T, _) in zip(res[fusion], SCHEDULE):
            assert np.isfinite(got).all()
            for r in range(T):
                rel = float(np.abs(got[r] - want[r]).max() / np.abs(want[r]).max())
                worst = max(worst, rel)
                assert rel <= FAST_MODE_BOUND, (fusion, T, r, rel)
                if got[r].argmax() != want[r].argmax():
                    assert margin(want[r]) <= 2 * rel, (fusion, T, r, rel, margin(want[r]))
    print("fast mode %s %s %s: worst row %.3g of the largest logit" % (model, ftype, kv, worst))
    for (a, _, la), (b, _, lb), (T, _) in zip(res[0], res[2], SCHEDULE):
        if T <= 4:
            assert lb < la, (T, la, lb)
    ctx.set_option("fusion", 2)


@pytest.mark.parametrize("model,ftype,kv", MOE_CASES)
def test_moe_steps_fast_mode(b200, ctx, model, ftype, kv):
    """Mixtral-shaped layers (build_moe_ffn op sequence) in the fast mode: per-pair GEMV routing for decode-sized ubatches, pairs grouped
    by expert on the device for the 5-token ubatch.  Rows whose router decision is a near-tie in the oracle are exempt from the bound
    (a different expert is a different function; the cpu-exact test above covers them bit for bit)."""
    import llama_forward as OF
    from __graft_entry__ import load_llama_graph
    lg = load_llama_graph()
    g = lg.LlamaGraph(b200, model=model, ftype=ftype, kv=kv, n_ctx=256, max_tokens=5)
    for fusion in (0, 2):
        for lw in g.layers:
            lw["k_cache"].zero_(); lw["v_cache"].zero_()
        OF.ROUTER_MARGINS.clear()
        outs = run_steps(b200, ctx, g, SCHEDULE, np.random.default_rng(5), fusion)
        margins = list(OF.ROUTER_MARGINS)                  # one entry per (ubatch, layer)
        checked = 0
        for si, ((got, want, _), (T, _)) in enumerate(zip(outs, SCHEDULE)):
            assert np.isfinite(got).all()
            tie = np.minimum.reduce(margins[si * g.L:(si + 1) * g.L]) < 0.02
            for r in range(T):
                if tie[r]:
                    continue
                rel = float(np.abs(got[r] - want[r]).max() / np.abs(want[r]).max())
                assert rel <= FAST_MODE_BOUND, (fusion, T, r, rel)
                checked += 1
        assert checked >= 10, "too many routing near-ties to say anything"
    ctx.set_option("fusion", 2)


def test_llama_decode_cuda_graph_replay(b200, ctx):
    """the same decode op list submitted repeatedly is captured once and replayed; results identical to eager"""
    import torch
    from __graft_entry__ import load_llama_graph
    lg = load_llama_graph()
    g = lg.LlamaGraph(b200, model="tiny-d128", ftype="q4_k_m", kv="q8_0", n_ctx=256, max_tokens=1)
    rng = np.random.default_rng(1)
    emb, pos, mask = g.set_inputs_host(1, 7, 256, rng)
    g.inp_embd[:g.E] = torch.from_numpy(emb.reshape(-1)).cuda()
    g.pos[:1] = torch.from_numpy(pos).cuda()
    g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).cuda()
    torch.cuda.synchronize()
    ops = g.build(1, 7, 256)
    ctx.set_option("cuda_graphs", 0)
    ctx.compute(ops); ctx.sync()
    eager = g.logits[:g.V].cpu().numpy().copy()
    ctx.set_option("cuda_graphs", 1)
    for pdl in (0, 1):
        ctx.set_option("pdl", pdl)
        g2 = g.build(1, 7 + pdl, 256)        # a different list per pdl setting (graphs are keyed on the op list)
        launches = []
        for _ in range(4):
            g.logits.zero_(); torch.cuda.synchronize()
            n0 = ctx.launches()
            ctx.compute(g2); ctx.sync()
            launches.append(ctx.launches() - n0)
            out = g.logits[:g.V].cpu().numpy()
            assert np.isfinite(out).all()
            if pdl == 0:
                assert np.abs(out - eager).max() <= 2e-5 * np.abs(eager).max()
        assert launches[-1] == 1 and launches[0] > 1, launches
    ctx.set_option("pdl", 0)
    ctx.set_option("cuda_graphs", 0)


@pytest.mark.parametrize("model,ftype", [("mid-d128", "q4_k_m"), ("tiny-d128", "q5_k_m"), ("tiny-d128", "q4_k_m")])
def test_ffn_pair_epilogue_bit_identical(b200, ctx, model, ftype):
    """option ffn_pair: the fused gate|up GEMV writes h = silu(gate) * up itself (gemv_bs1.cu pair mode: gate row parked in shared
    memory, picked up by the warp that finishes the up row) and the down GEMV reads h as plain f32 activations, instead of
    silu(gate) * up in the down GEMV's prologue -- same arithmetic (ggml_silu_lane, one rounded multiply): logits bit-identical,
    eager and under CUDA-graph replay"""
    import torch
    from __graft_entry__ import load_llama_graph
    lg = load_llama_graph()
    g = lg.LlamaGraph(b200, model=model, ftype=ftype, kv="f16", n_ctx=256, max_tokens=1)
    rng = np.random.default_rng(11)
    emb, pos, mask = g.set_inputs_host(1, 5, 256, rng)
    g.inp_embd[:g.E] = torch.from_numpy(emb.reshape(-1)).cuda()
    g.pos[:1] = torch.from_numpy(pos).cuda()
    g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).cuda()
    torch.cuda.synchronize()
    ops = g.build(1, 5, 256)
    ctx.set_option("fusion", 2); ctx.set_option("pdl", 1)
    outs = {}
    for graphs in (0, 1):
        ctx.set_option("cuda_graphs", graphs)
        for pair in (0, 1):
            ctx.set_option("ffn_pair", pair)
            for _ in range(3):
                g.logits.zero_(); torch.cuda.synchronize()
                ctx.compute(ops); ctx.sync()
            outs[(graphs, pair)] = g.logits[:g.V].cpu().numpy().copy()
    ctx.set_option("ffn_pair", 1); ctx.set_option("pdl", 0); ctx.set_option("cuda_graphs", 0)
    ref = outs[(0, 0)]
    assert np.isfinite(ref).all() and np.abs(ref).max() > 0
    for k, v in outs.items():
        assert np.array_equal(ref, v), k


def test_l2_lookahead_modes_do_not_change_results(b200, ctx):
    """option l2_prefetch (0 off, 1 next matmul with the first copies, 2 following launches' ranges after the launch's own copies, across
    the attention chain): a pure L2 hint -- logits bit-identical in every mode (gemv_bs1.cu bs1_l2_lookahead, graph.cu look-ahead pass)"""
    import torch
    from __graft_entry__ import load_llama_graph
    lg = load_llama_graph()
    g = lg.LlamaGraph(b200, model="mid-d128", ftype="q4_k_m", kv="f16", n_ctx=256, max_tokens=1)
    rng = np.random.default_rng(5)
    emb, pos, mask = g.set_inputs_host(1, 9, 256, rng)
    g.inp_embd[:g.E] = torch.from_numpy(emb.reshape(-1)).cuda()
    g.pos[:1] = torch.from_numpy(pos).cuda()
    g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).cuda()
    torch.cuda.synchronize()
    ops = g.build(1, 9, 256)
    ctx.set_option("fusion", 2); ctx.set_option("pdl", 1); ctx.set_option("cuda_graphs", 0)
    outs = []
    for mode in (0, 1, 2):
        ctx.set_option("l2_prefetch", mode)
        g.logits.zero_(); torch.cuda.synchronize()
        ctx.compute(ops); ctx.sync()
        outs.append(g.logits[:g.V].cpu().numpy().copy())
    ctx.set_option("l2_prefetch", 0); ctx.set_option("pdl", 0)
    assert np.isfinite(outs[0]).all() and np.abs(outs[0]).max() > 0
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])


@pytest.mark.parametrize("kv", ["f16", "q8_0"])
def test_llama_decode_graph_replay_follows_kv_head(b200, ctx, kv):
    """a real decode loop: every step stores its K/V rows one cell further (the only thing that changes in llama.cpp's
    graph from token to token).  The captured graph must be REPLAYED (1 launch per step) with the new destinations patched
    in, and every step's logits must equal the eager run bit for bit -- a stale destination would corrupt the cache."""
    import torch
    from __graft_entry__ import load_llama_graph
    lg = load_llama_graph()
    g = lg.LlamaGraph(b200, model="tiny-d128", ftype="q4_k_m", kv=kv, n_ctx=256, max_tokens=4)
    ctx.set_option("fusion", 2)
    ctx.set_option("pdl", 1)
    outs = {}
    for graphs in (0, 1):
        ctx.set_option("cuda_graphs", graphs)
        for lw in g.layers:
            lw["k_cache"].zero_(); lw["v_cache"].zero_()
        rng = np.random.default_rng(3)
        seq, launches = [], []
        for step, (T, kv_head) in enumerate([(4, 0)] + [(1, 4 + i) for i in range(10)]):
            emb, pos, mask = g.set_inputs_host(T, kv_head, 256, rng)
            g.inp_embd[:T * g.E] = torch.from_numpy(emb.reshape(-1)).cuda()
            g.pos[:T] = torch.from_numpy(pos).cuda()
            g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).cuda()
            torch.cuda.synchronize()
            n0 = ctx.launches()
            ctx.compute(g.build(T, kv_head, 256)); ctx.sync()
            launches.append(ctx.launches() - n0)
            seq.append(g.logits[:T * g.V].cpu().numpy().copy())
        outs[graphs] = (seq, launches)
    for a, b in zip(outs[0][0], outs[1][0]):
        assert np.isfinite(a).all() and np.array_equal(a, b)
    assert all(n == 1 for n in outs[1][1][3:]), outs[1][1]          # prompt, first decode (eager), second (capture), then replays
    assert all(n > 1 for n in outs[0][1])
    ctx.set_option("pdl", 0)
    ctx.set_option("cuda_graphs", 0)


def test_graph_replay_survives_scratch_growth(b200, ctx):
    """ADVICE r1 (high): a captured graph bakes scratch pointers in; growing a scratch area (a later, larger ubatch) frees
    and reallocates it.  Replaying the earlier graph afterwards must not touch freed memory: capture a decode step at
    n_kv = 256, run a 64-token prompt ubatch and a decode step over the whole 2048-cell cache (both grow scratch areas),
    then submit the first op list again and compare with its eager result bit for bit."""
    import torch
    from __graft_entry__ import load_llama_graph
    lg = load_llama_graph()
    g = lg.LlamaGraph(b200, model="tiny-d128", ftype="q4_k_m", kv="f16", n_ctx=2048, max_tokens=64)
    rng = np.random.default_rng(9)

    def load(T, kv_head, n_kv):
        emb, pos, mask = g.set_inputs_host(T, kv_head, n_kv, rng)
        g.inp_embd[:T * g.E] = torch.from_numpy(emb.reshape(-1)).cuda()
        g.pos[:T] = torch.from_numpy(pos).cuda()
        g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).cuda()
        torch.cuda.synchronize()
        return emb, pos, mask
    g.fill_cache(2000)
    small = load(1, 100, 256)
    ops_small = g.build(1, 100, 256)
    ctx.set_option("fusion", 2); ctx.set_option("pdl", 1); ctx.set_option("cuda_graphs", 0)
    ctx.compute(ops_small); ctx.sync()
    eager = g.logits[:g.V].cpu().numpy().copy()
    ctx.set_option("cuda_graphs", 1)
    for _ in range(3):                                   # first sighting, capture, replay
        ctx.compute(ops_small); ctx.sync()
    assert np.array_equal(g.logits[:g.V].cpu().numpy(), eager)
    load(64, 1000, 1280)
    ctx.compute(g.build(64, 1000, 1280)); ctx.sync()      # prompt ubatch: activation scratch grows
    load(1, 1999, 2048)
    for _ in range(3):
        ctx.compute(g.build(1, 1999, 2048)); ctx.sync()   # long context: more KV splits
    # back to the first list (same inputs as at capture time)
    emb, pos, mask = small
    g.inp_embd[:g.E] = torch.from_numpy(emb.reshape(-1)).cuda()
    g.pos[:1] = torch.from_numpy(pos).cuda()
    g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).cuda()
    torch.cuda.synchronize()
    for _ in range(3):
        g.logits.zero_(); torch.cuda.synchronize()
        ctx.compute(ops_small); ctx.sync()
        assert np.array_equal(g.logits[:g.V].cpu().numpy(), eager)
    ctx.set_option("pdl", 0); ctx.set_option("cuda_graphs", 0)
