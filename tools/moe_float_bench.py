"""F16 / BF16 MoE expert matmuls (MUL_MAT_ID) on the B200: per-op timing on Mixtral-8x7B expert shapes, the streaming / GEMM crossover,
whole-model Mixtral-8x7B bf16 steps, and the quantised bench.py value.

    python tools/moe_float_bench.py --out DIR [--no-model] [--no-bench] [--quick]

1. Per op: up/gate (N 14336, K 4096) and down (N 4096, K 14336), 8 experts, top-2, f16 and bf16, n_tok tokens, balanced and skewed
   routing: b200_op_compute of one MUL_MAT_ID timed with CUDA events after warm-up, two expert stacks (940 MB each) alternated, so every
   timed launch reads its experts from HBM (even bs1 reads 2 x 117 MB > the 126 MB L2).  Algorithmic bytes = live experts x N K 2 +
   f32 activations in and out; FLOPs = 2 N K pairs.  Compared with
     - the dense kernels on one expert matrix at M = pairs per live expert, times the live experts (the ceiling grouping approaches);
     - a torch/cuBLAS MoE with ids copied to the host and a host loop over experts (gather + F.linear), as ggml-cuda does.
2. Crossover: the same routing over 8 live experts through a view of 8 experts (grouped GEMM from 32 x 8 = 256 pairs) and a view of 16
   (streaming kernel below 512 pairs), at 128..224 tokens: both kernels on identical work.
3. LlamaGraph("mixtral") bf16 through b200_graph_compute: bs1 decode at depth 512 with CUDA-graph replay, a 32-slot step and a 512-token
   prompt ubatch, next to the byte ceiling (weights with only the routed experts' share of the expert bytes, KV, activations).
4. `python bench.py --no-cpu` (the quantised flagship) in the same call, compared with profiles/r2_bench.json.
Writes DIR/moe_float_weights.jsonl and DIR/moe_float_weights.md; the card name and power limit come first."""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SHAPES = [("up", 14336, 4096), ("down", 4096, 14336)]        # (name, N rows, K)
N_TOKS = [1, 2, 4, 8, 16, 32, 64, 128, 512]
CROSS_TOKS = [128, 160, 192, 224]
E, NU = 8, 2
SKEW = np.array([10, 4, 2, 1, 1, 0.5, 0.5, 0.2])


def peaks():
    hbm, bf16, src = 6561.0, 1631.8, "DESIGN.md section 4 (measured copy / bf16 burst)"
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        hbm, bf16, src = float(d.get("hbm_gbs", hbm)), float(d.get("bf16_tflops", bf16)), "MEASURED_PEAKS.json"
    return hbm, bf16, src


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip()


def routing(rng, n_tok, skew):
    p = SKEW / SKEW.sum() if skew else None
    return np.stack([np.concatenate([c := rng.choice(E, NU, replace=False, p=p), np.setdiff1d(np.arange(E), c)]) for _ in range(n_tok)]).astype(np.int32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--no-model", action="store_true")
    ap.add_argument("--no-bench", action="store_true")
    ap.add_argument("--quick", action="store_true", help="bf16, balanced routing, 3 token counts (rehearsal)")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    import torch
    import torch.nn.functional as F
    from __graft_entry__ import load_llama_graph, load_package
    b200 = load_package()
    L = b200.lib()
    assert torch.cuda.is_available(), "needs the GPU"
    hbm, bf16, peak_src = peaks()
    info = {"card": card(), "hbm_peak_gbs": hbm, "bf16_peak_tflops": bf16, "peak_source": peak_src,
            "l2_note": "two 940 MB expert stacks alternated; the routed experts of one launch alone exceed the 126 MB L2"}
    print("card (name, power limit, max SM clock): %s" % info["card"])
    print("peaks: HBM %.0f GB/s, bf16 %.1f TFLOP/s (%s)" % (hbm, bf16, peak_src))
    log = open(os.path.join(a.out, "moe_float_weights.jsonl"), "w")
    log.write(json.dumps(info) + "\n")
    md = ["# F16 / BF16 MoE expert matmuls (MUL_MAT_ID)", "", "Card (name, power limit, max SM clock): %s. Peaks: HBM %.0f GB/s, bf16 %.1f TFLOP/s (%s)." % (
        info["card"], hbm, bf16, peak_src), "", "Produced by `tools/moe_float_bench.py`. Expert buffers: " + info["l2_note"] + ".", ""]
    ctx = b200.Context(0)
    e0, e1 = L.b200_event_create(0), L.b200_event_create(0)

    def time_ops(ops, reps, warm):
        for i in range(warm):
            ctx.compute_op(ops[i % len(ops)])
        ctx.sync()
        L.b200_event_record(ctx.h, e0)
        for i in range(reps):
            ctx.compute_op(ops[i % len(ops)])
        L.b200_event_record(ctx.h, e1)
        L.b200_event_synchronize(e1)
        return L.b200_event_elapsed_ms(e0, e1) * 1e3 / reps

    def moe_op(t, A, n_exp, K, N, x, sel, out, n_tok):
        es = 2
        return b200.make_op(b200.OP_MUL_MAT_ID, b200.tensor(out.data_ptr(), b200.F32, [N, NU, n_tok]),
                            [b200.tensor(A.data_ptr(), t, [K, N, n_exp], nb=[es, K * es, K * es * N, K * es * N * n_exp], flags=b200.TENSOR_FLAG_WEIGHT),
                             b200.tensor(x.data_ptr(), b200.F32, [K, 1, n_tok]),
                             b200.tensor(sel.data_ptr(), b200.I32, [NU, n_tok], [4, E * 4, E * 4 * n_tok, E * 4 * n_tok])])

    types = (("bf16", b200.BF16, torch.bfloat16),) if a.quick else (("bf16", b200.BF16, torch.bfloat16), ("f16", b200.F16, torch.float16))
    toks = [1, 32, 512] if a.quick else N_TOKS
    md += ["## Per op (8 experts, top-2)", "",
           "| type | matrix | tokens | routing | live | µs | GB/s | HBM share | TFLOP/s | bf16 share | dense ceiling µs | grouped / dense | torch host loop µs | torch / ours |",
           "|---|---|---|---|---|---|---|---|---|---|---|---|---|---|"]
    for ftype, t, dt in types:
        for name, N, K in SHAPES:
            stacks = [((torch.rand(E, N, K, device="cuda") * 2 - 1) * 0.02).to(dt) for _ in range(2)]
            for n_tok in toks:
                for skew in ((False,) if a.quick else (False, True)):
                    rng = np.random.default_rng(n_tok + 7 * skew)
                    sel_h = routing(rng, n_tok, skew)
                    ids_h = sel_h[:, :NU]
                    sel = torch.from_numpy(sel_h).cuda()
                    x = torch.randn(n_tok, K, device="cuda")
                    out = torch.empty(n_tok, NU, N, device="cuda")
                    ops = [moe_op(t, A, E, K, N, x, sel, out, n_tok) for A in stacks]
                    torch.cuda.synchronize()
                    us = time_ops(ops, 40, 4)
                    # correctness of the timed output against float64 of the rounded operands
                    A = stacks[(40 - 1) % 2].double()
                    xr = x.to(dt).double()
                    ref = torch.zeros(n_tok, NU, N, dtype=torch.float64, device="cuda")
                    for s in range(NU):
                        for e in range(E):
                            m = torch.from_numpy(ids_h[:, s] == e).cuda()
                            if bool(m.any()):
                                ref[m, s] = xr[m] @ A[e].T
                    del A
                    rel = float((out.double() - ref).abs().max() / ref.abs().max())
                    counts = np.bincount(ids_h.reshape(-1), minlength=E)
                    live = int((counts > 0).sum())
                    npairs = n_tok * NU
                    byts = live * N * K * 2 + 4 * n_tok * K + 4 * npairs * N
                    flops = 2.0 * N * K * npairs
                    # dense ceiling: one expert matrix at M = pairs per live expert, rotated over the 8 experts of a stack, times the live experts
                    Md = int(math.ceil(npairs / live))
                    xd = torch.randn(Md, K, device="cuda")
                    od = torch.empty(Md, N, device="cuda")
                    dops = [b200.make_op(b200.OP_MUL_MAT, b200.tensor(od.data_ptr(), b200.F32, [N, Md]),
                                         [b200.tensor(stacks[0][e].data_ptr(), t, [K, N], flags=b200.TENSOR_FLAG_WEIGHT), b200.tensor(xd.data_ptr(), b200.F32, [K, Md])])
                            for e in range(E)]
                    torch.cuda.synchronize()
                    us_dense = time_ops(dops, 40, 8) * live
                    # torch/cuBLAS MoE: ids to the host, loop over experts (gather, F.linear on rounded operands, scatter)
                    def torch_moe(Ast):
                        idh = sel[:, :NU].cpu().numpy()
                        xr16 = x.to(dt)
                        res = torch.empty(n_tok, NU, N, device="cuda", dtype=dt)
                        for e in range(E):
                            tt, ss = np.nonzero(idh == e)
                            if tt.size:
                                ti, si = torch.from_numpy(tt).cuda(), torch.from_numpy(ss).cuda()
                                res[ti, si] = F.linear(xr16[ti], Ast[e])
                        return res
                    for i in range(2):
                        torch_moe(stacks[i])
                    torch.cuda.synchronize()
                    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s0.record()
                    for i in range(10):
                        torch_moe(stacks[i % 2])
                    s1.record()
                    torch.cuda.synchronize()
                    us_torch = s0.elapsed_time(s1) * 1e3 / 10
                    rec = {"ftype": ftype, "matrix": name, "N": N, "K": K, "n_tok": n_tok, "routing": "skewed" if skew else "balanced", "live_experts": live,
                           "pairs_per_expert_max": int(counts.max()), "kernel": "gemm_f16_tc_grouped" if npairs >= 32 * E else "gemv_f16_grouped", "us": us,
                           "bytes": byts, "gbs": byts / us / 1e3, "hbm_frac": byts / us / 1e3 / hbm, "tflops": flops / us / 1e6, "bf16_frac": flops / us / 1e6 / bf16,
                           "us_dense_ceiling": us_dense, "dense_M": Md, "grouped_over_dense_time": us / us_dense, "us_torch_host_loop": us_torch,
                           "torch_over_ours": us_torch / us, "max_rel_err_vs_f64": rel}
                    log.write(json.dumps(rec) + "\n"); log.flush()
                    line = "| %s | %s %dx%d | %d | %s | %d | %.1f | %.0f | %.2f | %.1f | %.3f | %.1f | %.2f | %.1f | %.1f |" % (
                        ftype, name, N, K, n_tok, rec["routing"], live, us, rec["gbs"], rec["hbm_frac"], rec["tflops"], rec["bf16_frac"], us_dense,
                        us / us_dense, us_torch, us_torch / us)
                    md.append(line)
                    print(line, " err %.1e" % rel, rec["kernel"])
            del stacks
            torch.cuda.empty_cache()

    # ---- crossover: identical work through the GEMM (8-expert view) and the streaming kernel (16-expert view of a 16-expert stack)
    md += ["", "## Streaming vs GEMM on identical work (bf16, balanced routing over 8 experts)", "",
           "| matrix | tokens | pairs | grouped GEMM µs (8-expert view) | streaming µs (16-expert view) | streaming / GEMM |", "|---|---|---|---|---|---|"]
    for name, N, K in SHAPES:
        A16 = ((torch.rand(2 * E, N, K, device="cuda") * 2 - 1) * 0.02).to(torch.bfloat16)
        for n_tok in ([128, 192] if a.quick else CROSS_TOKS):
            sel = torch.from_numpy(routing(np.random.default_rng(n_tok), n_tok, False)).cuda()
            x = torch.randn(n_tok, K, device="cuda")
            o1, o2 = torch.empty(n_tok, NU, N, device="cuda"), torch.empty(n_tok, NU, N, device="cuda")
            op8, op16 = moe_op(b200.BF16, A16, E, K, N, x, sel, o1, n_tok), moe_op(b200.BF16, A16, 2 * E, K, N, x, sel, o2, n_tok)
            torch.cuda.synchronize()
            us8, us16 = time_ops([op8], 30, 3), time_ops([op16], 30, 3)
            same = bool(torch.allclose(o1, o2, rtol=1e-4, atol=1e-4 * float(o1.abs().max())))
            rec = {"crossover": True, "matrix": name, "n_tok": n_tok, "pairs": n_tok * NU, "us_gemm": us8, "us_stream": us16, "stream_over_gemm": us16 / us8,
                   "outputs_agree": same}
            log.write(json.dumps(rec) + "\n"); log.flush()
            line = "| %s | %d | %d | %.1f | %.1f | %.2f |" % (name, n_tok, n_tok * NU, us8, us16, us16 / us8)
            md.append(line)
            print(line, "agree" if same else "OUTPUTS DIFFER")
        del A16
        torch.cuda.empty_cache()

    if not a.no_model:
        lg = load_llama_graph()
        slots, depth, PP = 32, 512, 512
        n_ctx = ((slots * depth + slots + 255) // 256 + 1) * 256
        g = lg.LlamaGraph(b200, model="mixtral", ftype="bf16", kv="f16", n_ctx=n_ctx, max_tokens=PP)
        g.fill_cache(slots * depth)
        rng = np.random.default_rng(1)

        def upload(emb, pos, mask, T):
            g.inp_embd[:T * g.E] = torch.from_numpy(emb.reshape(-1)).cuda()
            g.pos[:T] = torch.from_numpy(pos).cuda()
            g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).cuda()
            torch.cuda.synchronize()

        def timed(ops, reps, warm):
            arr = (b200.Op * len(ops))(*ops)
            n0 = ctx.launches()
            b200.check(L.b200_graph_compute(ctx.h, arr, len(ops)), "step"); ctx.sync()
            launches = ctx.launches() - n0
            for _ in range(warm):
                b200.check(L.b200_graph_compute(ctx.h, arr, len(ops)), "step")
            ctx.sync()
            n1 = ctx.launches()
            L.b200_event_record(ctx.h, e0)
            for _ in range(reps):
                b200.check(L.b200_graph_compute(ctx.h, arr, len(ops)), "step")
            L.b200_event_record(ctx.h, e1)
            L.b200_event_synchronize(e1)
            return L.b200_event_elapsed_ms(e0, e1) / reps, int(launches), (ctx.launches() - n1) / reps

        def ceiling_bytes(n_tok, n_kv, live_frac):
            sb = g.step_bytes(n_tok, n_kv)
            return sb["total"] - g.expert_bytes * (1.0 - live_frac)

        ctx.set_option("fusion", 2)
        res = {"ftype": "bf16", "model": "mixtral", "weight_bytes": g.weight_bytes, "expert_bytes": g.expert_bytes}
        ctx.set_option("cuda_graphs", 1)
        n_kv = (depth + 1 + 255) // 256 * 256
        emb, pos, mask = g.set_inputs_host(1, depth, n_kv, rng)
        upload(emb, pos, mask, 1)
        ms, launches, per_rep = timed(g.build(1, depth, n_kv), 30, 5)
        sb = ceiling_bytes(1, n_kv, NU / E)
        res["bs1_decode"] = {"tok_s": 1e3 / ms, "ms": ms, "launches_eager": launches, "launches_per_timed_step": per_rep, "bytes": sb,
                             "ceiling_tok_s": hbm * 1e9 / sb, "hbm_frac": sb / (ms / 1e3) / 1e9 / hbm, "finite": bool(torch.isfinite(g.logits[:g.V]).all().item())}
        n_kv = (slots * depth + slots + 255) // 256 * 256
        emb, pos, mask, kv_head = g.set_inputs_slots_host(slots, depth, n_kv, rng)
        upload(emb, pos, mask, slots)
        ms, launches, per_rep = timed(g.build(slots, kv_head, n_kv), 10, 3)
        sb = ceiling_bytes(slots, n_kv, 1.0)
        res["bs32_step"] = {"tok_s": slots * 1e3 / ms, "ms": ms, "launches_eager": launches, "launches_per_timed_step": per_rep, "bytes": sb,
                            "ceiling_tok_s": slots * hbm * 1e9 / sb, "finite": bool(torch.isfinite(g.logits[:slots * g.V]).all().item())}
        ctx.set_option("cuda_graphs", 0)
        emb, pos, mask = g.set_inputs_host(PP, 0, PP, rng)
        upload(emb, pos, mask, PP)
        ms, launches, _ = timed(g.build(PP, 0, PP, n_outputs=1), 5, 2)
        dense_w = (g.weight_bytes - g.expert_bytes) / 2 + g.expert_bytes / 2 * NU / E        # parameters each token multiplies
        flops = 2.0 * dense_w * PP - 2.0 * g.V * g.E * (PP - 1) + 4.0 * g.L * g.H * g.D * PP * PP / 2
        res["pp512"] = {"tok_s": PP * 1e3 / ms, "ms": ms, "launches": launches, "flops": flops, "tflops": flops / (ms / 1e3) / 1e12,
                        "bf16_frac": flops / (ms / 1e3) / 1e12 / bf16, "finite": bool(torch.isfinite(g.logits[:g.V]).all().item())}
        log.write(json.dumps(res) + "\n"); log.flush()
        b1, b32, pp = res["bs1_decode"], res["bs32_step"], res["pp512"]
        md += ["", "## Mixtral-8x7B bf16 (32 layers, random weights) through b200_graph_compute", "",
               "| step | tok/s | ms | byte ceiling tok/s (arithmetic) | notes |", "|---|---|---|---|---|",
               "| bs1 decode, depth 512, graph replay | %.1f | %.2f | %.0f (%.1f GB/token) | %.2f of HBM peak; %d launches eager, %.0f per replayed step |" % (
                   b1["tok_s"], b1["ms"], b1["ceiling_tok_s"], b1["bytes"] / 1e9, b1["hbm_frac"], b1["launches_eager"], b1["launches_per_timed_step"]),
               "| 32-slot step, depth 512 | %.0f | %.2f | %.0f | %d launches eager, %.0f per timed step |" % (
                   b32["tok_s"], b32["ms"], b32["ceiling_tok_s"], b32["launches_eager"], b32["launches_per_timed_step"]),
               "| 512-token prompt ubatch | %.0f | %.2f | - | %.0f TFLOP/s = %.2f of the bf16 peak; %d launches |" % (
                   pp["tok_s"], pp["ms"], pp["tflops"], pp["bf16_frac"], pp["launches"])]
        print("\n".join(md[-5:]), "finite", b1["finite"], b32["finite"], pp["finite"])
        g.keep.clear(); g.layers.clear()
        del g
        torch.cuda.empty_cache()
    ctx.close()

    if not a.no_bench:
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--no-cpu"], capture_output=True, text=True, cwd=ROOT)
        line = [ln for ln in out.stdout.strip().splitlines() if ln.startswith("{")]
        assert out.returncode == 0 and line, out.stderr[-3000:]
        cur = json.loads(line[-1])
        last = json.loads(open(os.path.join(ROOT, "profiles", "r2_bench.json")).readline())
        d = cur["value"] / last["value"] - 1
        rec = {"bench_py_no_cpu": cur["value"], "unit": cur.get("unit"), "recorded_r2": last["value"], "rel_change": d}
        log.write(json.dumps(rec) + "\n")
        md += ["", "## Quantised flagship", "", "`bench.py --no-cpu`: %.1f %s vs %.1f recorded in profiles/r2_bench.json (%+.2f%%)." % (
            cur["value"], cur.get("unit"), last["value"], 100 * d)]
        print(md[-1])
    log.close()
    open(os.path.join(a.out, "moe_float_weights.md"), "w").write("\n".join(md) + "\n")


if __name__ == "__main__":
    main()
