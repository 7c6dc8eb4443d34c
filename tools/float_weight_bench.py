"""F16 / BF16 weight matmuls on the B200: per-shape kernel timing, whole-model Llama-3-8B steps, and the quantised bench.py value.

    python tools/float_weight_bench.py --out DIR [--no-model] [--no-bench]

1. Per shape (the Llama-3-8B matrices) x M token columns x {f16, bf16}: b200_op_compute of one MUL_MAT timed with CUDA events after
   warm-up, weight buffers rotated so that the working set exceeds the 126 MB L2 (every timed launch reads its weights from HBM).
   Reported against the HBM and bf16 peaks (MEASURED_PEAKS.json when present, else the DESIGN.md section 4 values), with
   torch.nn.functional.linear (cuBLAS) on the same rounded operands as the bar, and the old warp-per-output float kernel (still
   reached through cpu_exact mode) at M = 1, 32 and 33.
2. LlamaGraph("llama3-8b") in bf16 and f16 through b200_graph_compute: bs1 decode at depth 512 with CUDA-graph replay, a 32-slot
   continuous-batching step and a 512-token prompt ubatch.
3. `python bench.py --no-cpu` (the quantised flagship) in the same process tree, compared with profiles/r2_bench.json.
Writes DIR/float_weights.jsonl (one JSON object per measurement) and prints a summary; the card name and power limit come first."""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SHAPES = [(4096, 4096), (1024, 4096), (14336, 4096), (4096, 14336), (128256, 4096)]      # (N rows, K)
MS = [1, 4, 8, 16, 32, 33, 64, 128, 512]
OLD_MS = (1, 32, 33)
L2_BYTES = 126 << 20


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--no-model", action="store_true")
    ap.add_argument("--no-bench", action="store_true")
    ap.add_argument("--shapes", default="all", help="'small': the first two shapes only (rehearsal)")
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
            "l2_note": "weight buffers rotated: working set > 2 x 126 MB L2 in every timed loop"}
    print("card (name, power limit, max SM clock): %s" % info["card"])
    print("peaks: HBM %.0f GB/s, bf16 %.1f TFLOP/s (%s)" % (hbm, bf16, peak_src))
    log = open(os.path.join(a.out, "float_weights.jsonl"), "w")
    log.write(json.dumps(info) + "\n")
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

    shapes = SHAPES if a.shapes == "all" else SHAPES[:2]
    for ftype, t, dt in (("bf16", b200.BF16, torch.bfloat16), ("f16", b200.F16, torch.float16)):
        for N, K in shapes:
            wbytes = 2 * N * K
            nbuf = max(2, math.ceil(2 * L2_BYTES / wbytes))
            ws = [((torch.rand(N, K, device="cuda") * 2 - 1) * 0.02).to(dt) for _ in range(nbuf)]
            for M in MS:
                x = torch.randn(M, K, device="cuda")
                xr = x.to(dt)
                out = torch.empty(M, N, device="cuda")
                ops = [b200.make_op(b200.OP_MUL_MAT, b200.tensor(out.data_ptr(), b200.F32, [N, M]),
                                    [b200.tensor(w.data_ptr(), t, [K, N], flags=b200.TENSOR_FLAG_WEIGHT), b200.tensor(x.data_ptr(), b200.F32, [K, M])]) for w in ws]
                torch.cuda.synchronize()
                us = time_ops(ops, max(20, 2 * nbuf), nbuf)
                got = out.clone()
                # cuBLAS on the same rounded operands (bf16/f16 output, f32 accumulate)
                for i in range(nbuf):
                    F.linear(xr, ws[i])
                torch.cuda.synchronize()
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                reps = max(20, 2 * nbuf)
                s0.record()
                for i in range(reps):
                    F.linear(xr, ws[i % nbuf])
                s1.record()
                torch.cuda.synchronize()
                us_cublas = s0.elapsed_time(s1) * 1e3 / reps
                ref = F.linear(xr.double(), ws[(max(20, 2 * nbuf) - 1) % nbuf].double()).float()
                rel = float((got - ref).abs().max() / ref.abs().max())
                us_old = None
                if M in OLD_MS:
                    ctx.set_option("cpu_exact", 1)
                    us_old = time_ops(ops[:1], 3, 1)
                    ctx.set_option("cpu_exact", 0)
                byts = wbytes + 4 * M * K + 4 * M * N
                flops = 2.0 * N * K * M
                t_min_bytes, t_min_flops = byts / (hbm * 1e9) * 1e6, flops / (bf16 * 1e12) * 1e6
                bound = "hbm" if t_min_bytes >= t_min_flops else "tensor"
                rec = {"ftype": ftype, "N": N, "K": K, "M": M, "kernel": "gemv_f16" if M <= 32 else "gemm_f16_tc", "us": us, "gbs": byts / us / 1e3,
                       "hbm_frac": byts / us / 1e3 / hbm, "tflops": flops / us / 1e6, "bf16_frac": flops / us / 1e6 / bf16, "bound": bound,
                       "frac_of_bound": max(t_min_bytes, t_min_flops) / us, "us_cublas": us_cublas, "vs_cublas": us_cublas / us, "us_old_float_kernel": us_old,
                       "max_rel_err_vs_f64": rel, "weight_buffers": nbuf}
                log.write(json.dumps(rec) + "\n"); log.flush()
                print("%-4s %6d x %5d M=%3d %-11s %9.1f us %7.0f GB/s (%.2f HBM) %7.1f TFLOP/s (%.3f bf16) [%s-bound %.2f]  cuBLAS %9.1f us (x%.2f)%s  err %.1e" % (
                    ftype, N, K, M, rec["kernel"], us, rec["gbs"], rec["hbm_frac"], rec["tflops"], rec["bf16_frac"], bound, rec["frac_of_bound"],
                    us_cublas, rec["vs_cublas"], "  old %9.1f us" % us_old if us_old else "", rel))
            del ws
            torch.cuda.empty_cache()

    if not a.no_model:
        lg = load_llama_graph()
        for ftype in ("bf16", "f16"):
            slots, depth, PP = 32, 512, 512
            n_ctx = ((slots * depth + slots + 255) // 256 + 1) * 256
            g = lg.LlamaGraph(b200, model="llama3-8b", ftype=ftype, kv="f16", n_ctx=n_ctx, max_tokens=PP)
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

            ctx.set_option("fusion", 2)
            res = {"ftype": ftype, "model": "llama3-8b", "weight_bytes": g.weight_bytes}
            # bs1 decode at depth 512, CUDA-graph replay
            ctx.set_option("cuda_graphs", 1)
            n_kv = (depth + 1 + 255) // 256 * 256
            emb, pos, mask = g.set_inputs_host(1, depth, n_kv, rng)
            upload(emb, pos, mask, 1)
            ms, launches, per_rep = timed(g.build(1, depth, n_kv), 50, 5)
            sb = g.step_bytes(1, n_kv)["total"]
            res["bs1_decode"] = {"tok_s": 1e3 / ms, "ms": ms, "launches_eager": launches, "launches_per_timed_step": per_rep, "bytes": sb,
                                 "ceiling_tok_s": hbm * 1e9 / sb, "hbm_frac": sb / (ms / 1e3) / 1e9 / hbm,
                                 "finite": bool(torch.isfinite(g.logits[:g.V]).all().item())}
            # 32-slot continuous-batching step
            n_kv = (slots * depth + slots + 255) // 256 * 256
            emb, pos, mask, kv_head = g.set_inputs_slots_host(slots, depth, n_kv, rng)
            upload(emb, pos, mask, slots)
            ms, launches, per_rep = timed(g.build(slots, kv_head, n_kv), 20, 3)
            kvb = 2 * g.L * slots * (depth + 1) * lg.row_size(g.kv_type, g.Hkv * g.D)
            res["bs32_step"] = {"tok_s": slots * 1e3 / ms, "ms": ms, "launches_eager": launches, "launches_per_timed_step": per_rep,
                                "bytes": g.weight_bytes + kvb, "ceiling_tok_s": slots * hbm * 1e9 / (g.weight_bytes + kvb),
                                "finite": bool(torch.isfinite(g.logits[:slots * g.V]).all().item())}
            # 512-token prompt ubatch (logits of the last token, as llama.cpp asks)
            ctx.set_option("cuda_graphs", 0)
            emb, pos, mask = g.set_inputs_host(PP, 0, PP, rng)
            upload(emb, pos, mask, PP)
            ms, launches, _ = timed(g.build(PP, 0, PP, n_outputs=1), 10, 2)
            flops = 2.0 * (g.weight_bytes / 2) * PP - 2.0 * g.V * g.E * (PP - 1) + 4.0 * g.L * g.H * g.D * PP * PP / 2
            res["pp512"] = {"tok_s": PP * 1e3 / ms, "ms": ms, "launches": launches, "flops": flops, "tflops": flops / (ms / 1e3) / 1e12,
                            "bf16_frac": flops / (ms / 1e3) / 1e12 / bf16, "ceiling_ms": flops / (bf16 * 1e12) * 1e3,
                            "finite": bool(torch.isfinite(g.logits[:g.V]).all().item())}
            log.write(json.dumps(res) + "\n"); log.flush()
            print("%s llama3-8b: bs1 decode %.1f tok/s (%.3f ms, ceiling %.0f tok/s, %.2f of HBM), bs32 %.0f tok/s (%.2f ms, ceiling %.0f), pp512 %.0f tok/s "
                  "(%.2f ms, %.0f TFLOP/s = %.2f of bf16 peak, ceiling %.2f ms); finite %s %s %s" % (
                      ftype, res["bs1_decode"]["tok_s"], res["bs1_decode"]["ms"], res["bs1_decode"]["ceiling_tok_s"], res["bs1_decode"]["hbm_frac"],
                      res["bs32_step"]["tok_s"], res["bs32_step"]["ms"], res["bs32_step"]["ceiling_tok_s"], res["pp512"]["tok_s"], res["pp512"]["ms"],
                      res["pp512"]["tflops"], res["pp512"]["bf16_frac"], res["pp512"]["ceiling_ms"], res["bs1_decode"]["finite"], res["bs32_step"]["finite"],
                      res["pp512"]["finite"]))
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
        rec = {"bench_py_no_cpu": cur["value"], "unit": cur.get("unit"), "recorded_r2": last["value"], "rel_change": d, "within_2pct": abs(d) <= 0.02}
        log.write(json.dumps(rec) + "\n")
        open(os.path.join(a.out, "bench_no_cpu.json"), "w").write(line[-1] + "\n")
        print("bench.py --no-cpu: %.1f %s vs recorded %.1f (profiles/r2_bench.json): %+.2f%%" % (cur["value"], cur.get("unit"), last["value"], 100 * d))
    log.close()


if __name__ == "__main__":
    main()
