"""Row-split F16 / BF16 weight matmuls (B200_TENSOR_FLAG_SPLIT, llama.cpp's --split-mode row) on the Llama-3-70B matrices.

    python tools/split_float_bench.py --out DIR [--shapes small]

For bf16 and f16, every matrix and M in {1, 32, 512} token columns: one MUL_MAT through b200_op_compute on device 0, timed with CUDA
events after warm-up, then the same matrix row-split into 2 shards on device 0 (the split path run back to back on one GPU, with each
half timed alone: the compute each GPU of a 2-GPU split does), over 2 GPUs and over all visible GPUs (shard boundaries on multiples
of 128 rows at equal fractions, as the plugin's split_rows).  x and dst live on device 0, as llama.cpp keeps them.  Weight buffers
are rotated so that every timed launch reads its weights from HBM, not from the 126 MB L2: the unsplit working set is at least 4 x
the L2, so a half-height shard's is at least 2 x; on more GPUs a shard's share can fall below that (the JSONL records each
configuration's per-GPU working set).  Reported per configuration:
  us, per-GPU GB/s (algorithmic bytes of the busiest shard: its weight rows, x once, its dst rows) and its fraction of the copy
  peak measured in the same run, speedup over one GPU, and the fork/join overhead: split time minus the slowest shard timed alone
  on its own device (reading x from and writing dst to device 0, as inside the split).
Split outputs are compared with the unsplit output (max |diff| over max |unsplit|): equal up to f32 summation order.
Writes DIR/split_float_weights.jsonl and DIR/split_float_weights.md; the card names and power limits come first.  Configurations the
machine cannot run (fewer GPUs) are written as "not measured"."""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SHAPES = [("wq", 8192, 8192), ("wk|wv", 1024, 8192), ("gate/up", 28672, 8192), ("down", 8192, 28672), ("output", 128256, 8192)]   # (N rows, K)
MS = [1, 32, 512]
L2_BYTES = 126 << 20
SPLIT = 2                       # B200_TENSOR_FLAG_SPLIT
ROUNDING = 128                  # the plugin's SPLIT_ROUNDING


class Split(C.Structure):
    """b200_split of include/ggml_b200.h"""
    _fields_ = [("n_dev", C.c_int32), ("device", C.c_int32 * 16), ("shard", C.c_void_p * 16), ("row_low", C.c_int64 * 17)]


def cards():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return [ln.strip() for ln in q.stdout.strip().splitlines()]


def row_low(N, n):
    return [0] + [N * d // n // ROUNDING * ROUNDING for d in range(1, n)] + [N]


def copy_peak_gbs(torch):
    """device-to-device copy of 4 GiB on device 0: read + write bytes over the best of 5 event-timed copies"""
    a = torch.empty(1 << 30, dtype=torch.float32, device="cuda:0")
    b = torch.empty_like(a)
    b.copy_(a)
    best = float("inf")
    for _ in range(5):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        b.copy_(a)
        e.record()
        torch.cuda.synchronize()
        best = min(best, s.elapsed_time(e) / 1e3)
    return 2 * a.numel() * 4 / best / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default="all", help="'small': wq and wk|wv only (rehearsal)")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    import torch
    from __graft_entry__ import load_package
    b200 = load_package()
    L = b200.lib()
    assert torch.cuda.is_available(), "needs the GPU"
    ngpu = torch.cuda.device_count()
    # split configurations: label -> device of every shard.  "2 shards, 1 GPU" runs both shards on device 0, one after the other: it
    # times each half-height shard alone as the planner schedules it, which is the compute a 2-GPU split gives each GPU
    splits = {"2 shards, 1 GPU": [0, 0]}
    for n in sorted({2, ngpu}):
        if 1 < n <= ngpu:
            splits["%d GPUs" % n] = list(range(n))
    info = {"cards": cards(), "gpus": ngpu, "copy_peak_gbs": copy_peak_gbs(torch), "splits": splits,
            "not_measured": [] if ngpu >= 2 else ["row-split over 2 GPUs and over all visible GPUs: 1 GPU visible"]}
    print("cards (index, name, power limit, max SM clock): %s" % "; ".join(info["cards"]))
    print("copy peak (device 0, D2D copy, read + write): %.0f GB/s" % info["copy_peak_gbs"])
    log = open(os.path.join(a.out, "split_float_weights.jsonl"), "w")
    log.write(json.dumps(info) + "\n")
    ctxs = [b200.Context(d) for d in range(ngpu)]
    evs = [(L.b200_event_create(d), L.b200_event_create(d)) for d in range(ngpu)]

    def time_ops(dev, ops, reps, warm):
        ctx, (e0, e1) = ctxs[dev], evs[dev]
        for i in range(warm):
            ctx.compute_op(ops[i % len(ops)])
        ctx.sync()
        L.b200_event_record(ctx.h, e0)
        for i in range(reps):
            ctx.compute_op(ops[i % len(ops)])
        L.b200_event_record(ctx.h, e1)
        L.b200_event_synchronize(e1)
        return L.b200_event_elapsed_ms(e0, e1) * 1e3 / reps

    def mm(t, w_ptr, K, N, x, dst, flags=0):
        M = x.shape[0]
        wt = b200.tensor(w_ptr, t, [K, N], flags=b200.TENSOR_FLAG_WEIGHT | flags)
        dt = b200.tensor(dst.data_ptr(), b200.F32, [N, M], nb=[4, dst.shape[1] * 4, dst.shape[1] * 4 * M, dst.shape[1] * 4 * M])
        return b200.make_op(b200.OP_MUL_MAT, dt, [wt, b200.tensor(x.data_ptr(), b200.F32, [K, M])])

    rows = []
    shapes = SHAPES if a.shapes == "all" else SHAPES[:2]
    for ftype, t, dt in (("bf16", b200.BF16, torch.bfloat16), ("f16", b200.F16, torch.float16)):
        for name, N, K in shapes:
            wbytes = 2 * N * K
            nbuf = max(2, math.ceil(4 * L2_BYTES / wbytes))        # a half-height shard's set: >= 2 x L2
            ws = [((torch.rand(N, K, device="cuda:0") * 2 - 1) * 0.02).to(dt) for _ in range(nbuf)]
            # shards of every buffer for every split: tables[label][buffer], shard d on devs[d] (+ 512 bytes of slack)
            tables, keep = {}, []
            for label, devs in splits.items():
                n = len(devs)
                rl = row_low(N, n)
                tables[label] = []
                for w in ws:
                    sp = Split()
                    sp.n_dev = n
                    for d in range(n):
                        sp.device[d], sp.row_low[d] = devs[d], rl[d]
                        s = torch.zeros((rl[d + 1] - rl[d]) * K + 256, dtype=dt, device="cuda:%d" % devs[d])
                        s[:(rl[d + 1] - rl[d]) * K] = w[rl[d]:rl[d + 1]].reshape(-1).to(s.device)
                        keep.append(s)
                        sp.shard[d] = s.data_ptr()
                    sp.row_low[n] = N
                    tables[label].append(sp)
            for M in MS:
                x = torch.randn(M, K, device="cuda:0")
                out1 = torch.empty(M, N, device="cuda:0")
                reps = max(20, 2 * nbuf)
                torch.cuda.synchronize()
                us1 = time_ops(0, [mm(t, w.data_ptr(), K, N, x, out1) for w in ws], reps, nbuf)
                ref = out1.clone()                 # the last timed launch used ws[(reps - 1) % nbuf]
                last = (reps - 1) % nbuf
                byts1 = wbytes + 4 * M * K + 4 * M * N
                rec = {"ftype": ftype, "matrix": name, "N": N, "K": K, "M": M, "split": "1 GPU", "gpus": 1, "us": us1, "gbs_per_gpu": byts1 / us1 / 1e3,
                       "copy_peak_frac": byts1 / us1 / 1e3 / info["copy_peak_gbs"], "tflops": 2.0 * N * K * M / us1 / 1e6,
                       "weight_buffers": nbuf, "working_set_per_gpu_mb": nbuf * wbytes / 2**20}
                rows.append(rec)
                log.write(json.dumps(rec) + "\n"); log.flush()
                print("%-4s %-7s %6d x %5d M=%3d 1 GPU   %9.1f us %7.0f GB/s (%.2f of copy peak) %6.1f TFLOP/s" % (
                    ftype, name, N, K, M, us1, rec["gbs_per_gpu"], rec["copy_peak_frac"], rec["tflops"]))
                for label, devs in splits.items():
                    n = len(devs)
                    rl = row_low(N, n)
                    outs = torch.empty(M, N, device="cuda:0")
                    ops = [mm(t, C.addressof(sp), K, N, x, outs, SPLIT) for sp in tables[label]]
                    us = time_ops(0, ops, reps, nbuf)
                    ctxs[0].compute_op(ops[last]); ctxs[0].sync()
                    diff = float((outs - ref).abs().max() / ref.abs().max())
                    # every shard alone on its own device, x and dst in device 0 memory (peer access is on after the split ran)
                    shard_us = []
                    for d in range(n):
                        nr = rl[d + 1] - rl[d]
                        dst_d = outs[:, rl[d]:]          # dst rows of the shard: same column stride as inside the split
                        sops = [b200.make_op(b200.OP_MUL_MAT, b200.tensor(dst_d.data_ptr(), b200.F32, [nr, M], nb=[4, N * 4, N * 4 * M, N * 4 * M]),
                                             [b200.tensor(sp.shard[d], t, [K, nr], flags=b200.TENSOR_FLAG_WEIGHT), b200.tensor(x.data_ptr(), b200.F32, [K, M])])
                                for sp in tables[label]]
                        shard_us.append(time_ops(devs[d], sops, reps, nbuf))
                    busiest = max(rl[d + 1] - rl[d] for d in range(n))
                    one_dev = len(set(devs)) == 1
                    # GB/s per GPU: the busiest shard's bytes over the split's time; on one device the shards run back to back, all bytes
                    byts = byts1 if one_dev else 2 * busiest * K + 4 * M * K + 4 * M * busiest
                    rec = {"ftype": ftype, "matrix": name, "N": N, "K": K, "M": M, "split": label, "gpus": len(set(devs)), "row_low": rl, "us": us,
                           "gbs_per_gpu": byts / us / 1e3, "copy_peak_frac": byts / us / 1e3 / info["copy_peak_gbs"], "speedup": us1 / us,
                           "shard_alone_us": shard_us, "max_rel_diff_vs_1gpu": diff, "weight_buffers": nbuf,
                           "working_set_per_gpu_mb": nbuf * (wbytes if one_dev else 2 * busiest * K) / 2**20}
                    if one_dev:      # shards in sequence: the split's own cost over the shards' sum, and the best case of one shard per GPU
                        rec["overhead_us"] = us - sum(shard_us)
                        rec["speedup_bound_one_shard_per_gpu"] = us1 / max(shard_us)
                    else:
                        rec["fork_join_us"] = us - max(shard_us)
                    rows.append(rec)
                    log.write(json.dumps(rec) + "\n"); log.flush()
                    print("%-4s %-7s %6d x %5d M=%3d %-15s %9.1f us %7.0f GB/s/GPU (%.2f) x%.2f  shards alone %s us  %s  diff %.1e" % (
                        ftype, name, N, K, M, label, us, rec["gbs_per_gpu"], rec["copy_peak_frac"], rec["speedup"], "/".join("%.1f" % s for s in shard_us),
                        ("overhead %+.1f us, bound x%.2f" % (rec["overhead_us"], rec["speedup_bound_one_shard_per_gpu"])) if one_dev else
                        "fork/join %+.1f us" % rec["fork_join_us"], diff))
            del ws, tables, keep
            torch.cuda.empty_cache()
    log.close()
    for c in ctxs:
        c.close()
    write_md(os.path.join(a.out, "split_float_weights.md"), info, rows, splits)


def write_md(path, info, rows, splits):
    multi = [lb for lb in splits if lb != "2 shards, 1 GPU"] or ["2 GPUs"]      # the multi-GPU columns, "not measured" when absent
    cols = ["1 GPU", "2 shards, 1 GPU"] + multi
    heads = {"1 GPU": "1 GPU: us, GB/s (frac of copy peak)",
             "2 shards, 1 GPU": "2 shards on 1 GPU: us, shards alone us, overhead us, speedup bound, rel diff"}
    with open(path, "w") as f:
        f.write("# Row-split F16 / BF16 weight matmuls (`tools/split_float_bench.py`)\n\n")
        f.write("Machine: %d visible GPU(s): %s (index, name, power limit, max SM clock).  Copy peak measured in the same run (device 0, "
                "device-to-device copy, read + write bytes): %.0f GB/s.\n\n" % (info["gpus"], "; ".join(info["cards"]), info["copy_peak_gbs"]))
        f.write("One `MUL_MAT` per matrix (Llama-3-70B shapes), CUDA-event time per launch after warm-up, weight buffers rotated (unsplit "
                "working set >= 4 x the 126 MB L2, a half-height shard's >= 2 x; `weight_buffers` in the JSONL).  GB/s per GPU: algorithmic bytes of the busiest GPU's shard "
                "(its weight rows, x, its dst rows) over the split's time.  \"2 shards on 1 GPU\": both halves on device 0, run one after the "
                "other by the split path; \"shards alone\" times each half alone, which is the compute each GPU of a 2-GPU split does; "
                "overhead = split time - sum of the shards alone; speedup bound = 1-GPU time / slowest shard alone, a 2-GPU split without "
                "fork/join or NVLink cost.  Multi-GPU columns: speedup over 1 GPU, fork/join = split time - slowest shard alone on its GPU, "
                "rel diff (every split) = max |split - unsplit| / max |unsplit|.\n\n")
        if info["gpus"] < 2:
            f.write("Row-split over 2 GPUs and over all visible GPUs: not measured (%d GPU visible).\n\n" % info["gpus"])
        f.write("| type | matrix | N x K | M | " + " | ".join(heads.get(c, c + ": us, GB/s/GPU (frac), speedup, fork/join us, rel diff") for c in cols) + " |\n")
        f.write("|---|---|---|---|" + "---|" * len(cols) + "\n")
        keyed = {(r["ftype"], r["matrix"], r["M"], r["split"]): r for r in rows}
        for (ft, name, M, lb), r in keyed.items():
            if lb != "1 GPU":
                continue
            cells = []
            for c in cols:
                s = keyed.get((ft, name, M, c))
                if s is None:
                    cells.append("not measured")
                elif c == "1 GPU":
                    cells.append("%.1f, %.0f (%.2f)" % (s["us"], s["gbs_per_gpu"], s["copy_peak_frac"]))
                elif "overhead_us" in s:
                    cells.append("%.1f, %s, %+.1f, x%.2f, %.1e" % (s["us"], " / ".join("%.1f" % v for v in s["shard_alone_us"]), s["overhead_us"],
                                                                  s["speedup_bound_one_shard_per_gpu"], s["max_rel_diff_vs_1gpu"]))
                else:
                    cells.append("%.1f, %.0f (%.2f), x%.2f, %+.1f, %.1e" % (s["us"], s["gbs_per_gpu"], s["copy_peak_frac"], s["speedup"], s["fork_join_us"],
                                                                         s["max_rel_diff_vs_1gpu"]))
            f.write("| %s | %s | %d x %d | %d | %s |\n" % (ft, name, r["N"], r["K"], M, " | ".join(cells)))


if __name__ == "__main__":
    main()
