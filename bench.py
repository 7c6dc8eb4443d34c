#!/usr/bin/env python
"""bench.py -- Llama-3-8B Q4_K_M batch-1 decode on B200 through the ggml-b200 C ABI (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one decoded token: one pass of the whole hot path (32 layers of rms_norm -> Q4_K/Q6_K GEMV x7 -> rope ->
KV store -> flash_attn_ext -> ..., then the 128256-row output GEMV) over a 512-token context.

  value     tok/s with every input resident in HBM (CUDA events on the library's stream, CUDA-graph replay)
  e2e       tok/s through the reference-facing call with HOST buffers: per step the pinned host->device copies of the
            token embedding, position and KQ mask, b200_graph_compute, and the device->host read of the logits
  e2e_llama (extra) the same workload through the UNMODIFIED llama.cpp runtime (llama_decode) with libggml-b200.so
            loaded as its backend plugin -- what cortex.llamacpp's LlamaServerContext calls
  roofline  the Q4_K decode GEMV (dominant kernel): algorithmic bytes / CUDA-event time over all Q4_K matmuls of a step
  cpu_baseline / --impl reference: the reference's own ggml CPU backend (oracle/_ref, built from /root/reference) on the
            same GGUF shapes, all host threads, bounded sample of decode steps.

N > 1 (torchrun): every rank runs an independent replica of the model on its own GPU (slot data parallelism,
SURVEY.md 8e: no collective on the data path); value = tokens of all ranks / max-over-ranks time.  scaling = weak.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
HARNESS = os.path.join(REF_DIR, "logits_dump")
BACKEND_SO = os.path.join(ROOT, "cortex.llamacpp_b200", "libggml-b200.so")
MODEL, FTYPE, KV, DEPTH = "llama3-8b", "q4_k_m", "f16", 512
METRIC = "Llama-3-8B Q4_K_M decode tok/s (bs1)"
WORKLOAD = "Llama-3-8B Q4_K_M (random-init GGUF blocks) bs1 decode, f16 KV, flash_attn, context depth %d" % DEPTH
# N > 1: the north-star split -- ONE Llama-3-70B stream, weights row-split over the N GPUs (strong scaling)
TP_METRIC = "Llama-3-70B Q4_K_M row-split tensor-parallel decode tok/s (bs1)"


def tp_workload(model, world):
    return "%s Q4_K_M (random-init GGUF blocks) bs1 decode, row-split over %d GPUs (all-reduce after wo and down), f16 KV, flash_attn, context depth %d" % (model, world, DEPTH)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """samples nvidia-smi clocks / throttle reasons during the timed region"""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        self.stop_flag = True
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].startswith("Active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def run_harness(ngl, n_prompt, n_gen, warm, threads, gguf, timeout=900):
    env = dict(os.environ)
    env["LD_LIBRARY_PATH"] = os.path.join(ROOT, "cortex.llamacpp_b200") + ":" + REF_DIR + ":" + env.get("LD_LIBRARY_PATH", "")
    env["LOGITS_DUMP_WARMUP"] = str(warm)
    if ngl > 0:
        env["GGML_BACKEND_PATH"] = BACKEND_SO
        env.setdefault("GGML_B200_GRAPHS", "1")
    else:
        env.pop("GGML_BACKEND_PATH", None)
    out = subprocess.run([HARNESS, gguf, "-", str(ngl), str(n_prompt), str(n_gen), KV, "1", str(threads)], env=env,
                         capture_output=True, text=True, timeout=timeout)
    for line in reversed(out.stdout.strip().splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError("harness failed (rc %d): %s" % (out.returncode, out.stderr[-800:]))


def ensure_gguf(model=MODEL, layers=0):
    path = "/tmp/b200_bench_%s_%s%s.gguf" % (model, FTYPE, "_l%d" % layers if layers else "")
    if not os.path.exists(path):
        cmd = [sys.executable, os.path.join(ROOT, "tools", "make_gguf.py"), "--model", model, "--ftype", FTYPE, "--out", path + ".tmp"]
        if layers:
            cmd += ["--layers", str(layers)]
        subprocess.check_call(cmd, stderr=subprocess.DEVNULL)
        os.replace(path + ".tmp", path)
    return path


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def reference_arm(a):
    """the reference's own CPU backend (unmodified llama.cpp sources compiled by oracle/Makefile) on the host cores"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    line = {"impl": "reference", "metric": METRIC, "unit": "tok/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8 x int4..6 block dots (q8_K/q8_0 activations), f32 accumulate",
            "data": "synthetic", "config": {"workload": WORKLOAD}}
    if not os.path.exists(HARNESS):
        line["unavailable"] = "oracle/_ref was not built (run __graft_entry__.build() where /root/reference exists)"
        print(json.dumps(line))
        return
    threads = host_threads()
    if a.gpus > 1 and a.tp_model:
        # the N-GPU arm measures ONE tensor-parallel stream of the 70B model: the CPU reference runs that model's decode step.  Bounded
        # sample: a decode step is linear in the layer count, so two 70B-shaped GGUFs with 4 and 8 of the 80 layers are timed and the
        # full model is  fixed + 80 x per_layer  (40 GB of weights per token would otherwise take minutes per step on the host cores)
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        from make_gguf import MODELS
        L_full = MODELS[a.tp_model][0]
        steps = max(2, min(a.steps, 8))
        t = {}
        for nl in (4, 8):
            r = run_harness(0, DEPTH, steps, 1, threads, ensure_gguf(a.tp_model, nl), timeout=1800)
            t[nl] = 1.0 / r["decode_tok_s"]
        per_layer = (t[8] - t[4]) / 4.0
        fixed = max(0.0, t[4] - 4.0 * per_layer)
        v = 1.0 / (fixed + L_full * per_layer)
        line.update({"metric": TP_METRIC, "scaling": "strong", "config": {"workload": tp_workload(a.tp_model, a.gpus)}})
        sample = "%d decode steps after a %d-token prompt on 4- and 8-layer %s-shaped GGUFs, extrapolated linearly to %d layers (%.1f ms per layer + %.1f ms fixed)" % (
            steps, DEPTH, a.tp_model, L_full, per_layer * 1e3, fixed * 1e3)
    else:
        gguf = ensure_gguf()
        steps = a.steps
        r = run_harness(0, DEPTH, steps, min(a.warmup, 2), threads, gguf)
        v = r["decode_tok_s"]
        sample = "%d decode steps after a %d-token prompt, llama_decode on the ggml CPU backend (AVX2 build)" % (steps, DEPTH)
    line.update({"value": v, "ms_per_step": 1000.0 / v, "steps": steps,
                 "cpu_baseline": {"value": v, "unit": "tok/s", "cores": threads, "kind": "reference", "sample": sample},
                 "e2e": {"value": v, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                 "gpu_launches": 0})
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layers", type=int, default=0, help="debug: fewer layers (the reported line is then INVALID for the metric)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / e2e_llama legs (profiling runs)")
    ap.add_argument("--graphs", type=int, default=1)
    ap.add_argument("--pdl", type=int, default=int(os.environ.get("GGML_B200_PDL", "1")))
    ap.add_argument("--fusion", type=int, default=2)
    ap.add_argument("--l2pf", type=int, default=0)
    ap.add_argument("--no-batch", action="store_true", help="skip the bs32-decode / prefill legs")
    ap.add_argument("--tp-model", default="llama3-70b", help="N>1: model of the extra row-split tensor-parallel leg ('' = skip)")
    ap.add_argument("--tp-layers", type=int, default=0, help="debug: fewer layers in the TP leg (reported as INVALID)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the logits of the last timed step (rank 0) to DIR/logits.npy, "
                    "float32 [1, n_vocab]; inputs and weights are seeded, so two builds can be compared output for output")
    a = ap.parse_args()
    if a.impl == "reference":
        return reference_arm(a)

    import torch
    import torch.distributed as dist
    from __graft_entry__ import load_llama_graph, load_package
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU: there is no CPU fallback"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    b200 = load_package()
    lg = load_llama_graph()
    L = b200.lib()
    ctx = b200.Context(local)
    W = max(a.warmup, 3)
    K = a.steps
    n_ctx = 1024
    g = lg.LlamaGraph(b200, model=MODEL, ftype=FTYPE, kv=KV, n_ctx=n_ctx, layers=a.layers, device=local, max_tokens=1)
    g.fill_cache(DEPTH)
    kv_head, n_kv = DEPTH, (DEPTH + 1 + 255) // 256 * 256
    rng = np.random.default_rng(rank)
    emb, pos, mask = g.set_inputs_host(1, kv_head, n_kv, rng)
    # pinned host staging (what the scheduler's host buffer type provides) + device inputs
    h_emb = torch.from_numpy(emb.reshape(-1)).pin_memory()
    h_pos = torch.from_numpy(pos).pin_memory()
    h_mask = torch.from_numpy(mask.reshape(-1)).pin_memory()
    h_logits = torch.empty(g.V, dtype=torch.float32).pin_memory()
    g.inp_embd[:g.E] = h_emb.cuda(local)
    g.pos[:1] = h_pos.cuda(local)
    g.mask_f32[:h_mask.numel()] = h_mask.cuda(local)
    torch.cuda.synchronize()
    ops = g.build(1, kv_head, n_kv)
    ops_arr = (b200.Op * len(ops))(*ops)
    ctx.set_option("cuda_graphs", a.graphs)
    ctx.set_option("pdl", a.pdl)
    ctx.set_option("fusion", a.fusion)
    ctx.set_option("l2_prefetch", a.l2pf)

    def step():
        b200.check(L.b200_graph_compute(ctx.h, ops_arr, len(ops)), "graph_compute")

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    e0, e1 = L.b200_event_create(local), L.b200_event_create(local)

    # ---------------------------------------------------------------- value: inputs resident in HBM
    n_before = ctx.launches()
    step(); ctx.sync()
    launches_eager = ctx.launches() - n_before              # kernels of one step (graph replay launches the same nodes)
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(W):
        step()
    barrier()
    L.b200_event_record(ctx.h, e0)
    for _ in range(K):
        step()
    L.b200_event_record(ctx.h, e1)
    L.b200_event_synchronize(e1)
    barrier()
    ms = L.b200_event_elapsed_ms(e0, e1)
    if a.dump_outputs and rank == 0:          # the later legs overwrite g.logits (the roofline leg skips attention)
        os.makedirs(a.dump_outputs, exist_ok=True)
        np.save(os.path.join(a.dump_outputs, "logits.npy"), g.logits[:g.V].reshape(1, g.V).cpu().numpy())
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * K / (ms / 1e3)

    # ---------------------------------------------------------------- e2e: host buffers, copies inside the timed region
    def e2e_step():
        b200.check(L.b200_memcpy_h2d_async(ctx.h, g.inp_embd.data_ptr(), h_emb.data_ptr(), g.E * 4), "h2d")
        b200.check(L.b200_memcpy_h2d_async(ctx.h, g.pos.data_ptr(), h_pos.data_ptr(), 4), "h2d")
        b200.check(L.b200_memcpy_h2d_async(ctx.h, g.mask_f32.data_ptr(), h_mask.data_ptr(), h_mask.numel() * 4), "h2d")
        step()
        b200.check(L.b200_memcpy_d2h_async(ctx.h, h_logits.data_ptr(), g.logits.data_ptr(), g.V * 4), "d2h")
        ctx.sync()                                           # the sampler reads the logits on the host every step
    for _ in range(W):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e = {"value": world * K / e2e_s, "unit": "tok/s", "h2d_bytes_per_step": g.E * 4 + 4 + h_mask.numel() * 4, "d2h_bytes_per_step": g.V * 4,
           "path": "b200_memcpy_h2d_async x3 -> b200_graph_compute -> b200_memcpy_d2h_async -> b200_synchronize (C ABI, pinned host buffers)"}
    assert np.isfinite(h_logits.numpy()).all(), "non-finite logits"

    # ---------------------------------------------------------------- roofline of the dominant kernel (batch-1 decode GEMV)
    # The SAME captured step with flash_attn and rope+store not launched (option debug_skip=3): what remains are the fused
    # GEMV launches of the step exactly as they run in the timed region (one per qkv / wo / gate|up / down / output matmul,
    # graph replay, PDL) plus one 3 us mask copy.  achieved = their algorithmic bytes / CUDA-event time.
    peak, peak_src = measured_peaks()
    n_gemv = 4 * g.L + 1
    sb = g.step_bytes(1, n_kv)
    alg = sb["weights"] + sb["act"]
    ctx.set_option("debug_skip", 3)
    for _ in range(W):
        step()
    ctx.sync()
    reps = max(8, K // 4)
    L.b200_event_record(ctx.h, e0)
    for _ in range(reps):
        step()
    L.b200_event_record(ctx.h, e1)
    L.b200_event_synchronize(e1)
    k_ms = L.b200_event_elapsed_ms(e0, e1) / reps
    ctx.set_option("debug_skip", 0)
    achieved = alg / (k_ms / 1e3) / 1e9
    traffic = None
    tp_file = os.path.join(ROOT, "profiles", "r2_ncu_bs1_traffic.json")      # dram bytes per launch, all 129 GEMV launches of a step (committed ncu capture: same population as algorithmic_bytes_per_launch_avg)
    if os.path.exists(tp_file):
        try:
            traffic = json.load(open(tp_file))["dram_bytes_per_launch_avg"]
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": "b200_gemv_bs1_kernel (batch-1 decode GEMV over Q4_K/Q6_K GGUF blocks; the %d fused launches of a step as they run in the timed region: graph replay, PDL)" % n_gemv,
                "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "algorithmic_bytes_per_launch_avg": alg / n_gemv, "avg_launch_us": 1e3 * k_ms / n_gemv,
                "whole_step": {"algorithmic_bytes": sb["total"], "achieved_gbs": sb["total"] * (K / (ms / 1e3)) / 1e9,
                               "frac": sb["total"] * (K / (ms / 1e3)) / 1e9 / peak, "breakdown": sb}}

    clocks = sampler.summary()               # sampled from the first warm-up step through the value, e2e and roofline legs: always under load
    line = {"metric": METRIC, "value": value, "unit": "tok/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int8 x int4..6 block dots (q8_K/q8_0 activations), f32 accumulate", "data": "synthetic",
            "config": {"workload": WORKLOAD, "l2": "inputs larger than L2: %.2f GB of weights streamed per step vs 126 MB L2" % (g.weight_bytes / 1e9),
                       "n_kv": n_kv, "cuda_graphs": a.graphs, "pdl": a.pdl, "fusion": a.fusion, "l2_prefetch": a.l2pf, "replicas": world,
                       "layers": g.L if a.layers else "all (%d)" % g.L},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches_eager) * K, "roofline": roofline}
    if a.layers:
        line["INVALID"] = "--layers override: not the named model"

    # ---------------------------------------------------------------- CPU baseline + llama.cpp-level e2e (rank 0, N=1)
    if rank == 0 and world == 1 and not a.no_cpu and not a.layers and os.path.exists(HARNESS):
        try:
            gguf = ensure_gguf()
            threads = host_threads()
            if os.path.exists(BACKEND_SO):
                r = run_harness(99, DEPTH, K, W, 4, gguf)
                line["e2e_llama"] = {"value": r["decode_tok_s"], "unit": "tok/s", "prefill_tok_s": r["prefill_tok_s"],
                                     "path": "llama_decode (unmodified llama.cpp runtime) -> ggml_backend_sched -> libggml-b200.so graph_compute; logits read on host every step"}
                # the drop-in path is the end-to-end number; the direct C-ABI loop stays beside it
                line["e2e_capi"] = line["e2e"]
                line["e2e"] = {"value": r["decode_tok_s"], "unit": "tok/s", "h2d_bytes_per_step": e2e["h2d_bytes_per_step"], "d2h_bytes_per_step": e2e["d2h_bytes_per_step"],
                               "path": "reference-facing plugin: llama_decode (unmodified llama.cpp runtime, host token + host logits every step) -> ggml_backend_sched -> libggml-b200.so -> C ABI"}
            r = run_harness(0, DEPTH, 8, 1, threads, gguf)
            line["cpu_baseline"] = {"value": r["decode_tok_s"], "unit": "tok/s", "cores": threads, "kind": "reference",
                                    "sample": "8 decode steps after a %d-token prompt, llama_decode on the reference ggml CPU backend" % DEPTH}
        except Exception as ex:           # the baseline is a report, never a reason to lose the GPU line
            line["cpu_baseline"] = {"value": None, "unit": "tok/s", "cores": host_threads(), "kind": "reference", "sample": "failed: %s" % str(ex)[:200]}
    # ---------------------------------------------------------------- N = 1: the other two numbers of the metric (bs32 decode, prefill)
    if world == 1 and not a.layers and not a.no_batch:
        try:
            g.keep.clear(); g.layers.clear()
            torch.cuda.empty_cache()
            line["batched"] = batch_legs(a, b200, lg, L, ctx, local, peak)
        except Exception as ex:
            line["batched"] = {"error": str(ex)[:300]}

    # ---------------------------------------------------------------- N > 1: row-split tensor-parallel leg (SURVEY.md 8e)
    if world > 1 and a.tp_model:
        try:
            del ops, ops_arr
            g.keep.clear(); g.layers.clear()
            del g
            torch.cuda.empty_cache()
            tp = tp_leg(a, b200, lg, L, ctx, rank, world, local, peak)
            line["tp"] = tp
            if "value" in tp and not a.tp_layers:
                # the driver-scored line at N > 1 is the north-star split (one 70B stream over N GPUs, strong scaling); the collective-free
                # replicas of the 8B model measured above stay as an extra key
                line["replicas"] = {"metric": METRIC, "value": line["value"], "unit": "tok/s", "scaling": "weak", "ms_per_step": line["ms_per_step"],
                                    "e2e": line["e2e"], "roofline": line["roofline"], "config": line["config"], "gpu_launches": line["gpu_launches"]}
                line.update({"metric": TP_METRIC, "value": tp["value"], "ms_per_step": tp["ms_per_step"], "scaling": "strong",
                             "config": {"workload": tp_workload(a.tp_model, world), "l2": "inputs larger than L2: %.2f GB of weight shards streamed per GPU per step" % (tp["per_gpu_bytes_per_step"] / 1e9),
                                        "cuda_graphs": a.graphs, "pdl": a.pdl, "fusion": a.fusion, "parallelism": "tp%d" % world},
                             "e2e": tp["e2e"], "clocks": tp["clocks"] if tp["clocks"].get("sm_mhz") else line["clocks"], "gpu_launches": tp["gpu_launches_per_step"] * K * world,
                             "roofline": {"bound": "hbm", "kernel": "b200_gemv_bs1_kernel over each GPU's weight shard (whole TP step incl. the %d all-reduces)" % tp["n_allreduce"],
                                          "achieved": tp["per_gpu_achieved_gbs"], "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": tp["per_gpu_hbm_frac"], "traffic": None}})
        except Exception as ex:
            line["tp"] = {"error": str(ex)[:300]}
    if rank == 0:
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def batch_legs(a, b200, lg, L, ctx, local, peak):
    """BASELINE.json config #3 shape: Llama-3-8B Q4_K_M, n_parallel = 32 slots, q8_0 KV cache.  Two ubatches through the same
    C ABI: (a) continuous-batching decode, 32 slots x 1 token at depth 512 per slot (weights read once per step: HBM roofline
    = weights + the slots' KV); (b) a 512-token prefill ubatch (tcgen05 int8 GEMM + tensor-core flash attention: tensor
    roofline, quoted against 2 x the measured bf16 peak because MEASURED_PEAKS.json holds no int8 number)."""
    import torch
    slots, depth, PP = 32, 512, 512
    n_ctx = ((slots * depth + slots + 255) // 256 + 1) * 256
    g = lg.LlamaGraph(b200, model=MODEL, ftype=FTYPE, kv="q8_0", n_ctx=n_ctx, device=local, max_tokens=PP)
    g.fill_cache(slots * depth)
    rng = np.random.default_rng(1)
    e0, e1 = L.b200_event_create(local), L.b200_event_create(local)
    out = {"kv": "q8_0", "slots": slots}

    def timed(ops, reps, warm):
        arr = (b200.Op * len(ops))(*ops)
        n0 = ctx.launches()
        b200.check(L.b200_graph_compute(ctx.h, arr, len(ops)), "batched step"); ctx.sync()
        launches = ctx.launches() - n0
        for _ in range(warm):
            b200.check(L.b200_graph_compute(ctx.h, arr, len(ops)), "batched step")
        ctx.sync()
        L.b200_event_record(ctx.h, e0)
        for _ in range(reps):
            b200.check(L.b200_graph_compute(ctx.h, arr, len(ops)), "batched step")
        L.b200_event_record(ctx.h, e1)
        L.b200_event_synchronize(e1)
        return L.b200_event_elapsed_ms(e0, e1) / reps, int(launches)

    def upload(emb, pos, mask, T):
        g.inp_embd[:T * g.E] = torch.from_numpy(emb.reshape(-1)).cuda(local)
        g.pos[:T] = torch.from_numpy(pos).cuda(local)
        g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).cuda(local)
        torch.cuda.synchronize()

    # (a) bs32 continuous-batching decode
    n_kv = (slots * depth + slots + 255) // 256 * 256
    emb, pos, mask, kv_head = g.set_inputs_slots_host(slots, depth, n_kv, rng)
    upload(emb, pos, mask, slots)
    ms, launches = timed(g.build(slots, kv_head, n_kv), max(8, a.steps // 4), 3)
    kv_row = lg.row_size(g.kv_type, g.Hkv * g.D)
    bytes_ = g.weight_bytes + 2 * g.L * slots * (depth + 1) * kv_row
    out["bs32_decode"] = {"value": slots / (ms / 1e3), "unit": "tok/s", "ms_per_step": ms, "depth_per_slot": depth, "gpu_launches_per_step": launches,
                          "hbm_bytes_per_step": bytes_, "achieved_gbs": bytes_ / (ms / 1e3) / 1e9, "hbm_frac": bytes_ / (ms / 1e3) / 1e9 / peak,
                          "assert_finite": bool(torch.isfinite(g.logits[:slots * g.V]).all().item())}
    # (b) prefill: one 512-token ubatch into an empty region of the cache
    emb, pos, mask = g.set_inputs_host(PP, 0, PP, rng)
    upload(emb, pos, mask, PP)
    ms, launches = timed(g.build(PP, 0, PP, n_outputs=1), max(4, a.steps // 8), 2)       # a prompt ubatch asks for the last token's logits only
    flops = 2.0 * (g.weight_bytes_by_type and sum(nb / (lg.BLOCK[t][1] / lg.BLOCK[t][0]) for t, nb in g.weight_bytes_by_type.items())) * PP
    flops -= 2.0 * g.V * g.E * (PP - 1)                        # logits for the last token only
    flops += 4.0 * g.L * g.H * g.D * PP * PP / 2
    bf16 = 1631.8
    try:
        bf16 = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
    except Exception:
        pass
    i8_peak, i8_note = 2 * bf16, "2 x measured bf16 burst (no int8 number in MEASURED_PEAKS.json)"
    try:                                     # measured on this pool's B200 with a bare tcgen05.mma kind::i8 loop (tools/micro/i8_peak.cu)
        i8_peak = float(json.load(open(os.path.join(ROOT, "profiles", "r2_i8_peak.json")))["int8_tops"])
        i8_note = "measured: bare tcgen05.mma kind::i8 loop, 148 CTAs (profiles/r2_i8_peak.txt)"
    except Exception:
        pass
    out["prefill_pp512"] = {"value": PP / (ms / 1e3), "unit": "tok/s", "ms_per_ubatch": ms, "gpu_launches_per_ubatch": launches, "flops_per_ubatch": flops,
                            "achieved_tops": flops / (ms / 1e3) / 1e12, "peak_tops": i8_peak, "peak_note": i8_note,
                            "tensor_frac": flops / (ms / 1e3) / 1e12 / i8_peak,
                            "assert_finite": bool(torch.isfinite(g.logits[:g.V]).all().item())}
    g.keep.clear(); g.layers.clear()
    torch.cuda.empty_cache()
    return out


def tp_leg(a, b200, lg, L, ctx, rank, world, local, peak):
    """Row-split tensor parallelism over all `world` GPUs: ONE model (default Llama-3-70B Q4_K_M, random-init shards drawn
    from a common seed), wq/wk/wv/gate/up split by rows, wo/down by K, B200_OP_ALLREDUCE (one-shot peer-memory kernel over
    NVLink) after wo and down.  scaling = strong: tok/s of the single bs1 stream; roofline = per-GPU shard bytes / step time."""
    import torch
    import torch.distributed as dist

    def exchange(blob):
        out = [None] * world
        dist.all_gather_object(out, blob)
        return out
    ctx.comm_init(rank, world, exchange)
    depth = DEPTH
    g = lg.LlamaGraph(b200, model=a.tp_model, ftype=FTYPE, kv=KV, n_ctx=1024, layers=a.tp_layers, device=local, max_tokens=1,
                      tp_rank=rank, tp_world=world)
    g.fill_cache(depth)
    kv_head, n_kv = depth, (depth + 1 + 255) // 256 * 256
    rng = np.random.default_rng(0)                               # same inputs on every rank
    emb, pos, mask = g.set_inputs_host(1, kv_head, n_kv, rng)
    g.inp_embd[:g.E] = torch.from_numpy(emb.reshape(-1)).cuda(local)
    g.pos[:1] = torch.from_numpy(pos).cuda(local)
    g.mask_f32[:mask.size] = torch.from_numpy(mask.reshape(-1)).cuda(local)
    torch.cuda.synchronize()
    ops = g.build(1, kv_head, n_kv)
    arr = (b200.Op * len(ops))(*ops)
    ctx.set_option("cuda_graphs", a.graphs); ctx.set_option("fusion", a.fusion)
    e0, e1 = L.b200_event_create(local), L.b200_event_create(local)
    W, K = max(a.warmup, 3), a.steps
    n0 = ctx.launches()
    tp_sampler = ClockSampler(local)
    tp_sampler.start()
    b200.check(L.b200_graph_compute(ctx.h, arr, len(ops)), "tp step"); ctx.sync()
    launches = ctx.launches() - n0
    for _ in range(W):
        b200.check(L.b200_graph_compute(ctx.h, arr, len(ops)), "tp step")
    ctx.sync(); dist.barrier(); torch.cuda.synchronize()
    L.b200_event_record(ctx.h, e0)
    for _ in range(K):
        b200.check(L.b200_graph_compute(ctx.h, arr, len(ops)), "tp step")
    L.b200_event_record(ctx.h, e1)
    L.b200_event_synchronize(e1)
    ctx.sync(); dist.barrier()
    ms = L.b200_event_elapsed_ms(e0, e1)
    t = torch.tensor([ms], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    # where the step goes (timing-only replays with kernel classes not launched; results of these replays are discarded)
    breakdown = {}
    for name, mask_ in (("no_allreduce", 8), ("no_attention", 3), ("no_gemv", 4)):
        ctx.set_option("debug_skip", mask_)
        for _ in range(3):
            b200.check(L.b200_graph_compute(ctx.h, arr, len(ops)), "tp step")
        ctx.sync(); dist.barrier(); torch.cuda.synchronize()
        L.b200_event_record(ctx.h, e0)
        for _ in range(8):
            b200.check(L.b200_graph_compute(ctx.h, arr, len(ops)), "tp step")
        L.b200_event_record(ctx.h, e1)
        L.b200_event_synchronize(e1)
        tt = torch.tensor([L.b200_event_elapsed_ms(e0, e1) / 8], device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        breakdown[name + "_ms"] = float(tt.item())
    ctx.set_option("debug_skip", 0)
    b200.check(L.b200_graph_compute(ctx.h, arr, len(ops)), "tp step"); ctx.sync(); dist.barrier()
    logits = g.logits[:g.V].clone()
    ref = logits.clone()
    dist.broadcast(ref, 0)
    same = bool(torch.equal(ref, logits))
    flag = torch.tensor([1 if same else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    # end to end through the C ABI: every rank uploads the step's inputs from pinned host memory, the step runs, the logits come back
    h_emb = torch.from_numpy(emb.reshape(-1)).pin_memory(); h_pos = torch.from_numpy(pos).pin_memory(); h_mask = torch.from_numpy(mask.reshape(-1)).pin_memory()
    h_logits = torch.empty(g.V, dtype=torch.float32).pin_memory()

    def e2e_step():
        b200.check(L.b200_memcpy_h2d_async(ctx.h, g.inp_embd.data_ptr(), h_emb.data_ptr(), g.E * 4), "h2d")
        b200.check(L.b200_memcpy_h2d_async(ctx.h, g.pos.data_ptr(), h_pos.data_ptr(), 4), "h2d")
        b200.check(L.b200_memcpy_h2d_async(ctx.h, g.mask_f32.data_ptr(), h_mask.data_ptr(), h_mask.numel() * 4), "h2d")
        b200.check(L.b200_graph_compute(ctx.h, arr, len(ops)), "tp step")
        b200.check(L.b200_memcpy_d2h_async(ctx.h, h_logits.data_ptr(), g.logits.data_ptr(), g.V * 4), "d2h")
        ctx.sync()
    for _ in range(3):
        e2e_step()
    dist.barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(K):
        e2e_step()
    dist.barrier()
    tt = torch.tensor([time.perf_counter() - t0], device="cuda")
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e = {"value": K / float(tt.item()), "unit": "tok/s", "h2d_bytes_per_step": g.E * 4 + 4 + h_mask.numel() * 4, "d2h_bytes_per_step": g.V * 4,
           "path": "per rank: b200_memcpy_h2d_async x3 -> b200_graph_compute (sharded step, B200_OP_ALLREDUCE over NVLink) -> b200_memcpy_d2h_async -> b200_synchronize"}
    sb = g.step_bytes(1, n_kv)
    tok_s = K / (ms / 1e3)
    out = {"clocks": tp_sampler.summary(), "e2e": e2e, "n_allreduce": 2 * g.L, "model": "%s %s row-split over %d GPUs (random-init shards of one common-seed model)" % (a.tp_model, FTYPE, world), "world": world,
           "value": tok_s, "unit": "tok/s", "scaling": "strong", "ms_per_step": ms / K, "steps": K, "warmup": W,
           "allreduce": "B200_OP_ALLREDUCE x%d per step: one-shot peer-memory kernel over NVLink (f32 [E] = %d bytes), residual add fused" % (2 * g.L, g.E * 4),
           "gpu_launches_per_step": int(launches), "logits_identical_on_all_ranks": bool(flag.item()),
           "per_gpu_bytes_per_step": sb["total"], "per_gpu_achieved_gbs": sb["total"] * tok_s / 1e9, "per_gpu_hbm_frac": sb["total"] * tok_s / 1e9 / peak,
           "hbm_roofline_tok_s": peak * 1e9 / sb["total"],
           "step_ms_with_kernel_classes_not_launched": breakdown}
    if a.tp_layers:
        out["INVALID"] = "--tp-layers override"
    return out


if __name__ == "__main__":
    main()
