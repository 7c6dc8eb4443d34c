"""Host-side mirror of the compute graph llama.cpp hands to a backend for the `llama` architecture.

This restates, node for node, what ``llm_build_llama`` (llama.cpp/src/llama-model.cpp:4093-4230) together with
``build_norm`` / ``build_ffn`` / ``build_attn`` (llama.cpp/src/llama-graph.cpp:675-832, 1187-1199, 1375-1439) emit per
ubatch with flash attention on, as a flat ``b200_op`` list over tensors resident in HBM.  It exists so that ``bench.py``,
``__graft_entry__.smoke()`` and the parity tests can drive exactly the op sequence the ggml backend
(``backend/ggml-b200.cpp``) forwards from ``graph_compute`` -- through the same C ABI, with no llama.cpp in the loop.

Weights are synthetic: random GGUF blocks of the K_M mixture ``llama-quant.cpp`` would choose (see
``tools/make_gguf.py``), generated directly in HBM.  torch is used only for device memory.
"""
import math
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tools"))
from make_gguf import MODELS, tensor_type  # noqa: E402

F32, F16, Q4_0, Q8_0, Q4_K, Q5_K, Q6_K, I32, BF16 = 0, 1, 2, 8, 12, 13, 14, 26, 30
BLOCK = {F32: (1, 4), F16: (1, 2), BF16: (1, 2), I32: (1, 4), Q4_0: (32, 18), Q8_0: (32, 34), Q4_K: (256, 144), Q5_K: (256, 176), Q6_K: (256, 210)}
KV_TYPES = {"f16": F16, "q8_0": Q8_0, "q4_0": Q4_0}


def row_size(t, k):
    be, bb = BLOCK[t]
    assert k % be == 0, (t, k)
    return k // be * bb


def device_rand_16bit(torch, t, nrows, K, amp, gen, device):
    """uniform(-amp, amp) weights of F16 / BF16 type ``t`` created in HBM, as raw bytes"""
    dt = torch.float16 if t == F16 else torch.bfloat16
    out = torch.empty(nrows * K, dtype=dt, device=device)
    step = 1 << 26
    for i0 in range(0, nrows * K, step):
        n = min(step, nrows * K - i0)
        out[i0:i0 + n] = ((torch.rand(n, device=device, generator=gen) * 2 - 1) * amp).to(dt)
    return out.view(torch.uint8)


def device_rand_blocks(torch, t, nrows, K, amp, gen, device):
    """random valid rows of quantised type ``t`` in GGUF block layout, created in HBM (same recipe as tools/make_gguf.py)"""
    be, bb = BLOCK[t]
    nb = nrows * (K // be)
    out = torch.empty(nb * bb + 256, dtype=torch.uint8, device=device)          # +256: tail padding as b200_alloc_size
    out[nb * bb:].zero_()
    step = 1 << 22
    for b0 in range(0, nb, step):
        n = min(step, nb - b0)
        blk = torch.randint(0, 256, (n, bb), dtype=torch.uint8, device=device, generator=gen)
        u = torch.rand(n, device=device, generator=gen) + 0.5
        sign = (torch.randint(0, 2, (n,), device=device, generator=gen) * 2 - 1).to(torch.float32)

        def f16(v):
            return v.to(torch.float16).view(torch.uint8).reshape(n, 2)
        if t == Q4_0:
            blk[:, 0:2] = f16(u * amp / 8 * sign)
        elif t == Q8_0:
            blk[:, 0:2] = f16(u * amp / 127 * sign)
        elif t in (Q4_K, Q5_K):
            qmax = 15 if t == Q4_K else 31
            d = u * amp / (31.5 * qmax)
            blk[:, 0:2] = f16(d)
            blk[:, 2:4] = f16(d * qmax / 2)
        elif t == Q6_K:
            blk[:, 208:210] = f16(u * amp / (64 * 32) * sign)
        out[b0 * bb:(b0 + n) * bb] = blk.reshape(-1)
    return out


def tp_plan(model_dims, world):
    """Megatron split of a llama layer over `world` ranks (SURVEY.md 8e): heads / KV heads / FFN columns per rank.
    wq|wk|wv and gate|up are split by OUTPUT ROWS (whole heads, whole FF rows), wo and down by K; K-quant shards must
    start on 256-element super-block boundaries.  Raises if the model does not divide."""
    H, Hkv, D, FF = model_dims
    if H % world or Hkv % world or FF % world:
        raise ValueError("tensor parallel %d does not divide H=%d Hkv=%d FF=%d" % (world, H, Hkv, FF))
    Hl, Hkvl, FFl = H // world, Hkv // world, FF // world
    if (Hl * D) % 256 or FFl % 256:
        raise ValueError("K-split shards must be multiples of 256 elements: H/N*D=%d FF/N=%d" % (Hl * D, FFl))
    return Hl, Hkvl, FFl


def shard_rows(buf, t, K, N, rank, world):
    """column-parallel shard: rows [rank*N/world, (rank+1)*N/world) of a [K, N] GGUF tensor are one contiguous byte range"""
    rb = row_size(t, K)
    n = N // world
    return buf[rank * n * rb:(rank + 1) * n * rb]


def shard_k(buf, t, K, N, rank, world):
    """row-parallel shard: columns [rank*K/world, (rank+1)*K/world) of every row = whole blocks; returns a contiguous copy
    (what a split buffer type's set_tensor would store on this rank).  Works on torch (device) and numpy (host) uint8."""
    be, bb = BLOCK[t]
    nbk = K // be
    assert nbk % world == 0, (K, be, world)
    per = nbk // world
    v = buf[:N * nbk * bb].reshape(N, nbk, bb)[:, rank * per:(rank + 1) * per, :]
    return v.reshape(-1).clone() if hasattr(v, "clone") else v.reshape(-1).copy()


class LlamaGraph:
    """Synthetic llama-architecture model in HBM + builders for the per-ubatch op list.

    n_ctx cells of KV cache per layer (one unified cache as llama_kv_cache_unified, llama-kv-cache.cpp:76-113).
    """

    def __init__(self, b200, model="llama3-8b", ftype="q4_k_m", kv="f16", n_ctx=4096, layers=0, seed=1234, device=0, max_tokens=1,
                 tp_rank=0, tp_world=1):
        """tp_world > 1: this process holds rank tp_rank's shard of a row-split tensor-parallel model.  Every rank draws the
        SAME full tensors from the same seed and keeps only its shard, so TP=N computes the same model as TP=1."""
        import torch
        self.torch, self.b200 = torch, b200
        self.dev = torch.device("cuda", device)
        L, E, H, Hkv, D, FF, V, rope_base, n_expert, n_used = MODELS[model]
        if layers:
            L = layers
        self.n_expert, self.n_used = n_expert, n_used
        if n_expert and tp_world > 1:
            raise NotImplementedError("tensor-parallel MoE")
        self.model, self.ftype = model, ftype
        self.tp_rank, self.tp_world = tp_rank, tp_world
        self.H_full, self.Hkv_full, self.FF_full = H, Hkv, FF
        Hf, Hkvf, FFf = H, Hkv, FF
        if tp_world > 1:
            H, Hkv, FF = tp_plan((H, Hkv, D, FF), tp_world)
        self.L, self.E, self.H, self.Hkv, self.D, self.FF, self.V, self.rope_base = L, E, H, Hkv, D, FF, V, rope_base
        self.kv_type = KV_TYPES[kv]
        self.n_ctx = n_ctx
        self.max_tokens = max_tokens
        gen = torch.Generator(device=self.dev)
        gen.manual_seed(seed)
        self.keep = []
        self.weight_bytes = 0
        self.weight_bytes_by_type = {}

        def weight(name, K, N, il, gain=1.0, split=None):
            """K, N are the FULL dimensions; split = None (replicated) | "rows" (column parallel) | "k" (row parallel)"""
            t = tensor_type(name, ftype, il, L, n_expert, Hf // Hkvf)
            amp = gain * math.sqrt(3.0 / K)
            if t == F32:
                buf = ((torch.rand(N * K, device=self.dev, generator=gen) * 2 - 1) * amp).view(torch.uint8)
            elif t in (F16, BF16):
                buf = device_rand_16bit(torch, t, N, K, amp, gen, self.dev)
            else:
                buf = device_rand_blocks(torch, t, N, K, amp, gen, self.dev)
            if tp_world > 1 and split == "rows":
                buf = torch.cat([shard_rows(buf, t, K, N, tp_rank, tp_world), torch.zeros(256, dtype=torch.uint8, device=self.dev)])
                N = N // tp_world
            elif tp_world > 1 and split == "k":
                buf = torch.cat([shard_k(buf, t, K, N, tp_rank, tp_world), torch.zeros(256, dtype=torch.uint8, device=self.dev)])
                K = K // tp_world
            self.keep.append(buf)
            nbytes = N * row_size(t, K)
            self.weight_bytes += nbytes
            self.weight_bytes_by_type[t] = self.weight_bytes_by_type.get(t, 0) + nbytes
            return b200.tensor(buf.data_ptr(), t, [K, N], flags=b200.TENSOR_FLAG_WEIGHT)

        def experts(name, K, N, il):
            """n_expert matrices [K, N] back to back (ggml layout [K, N, n_expert], llama-model.cpp ffn_*_exps)"""
            t = tensor_type(name, ftype, il, L, n_expert, Hf // Hkvf)
            if t in (F16, BF16):
                buf = device_rand_16bit(torch, t, N * n_expert, K, math.sqrt(3.0 / K), gen, self.dev)
            else:
                buf = device_rand_blocks(torch, t, N * n_expert, K, math.sqrt(3.0 / K), gen, self.dev)
            self.keep.append(buf)
            nbytes = n_expert * N * row_size(t, K)
            self.weight_bytes += nbytes
            self.weight_bytes_by_type[t] = self.weight_bytes_by_type.get(t, 0) + nbytes
            self.expert_bytes = getattr(self, "expert_bytes", 0) + nbytes
            rs = row_size(t, K)
            return b200.tensor(buf.data_ptr(), t, [K, N, n_expert], nb=[BLOCK[t][1], rs, rs * N, rs * N * n_expert], flags=b200.TENSOR_FLAG_WEIGHT)

        def norm():
            buf = (1.0 + 0.02 * torch.randn(E, device=self.dev, generator=gen)).to(torch.float32)
            self.keep.append(buf)
            return b200.tensor(buf.data_ptr(), F32, [E], flags=b200.TENSOR_FLAG_WEIGHT)

        self.layers = []
        for il in range(L):
            p = "blk.%d." % il
            lw = dict(
                attn_norm=norm(),
                wq=weight(p + "attn_q.weight", E, Hf * D, il, split="rows"), wk=weight(p + "attn_k.weight", E, Hkvf * D, il, split="rows"),
                wv=weight(p + "attn_v.weight", E, Hkvf * D, il, split="rows"), wo=weight(p + "attn_output.weight", Hf * D, E, il, split="k"),
                ffn_norm=norm())
            if n_expert:
                lw.update(gate_inp=weight(p + "ffn_gate_inp.weight", E, n_expert, il, gain=1.0),
                          gate_exps=experts(p + "ffn_gate_exps.weight", E, FFf, il), down_exps=experts(p + "ffn_down_exps.weight", FFf, E, il),
                          up_exps=experts(p + "ffn_up_exps.weight", E, FFf, il))
            else:
                lw.update(gate=weight(p + "ffn_gate.weight", E, FFf, il, split="rows"), down=weight(p + "ffn_down.weight", FFf, E, il, split="k"),
                          up=weight(p + "ffn_up.weight", E, FFf, il, split="rows"))
            rs = row_size(self.kv_type, Hkv * D)
            kc = torch.zeros(rs * n_ctx, dtype=torch.uint8, device=self.dev)
            vc = torch.zeros(rs * n_ctx, dtype=torch.uint8, device=self.dev)
            self.keep += [kc, vc]
            lw["k_cache"], lw["v_cache"] = kc, vc
            self.layers.append(lw)
        self.output_norm = norm()
        self.output = weight("output.weight", E, V, 0, gain=4.0)
        # ---- compute buffers (what ggml-alloc would hand out); sized for max_tokens per ubatch ----
        T = max_tokens

        def f32buf(n):
            b = torch.zeros(n, dtype=torch.float32, device=self.dev)
            self.keep.append(b)
            return b
        self.inp_embd = f32buf(E * T)
        self.pos = torch.zeros(T, dtype=torch.int32, device=self.dev)
        self.mask_f32 = f32buf(n_ctx * ((T + 63) // 64 * 64))
        self.mask_f16 = torch.zeros(n_ctx * ((T + 63) // 64 * 64), dtype=torch.float16, device=self.dev)
        self.cur = f32buf(E * T); self.cur2 = f32buf(E * T); self.resid = f32buf(E * T); self.resid2 = f32buf(E * T)
        self.q = f32buf(H * D * T); self.k = f32buf(Hkv * D * T); self.v = f32buf(Hkv * D * T)
        self.qr = f32buf(H * D * T); self.kr = f32buf(Hkv * D * T)
        self.att = f32buf(H * D * T)
        nu = max(1, n_used)
        self.g = f32buf(FF * T * nu); self.u = f32buf(FF * T * nu); self.gu = f32buf(FF * T * nu); self.tmpE = f32buf(E * T * nu)
        if n_expert:
            self.r_logits = f32buf(n_expert * T); self.r_probs = f32buf(n_expert * T); self.r_w = f32buf(n_used * T); self.r_wn = f32buf(n_used * T)
            self.r_sum = f32buf(T); self.moe_out = f32buf(E * T)
            self.r_sel = torch.zeros(n_expert * T, dtype=torch.int32, device=self.dev)
        self.logits = f32buf(V * T)
        torch.cuda.synchronize(self.dev)

    # ------------------------------------------------------------------------------------------------------------
    def fill_cache(self, n_cells, seed=7):
        """put plausible K/V rows into the first n_cells cells of every layer (synthetic context)"""
        torch = self.torch
        gen = torch.Generator(device=self.dev)
        gen.manual_seed(seed)
        HD = self.Hkv * self.D
        for lw in self.layers:
            for c in (lw["k_cache"], lw["v_cache"]):
                if self.kv_type == F16:
                    x = torch.randn(n_cells * HD, device=self.dev, generator=gen).to(torch.float16)
                    c[:n_cells * HD * 2] = x.view(torch.uint8)
                else:
                    blk = device_rand_blocks(torch, self.kv_type, n_cells, HD, 2.0, gen, self.dev)
                    c[:n_cells * row_size(self.kv_type, HD)] = blk[:n_cells * row_size(self.kv_type, HD)]
        torch.cuda.synchronize(self.dev)

    def build(self, n_tok, kv_head, n_kv, n_outputs=None):
        """op list of ONE ubatch: n_tok tokens written at cell kv_head, attending over cells [0, n_kv).  n_outputs: logits
        are computed for the LAST n_outputs tokens only (llama.cpp's inp_out_ids: a prompt ubatch asks for one row,
        llama-model.cpp:4196-4201; we apply the selection before the final norm); default all tokens -> self.logits[:n_out*V]"""
        b, T = self.b200, n_tok
        assert T <= self.max_tokens and n_kv <= self.n_ctx and kv_head + T <= self.n_ctx
        E, H, Hkv, D, FF, V = self.E, self.H, self.Hkv, self.D, self.FF, self.V
        t = b.tensor
        p = lambda x: x.data_ptr()                                         # noqa: E731
        ops = []
        Tp = (T + 63) // 64 * 64
        # mask f32 -> f16 once per graph (llama-graph.cpp:1325)
        ops.append(b.make_op(b.OP_CPY, t(p(self.mask_f16), F16, [n_kv, Tp]), [t(p(self.mask_f32), F32, [n_kv, Tp])]))
        rope_params = [0, D, 0, 0, 8192, float(self.rope_base), 1.0, 0.0, 1.0, 32.0, 1.0]
        kvt = self.kv_type
        rs_row = row_size(kvt, Hkv * D)
        rs_head = row_size(kvt, D)
        inp, other = self.inp_embd, self.resid
        for il, lw in enumerate(self.layers):
            xin = t(p(inp), F32, [E, T])
            # attention norm
            ops.append(b.make_op(b.OP_RMS_NORM, t(p(self.cur), F32, [E, T]), [xin], [1e-5]))
            ops.append(b.make_op(b.OP_MUL, t(p(self.cur2), F32, [E, T]), [t(p(self.cur), F32, [E, T]), lw["attn_norm"]]))
            xn = t(p(self.cur2), F32, [E, T])
            ops.append(b.make_op(b.OP_MUL_MAT, t(p(self.q), F32, [H * D, T]), [lw["wq"], xn]))
            ops.append(b.make_op(b.OP_MUL_MAT, t(p(self.k), F32, [Hkv * D, T]), [lw["wk"], xn]))
            ops.append(b.make_op(b.OP_MUL_MAT, t(p(self.v), F32, [Hkv * D, T]), [lw["wv"], xn]))
            post = t(p(self.pos), I32, [T])
            ops.append(b.make_op(b.OP_ROPE, t(p(self.qr), F32, [D, H, T]), [t(p(self.q), F32, [D, H, T]), post, None], rope_params))
            ops.append(b.make_op(b.OP_ROPE, t(p(self.kr), F32, [D, Hkv, T]), [t(p(self.k), F32, [D, Hkv, T]), post, None], rope_params))
            # KV store (llama-graph.cpp:1375-1397): 1-D views of the cache at kv_head
            kdst = t(p(lw["k_cache"]) + rs_row * kv_head, kvt, [Hkv * D * T])
            vdst = t(p(lw["v_cache"]) + rs_row * kv_head, kvt, [Hkv * D * T])
            ops.append(b.make_op(b.OP_CPY, kdst, [t(p(self.kr), F32, [D, Hkv, T])]))
            ops.append(b.make_op(b.OP_CPY, vdst, [t(p(self.v), F32, [Hkv * D, T])]))
            # flash attention: q permuted view [D, T, H], k/v 3-D views over n_kv cells (llama-graph.cpp:1411-1432)
            qv = t(p(self.qr), F32, [D, T, H], [4, D * H * 4, D * 4, D * H * T * 4])
            kv_ = t(p(lw["k_cache"]), kvt, [D, n_kv, Hkv], [BLOCK[kvt][1], rs_row, rs_head, rs_row * n_kv])
            vv = t(p(lw["v_cache"]), kvt, [D, n_kv, Hkv], [BLOCK[kvt][1], rs_row, rs_head, rs_row * n_kv])
            mk = t(p(self.mask_f16), F16, [n_kv, Tp])
            ops.append(b.make_op(b.OP_FLASH_ATTN_EXT, t(p(self.att), F32, [D, H, T]), [qv, kv_, vv, mk],
                                 [1.0 / math.sqrt(D), 0.0, 0.0]))
            ops.append(b.make_op(b.OP_MUL_MAT, t(p(self.tmpE), F32, [E, T]), [lw["wo"], t(p(self.att), F32, [H * D, T])]))
            if self.tp_world > 1:      # partial sums over this rank's heads -> sum over ranks (+ residual)
                ops.append(b.make_op(b.OP_ALLREDUCE, t(p(other), F32, [E, T]), [t(p(self.tmpE), F32, [E, T]), xin]))
            else:
                ops.append(b.make_op(b.OP_ADD, t(p(other), F32, [E, T]), [t(p(self.tmpE), F32, [E, T]), xin]))
            ffn_inp = t(p(other), F32, [E, T])
            # FFN
            ops.append(b.make_op(b.OP_RMS_NORM, t(p(self.cur), F32, [E, T]), [ffn_inp], [1e-5]))
            ops.append(b.make_op(b.OP_MUL, t(p(self.cur2), F32, [E, T]), [t(p(self.cur), F32, [E, T]), lw["ffn_norm"]]))
            nxt = self.resid2 if other is self.resid else self.resid
            if self.n_expert:
                # build_moe_ffn (llama-graph.cpp:834-952): router -> softmax -> top-k (argsort view) -> weights (get_rows, normalised) ->
                # up/gate experts -> silu * up -> down experts -> weighted sum over the used experts
                nE, nu = self.n_expert, self.n_used
                ops.append(b.make_op(b.OP_MUL_MAT, t(p(self.r_logits), F32, [nE, T]), [lw["gate_inp"], xn]))
                ops.append(b.make_op(b.OP_SOFT_MAX, t(p(self.r_probs), F32, [nE, T]), [t(p(self.r_logits), F32, [nE, T]), None], [1.0, 0.0]))
                ops.append(b.make_op(b.OP_ARGSORT, t(p(self.r_sel), I32, [nE, T]), [t(p(self.r_probs), F32, [nE, T])], [1]))
                sel = t(p(self.r_sel), I32, [nu, T], [4, nE * 4, nE * 4 * T, nE * 4 * T])          # ggml_top_k = view of the argsort
                ops.append(b.make_op(b.OP_GET_ROWS, t(p(self.r_w), F32, [1, nu, T]), [t(p(self.r_probs), F32, [1, nE, T]), sel]))
                ops.append(b.make_op(b.OP_SUM_ROWS, t(p(self.r_sum), F32, [1, T]), [t(p(self.r_w), F32, [nu, T])]))
                ops.append(b.make_op(b.OP_DIV, t(p(self.r_wn), F32, [nu, T]), [t(p(self.r_w), F32, [nu, T]), t(p(self.r_sum), F32, [1, T])]))
                x3 = t(p(self.cur2), F32, [E, 1, T])
                ops.append(b.make_op(b.OP_MUL_MAT_ID, t(p(self.u), F32, [FF, nu, T]), [lw["up_exps"], x3, sel]))
                ops.append(b.make_op(b.OP_MUL_MAT_ID, t(p(self.g), F32, [FF, nu, T]), [lw["gate_exps"], x3, sel]))
                ops.append(b.make_op(b.OP_SILU, t(p(self.gu), F32, [FF, nu, T]), [t(p(self.g), F32, [FF, nu, T])]))
                ops.append(b.make_op(b.OP_MUL, t(p(self.gu), F32, [FF, nu, T]), [t(p(self.u), F32, [FF, nu, T]), t(p(self.gu), F32, [FF, nu, T])]))
                ops.append(b.make_op(b.OP_MUL_MAT_ID, t(p(self.tmpE), F32, [E, nu, T]), [lw["down_exps"], t(p(self.gu), F32, [FF, nu, T]), sel]))
                ops.append(b.make_op(b.OP_MUL, t(p(self.tmpE), F32, [E, nu, T]), [t(p(self.tmpE), F32, [E, nu, T]), t(p(self.r_wn), F32, [1, nu, T])]))
                acc = t(p(self.tmpE), F32, [E, T], [4, E * nu * 4, E * nu * T * 4, E * nu * T * 4])
                for i in range(1, nu):
                    ei = t(p(self.tmpE) + i * E * 4, F32, [E, T], [4, E * nu * 4, E * nu * T * 4, E * nu * T * 4])
                    ops.append(b.make_op(b.OP_ADD, t(p(self.moe_out), F32, [E, T]), [acc, ei]))
                    acc = t(p(self.moe_out), F32, [E, T])
                ops.append(b.make_op(b.OP_ADD, t(p(nxt), F32, [E, T]), [acc, ffn_inp]))
                inp, other = nxt, (self.resid if nxt is self.resid2 else self.resid2)
                continue
            ops.append(b.make_op(b.OP_MUL_MAT, t(p(self.u), F32, [FF, T]), [lw["up"], xn]))
            ops.append(b.make_op(b.OP_MUL_MAT, t(p(self.g), F32, [FF, T]), [lw["gate"], xn]))
            ops.append(b.make_op(b.OP_SILU, t(p(self.gu), F32, [FF, T]), [t(p(self.g), F32, [FF, T])]))
            ops.append(b.make_op(b.OP_MUL, t(p(self.gu), F32, [FF, T]), [t(p(self.gu), F32, [FF, T]), t(p(self.u), F32, [FF, T])]))
            ops.append(b.make_op(b.OP_MUL_MAT, t(p(self.tmpE), F32, [E, T]), [lw["down"], t(p(self.gu), F32, [FF, T])]))
            if self.tp_world > 1:
                ops.append(b.make_op(b.OP_ALLREDUCE, t(p(nxt), F32, [E, T]), [t(p(self.tmpE), F32, [E, T]), ffn_inp]))
            else:
                ops.append(b.make_op(b.OP_ADD, t(p(nxt), F32, [E, T]), [t(p(self.tmpE), F32, [E, T]), ffn_inp]))
            inp, other = nxt, (self.resid if nxt is self.resid2 else self.resid2)
        To = T if n_outputs is None else min(T, n_outputs)
        off = (T - To) * E * 4
        ops.append(b.make_op(b.OP_RMS_NORM, t(p(self.cur), F32, [E, To]), [t(p(inp) + off, F32, [E, To])], [1e-5]))
        ops.append(b.make_op(b.OP_MUL, t(p(self.cur2), F32, [E, To]), [t(p(self.cur), F32, [E, To]), self.output_norm]))
        ops.append(b.make_op(b.OP_MUL_MAT, t(p(self.logits), F32, [V, To]), [self.output, t(p(self.cur2), F32, [E, To])]))
        return ops

    # ------------------------------------------------------------------------------------------------------------
    def step_bytes(self, n_tok, n_kv):
        """algorithmic HBM bytes of one ubatch (SURVEY.md 8d): every weight once, the visible KV cells once per layer
        (K and V), the KV rows written, f32 activations in/out of each matmul"""
        kv_read = 2 * self.L * n_kv * row_size(self.kv_type, self.Hkv * self.D)
        kv_write = 2 * self.L * n_tok * row_size(self.kv_type, self.Hkv * self.D)
        E, FF, V, HD, KD = self.E, self.FF, self.V, self.H * self.D, self.Hkv * self.D
        act = 4 * n_tok * (self.L * ((E + HD) + 2 * (E + KD) + (HD + E) + 2 * (E + FF) + (FF + E)) + (E + V))
        return dict(weights=self.weight_bytes, kv_read=kv_read, kv_write=kv_write, act=act,
                    total=self.weight_bytes + kv_read + kv_write + act)

    def set_inputs_slots_host(self, n_slots, depth, n_kv, rng):
        """continuous batching (n_parallel slots, one new token each): slot s owns cells [s*depth, (s+1)*depth) of the unified
        cache (llama_kv_cache_unified keeps a sequence's prompt contiguous), the n_slots new tokens go to cells
        [n_slots*depth, n_slots*depth + n_slots); mask row s allows its own cells and itself (llama-graph.cpp:1325 semantics)"""
        T = n_slots
        Tp = (T + 63) // 64 * 64
        kv_head = n_slots * depth
        emb = rng.standard_normal((T, self.E)).astype(np.float32)
        pos = np.full(T, depth, np.int32)
        mask = np.full((Tp, n_kv), -np.inf, np.float32)
        for s_ in range(T):
            mask[s_, s_ * depth:(s_ + 1) * depth] = 0.0
            mask[s_, kv_head + s_] = 0.0
        return emb, pos, mask, kv_head

    def set_inputs_host(self, n_tok, kv_head, n_kv, rng):
        """host-side inputs of one ubatch, as llama_context::set_inputs would produce: embeddings of the tokens
        (token_embd GET_ROWS runs on the CPU in llama.cpp, llama-model.cpp:1417), positions, causal mask"""
        Tp = (n_tok + 63) // 64 * 64
        emb = rng.standard_normal((n_tok, self.E)).astype(np.float32)
        pos = np.arange(kv_head, kv_head + n_tok, dtype=np.int32)
        mask = np.full((Tp, n_kv), -np.inf, np.float32)
        for i in range(n_tok):
            mask[i, :kv_head + i + 1] = 0.0
        return emb, pos, mask
