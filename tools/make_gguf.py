"""Synthetic random-init GGUF models of the shapes BASELINE.json names (no network, no reference code needed).

Writes GGUF v3 directly (format: llama.cpp/ggml/src/gguf.cpp) with
  * the llama / mixtral tensor set in the K_M mixtures llama-quant.cpp would produce
    (llama.cpp/src/llama-quant.cpp:129-131, 151-168, 235-255, 291-321): e.g. Q4_K_M = Q4_K everywhere, Q6_K for
    output.weight and for attn_v / ffn_down on the `use_more_bits` layers;
  * weights drawn directly in the quantised block layout (random quants and sub-scales, fp16 super-scales sized so a
    row has std ~ gain/sqrt(K)) -- "random-init weights of that architecture", seeded and reproducible;
  * a synthetic SPM vocabulary (<unk>, <s>, </s>, 256 byte tokens, then filler pieces) so llama.cpp's loader accepts it.

Usage: python tools/make_gguf.py --model llama3-8b --ftype q4_k_m --out /tmp/l3.gguf [--layers N] [--seed S]
"""
import argparse
import struct
import sys

import numpy as np

F32, F16, Q4_0, Q8_0, Q4_K, Q5_K, Q6_K, BF16 = 0, 1, 2, 8, 12, 13, 14, 30
BLOCK = {F32: (1, 4), F16: (1, 2), BF16: (1, 2), Q4_0: (32, 18), Q8_0: (32, 34), Q4_K: (256, 144), Q5_K: (256, 176), Q6_K: (256, 210)}
FTYPE_ID = {"f32": 0, "f16": 1, "bf16": 32, "q4_0": 2, "q8_0": 7, "q4_k_m": 15, "q5_k_m": 17}

MODELS = {
    #               L   E     H   Hkv D    FF     V       rope_base  n_expert n_used
    "tiny-d64":    (2,  256,  4,  2,  64,  512,   512,    10000.0,   0, 0),
    "tiny-d128":   (2,  512,  4,  2,  128, 1024,  512,    10000.0,   0, 0),
    "tiny-moe":    (2,  512,  4,  2,  128, 512,   512,    10000.0,   4, 2),
    "mid-d128":    (2,  2048, 16, 4,  128, 5632,  4096,   10000.0,   0, 0),
    "tinyllama":   (22, 2048, 32, 4,  64,  5632,  32000,  10000.0,   0, 0),
    "llama2-7b":   (32, 4096, 32, 32, 128, 11008, 32000,  10000.0,   0, 0),
    "llama3-8b":   (32, 4096, 32, 8,  128, 14336, 128256, 500000.0,  0, 0),
    "mixtral":     (32, 4096, 32, 8,  128, 14336, 32000,  1000000.0, 8, 2),
    "llama3-70b":  (80, 8192, 64, 8,  128, 28672, 128256, 500000.0,  0, 0),
}


def use_more_bits(i, n):
    return i < n // 8 or i >= 7 * n // 8 or (i - n // 8) % 3 == 2


def tensor_type(name, ftype, i_layer, n_layer, n_expert, n_gqa):
    """the type llama_tensor_get_type() would pick"""
    if name.endswith("_norm.weight") or "ffn_gate_inp" in name:
        return F32
    if ftype == "f32":
        return F32
    if ftype in ("f16", "bf16"):              # MOSTLY_F16 / MOSTLY_BF16: every matmul weight and token_embd
        return F16 if ftype == "f16" else BF16
    base = {"q4_0": Q4_0, "q8_0": Q8_0, "q4_k_m": Q4_K, "q5_k_m": Q5_K}[ftype]
    if name == "output.weight":
        return Q8_0 if ftype == "q8_0" else Q6_K
    if ftype in ("q4_k_m", "q5_k_m"):
        if "attn_v.weight" in name:
            if n_expert == 8:
                return Q8_0
            t = Q6_K if use_more_bits(i_layer, n_layer) else base
            if n_gqa >= 8 and t == Q4_K:          # 70B: attn_v is small and shared by 8 heads
                t = Q5_K
            return t
        if "attn_k.weight" in name and n_expert == 8:
            return Q8_0
        if "ffn_down" in name:
            return Q6_K if use_more_bits(i_layer, n_layer) else base
        if "attn_output.weight" in name and n_expert == 8 and ftype == "q4_k_m":
            return Q5_K
    return base


def to_16bit(t, x):
    """f32 array -> F16 or BF16 (round-to-nearest-even, as ggml_compute_fp32_to_bf16 for finite values) as uint16"""
    if t == F16:
        return x.astype(np.float16).view(np.uint16)
    u = x.astype(np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)


def rand_blocks(t, nrows, K, rng, amp):
    """random valid quantised rows whose dequantised values are roughly uniform in [-amp, amp]"""
    be, bb = BLOCK[t]
    nb = nrows * (K // be)
    blk = rng.integers(0, 256, size=(nb, bb), dtype=np.uint8)

    def f16(vals):
        return np.asarray(vals, np.float16).view(np.uint8).reshape(nb, 2)

    if t == Q4_0:
        blk[:, 0:2] = f16(rng.uniform(0.5, 1.5, nb) * amp / 8 * rng.choice([-1, 1], nb))
    elif t == Q8_0:
        blk[:, 0:2] = f16(rng.uniform(0.5, 1.5, nb) * amp / 127 * rng.choice([-1, 1], nb))
    elif t in (Q4_K, Q5_K):
        qmax = 15 if t == Q4_K else 31
        d = rng.uniform(0.5, 1.5, nb) * amp / (31.5 * qmax)
        blk[:, 0:2] = f16(d)
        blk[:, 2:4] = f16(d * qmax / 2)               # centres the block around zero on average
    elif t == Q6_K:
        blk[:, 208:210] = f16(rng.uniform(0.5, 1.5, nb) * amp / (64 * 32) * rng.choice([-1, 1], nb))
    return blk.reshape(-1)


class Writer:
    def __init__(self, path):
        self.f = open(path, "wb")
        self.kv = []
        self.tensors = []          # (name, ne, type, generator)

    @staticmethod
    def s(x):
        b = x.encode("utf-8")
        return struct.pack("<Q", len(b)) + b

    def add(self, key, vtype, payload):
        self.kv.append(self.s(key) + struct.pack("<I", vtype) + payload)

    def u32(self, k, v): self.add(k, 4, struct.pack("<I", v))
    def f32(self, k, v): self.add(k, 6, struct.pack("<f", v))
    def str(self, k, v): self.add(k, 8, self.s(v))
    def arr_str(self, k, vals): self.add(k, 9, struct.pack("<IQ", 8, len(vals)) + b"".join(self.s(v) for v in vals))
    def arr_f32(self, k, vals): self.add(k, 9, struct.pack("<IQ", 6, len(vals)) + np.asarray(vals, np.float32).tobytes())
    def arr_i32(self, k, vals): self.add(k, 9, struct.pack("<IQ", 5, len(vals)) + np.asarray(vals, np.int32).tobytes())

    def tensor(self, name, ne, t, gen):
        self.tensors.append((name, ne, t, gen))

    def finish(self):
        f = self.f
        f.write(struct.pack("<IIQQ", 0x46554747, 3, len(self.tensors), len(self.kv)))
        for kv in self.kv:
            f.write(kv)
        off = 0
        sizes = []
        for name, ne, t, _ in self.tensors:
            be, bb = BLOCK[t]
            n = int(np.prod(ne)) // be * bb
            f.write(self.s(name) + struct.pack("<I", len(ne)) + b"".join(struct.pack("<Q", d) for d in ne) + struct.pack("<IQ", t, off))
            sizes.append(n)
            off += (n + 31) // 32 * 32
        f.write(b"\0" * ((-f.tell()) % 32))
        total = 0
        for (name, ne, t, gen), n in zip(self.tensors, sizes):
            written = 0
            for chunk in gen():
                f.write(chunk.tobytes())
                written += chunk.nbytes
            assert written == n, (name, written, n)
            f.write(b"\0" * ((-n) % 32))
            total += n
        f.close()
        return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", required=True, choices=list(MODELS))
    ap.add_argument("--ftype", default="q4_k_m", choices=list(FTYPE_ID))
    ap.add_argument("--out", required=True)
    ap.add_argument("--layers", type=int, default=0, help="override the layer count (smaller files for tests)")
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--gain", type=float, default=1.0)
    ap.add_argument("--out-gain", type=float, default=4.0, help="extra gain on output.weight: widens logit margins (SURVEY appendix F)")
    a = ap.parse_args()
    L, E, H, Hkv, D, FF, V, rope_base, n_expert, n_used = MODELS[a.model]
    if a.layers:
        L = a.layers
    w = Writer(a.out)
    w.str("general.architecture", "llama")
    w.str("general.name", "synthetic-%s-%s" % (a.model, a.ftype))
    w.u32("llama.context_length", 8192 if a.model.startswith("llama3") else 4096)
    w.u32("llama.embedding_length", E)
    w.u32("llama.block_count", L)
    w.u32("llama.feed_forward_length", FF)
    w.u32("llama.attention.head_count", H)
    w.u32("llama.attention.head_count_kv", Hkv)
    w.u32("llama.rope.dimension_count", D)
    w.f32("llama.attention.layer_norm_rms_epsilon", 1e-5)
    w.f32("llama.rope.freq_base", rope_base)
    w.u32("llama.vocab_size", V)
    w.u32("general.file_type", FTYPE_ID[a.ftype])
    if n_expert:
        w.u32("llama.expert_count", n_expert)
        w.u32("llama.expert_used_count", n_used)
    # synthetic SPM vocabulary
    toks = ["<unk>", "<s>", "</s>"] + ["<0x%02X>" % i for i in range(256)]
    types = [2, 3, 3] + [6] * 256
    alphabet = "abcdefghijklmnopqrstuvwxyz"
    i = 0
    while len(toks) < V:
        n, s = i, ""
        while True:
            s = alphabet[n % 26] + s
            n //= 26
            if n == 0:
                break
        toks.append("▁" + s if i % 2 == 0 else s + "q")
        types.append(1)
        i += 1
    w.str("tokenizer.ggml.model", "llama")
    w.arr_str("tokenizer.ggml.tokens", toks)
    w.arr_f32("tokenizer.ggml.scores", [0.0] * 259 + [-float(j) for j in range(V - 259)])
    w.arr_i32("tokenizer.ggml.token_type", types)
    w.u32("tokenizer.ggml.bos_token_id", 1)
    w.u32("tokenizer.ggml.eos_token_id", 2)
    w.u32("tokenizer.ggml.unknown_token_id", 0)
    w.add("tokenizer.ggml.add_bos_token", 7, struct.pack("<B", 1))
    w.add("tokenizer.ggml.add_eos_token", 7, struct.pack("<B", 0))

    rng_master = np.random.default_rng(a.seed)

    def add_weight(name, K, N, n_mats, i_layer, gain=1.0):
        t = tensor_type(name, a.ftype, i_layer, L, n_expert, H // Hkv)
        seed = int(rng_master.integers(0, 2 ** 31))
        ne = [K, N] if n_mats == 1 else [K, N, n_mats]
        amp = gain * a.gain * np.sqrt(3.0 / K)

        def gen():
            rng = np.random.default_rng(seed)
            rows_total = N * n_mats
            step = max(1, (64 << 20) // max(1, K))          # ~64M elements per chunk
            for r0 in range(0, rows_total, step):
                nr = min(step, rows_total - r0)
                if t == F32:
                    yield (rng.uniform(-amp, amp, nr * K)).astype(np.float32)
                elif t in (F16, BF16):
                    yield to_16bit(t, rng.uniform(-amp, amp, nr * K).astype(np.float32))
                else:
                    yield rand_blocks(t, nr, K, rng, amp)
        w.tensor(name, ne, t, gen)

    def add_norm(name):
        seed = int(rng_master.integers(0, 2 ** 31))
        w.tensor(name, [E], F32, lambda: iter([(1.0 + 0.02 * np.random.default_rng(seed).standard_normal(E)).astype(np.float32)]))

    add_weight("token_embd.weight", E, V, 1, 0, gain=np.sqrt(E / 3.0))      # embeddings ~ unit scale
    for il in range(L):
        p = "blk.%d." % il
        add_norm(p + "attn_norm.weight")
        add_weight(p + "attn_q.weight", E, H * D, 1, il)
        add_weight(p + "attn_k.weight", E, Hkv * D, 1, il)
        add_weight(p + "attn_v.weight", E, Hkv * D, 1, il)
        add_weight(p + "attn_output.weight", H * D, E, 1, il)
        add_norm(p + "ffn_norm.weight")
        if n_expert:
            add_weight(p + "ffn_gate_inp.weight", E, n_expert, 1, il)
            add_weight(p + "ffn_gate_exps.weight", E, FF, n_expert, il)
            add_weight(p + "ffn_down_exps.weight", FF, E, n_expert, il)
            add_weight(p + "ffn_up_exps.weight", E, FF, n_expert, il)
        else:
            add_weight(p + "ffn_gate.weight", E, FF, 1, il)
            add_weight(p + "ffn_down.weight", FF, E, 1, il)
            add_weight(p + "ffn_up.weight", E, FF, 1, il)
    add_norm("output_norm.weight")
    add_weight("output.weight", E, V, 1, 0, gain=a.out_gain)
    total = w.finish()
    print("wrote %s: %.2f GiB of tensor data, %d layers" % (a.out, total / 2 ** 30, L), file=sys.stderr)


if __name__ == "__main__":
    main()
