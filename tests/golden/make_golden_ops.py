"""Golden vectors for the glue ops and flash attention of the hot path, produced by THE REFERENCE ITSELF: one-op ggml graphs
built through the reference's public C API (ggml.h) and executed by its CPU backend (oracle/_ref/libggml-{base,cpu}.so,
compiled from /root/reference/llama.cpp by oracle/Makefile) -- the same thing tests/test-backend-ops.cpp does per case.
The reference ships no golden vectors for these ops (SURVEY.md 8c); these fixtures pin oracle.c's restatements of
rms_norm, rope (norm/neox, freq factors, YaRN), soft_max, silu*mul and flash_attn_ext (f16 / q8_0 / q4_0 KV, GQA, -inf masks)
where the reference libraries are not around (the GPU box).  Run from the repo root:  python tests/golden/make_golden_ops.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import reflib as R  # noqa: E402

FA_CASES = [  # name, D, H, Hkv, n_q, n_kv, kv type
    ("f16_d128", 128, 8, 2, 3, 256, R.F16), ("q8_0_d128", 128, 8, 2, 3, 256, R.Q8_0), ("q4_0_d128", 128, 4, 4, 2, 128, R.Q4_0),
    ("f16_d64", 64, 4, 1, 1, 192, R.F16), ("f16_d128_long", 128, 2, 1, 1, 1024, R.F16),
]


def fa_inputs(rng, D, H, Hkv, n_q, n_kv, kvt):
    r = R.ref()
    q = rng.standard_normal((H, n_q, D)).astype(np.float32)
    kf = rng.standard_normal((Hkv * n_kv, D)).astype(np.float32)
    vf = rng.standard_normal((Hkv * n_kv, D)).astype(np.float32)
    if kvt == R.F16:
        kb, vb = kf.astype(np.float16).view(np.uint8).reshape(-1), vf.astype(np.float16).view(np.uint8).reshape(-1)
    else:
        kb, vb = r.quantize_weights(kvt, kf), r.quantize_weights(kvt, vf)
    n_q_pad = (n_q + 63) // 64 * 64
    mask = np.zeros((n_q_pad, n_kv), np.float16)
    for i in range(n_q):                       # causal tail + a masked-out slot in the middle (unified multi-sequence cache)
        mask[i, n_kv - (n_q - 1 - i) * 5 - 1 + 1:] = -np.inf
        mask[i, 40:72] = -np.inf
    return q, kb, vb, mask


def main():
    rng = np.random.default_rng(20261018)
    out = {}
    x = rng.standard_normal((5, 512)).astype(np.float32) * np.array([1, 1e-3, 30, 1, 1], np.float32)[:, None]
    out["rms_x"] = x
    out["rms_y"] = R.ref_rms_norm(x, 1e-5)
    xr = rng.standard_normal((3, 4, 128)).astype(np.float32)
    pos = np.array([0, 7, 4001], np.int32)
    ff = (1.0 + rng.uniform(0, 7, 64)).astype(np.float32)
    out["rope_x"], out["rope_pos"], out["rope_ff"] = xr, pos, ff
    out["rope_norm"] = R.ref_rope(xr, pos, 128, 0, 10000.0)
    out["rope_neox"] = R.ref_rope(xr, pos, 128, 2, 10000.0)
    out["rope_l3_ff"] = R.ref_rope(xr, pos, 128, 0, 500000.0, n_ctx_orig=8192, freq_factors=ff)
    out["rope_yarn"] = R.ref_rope(xr, pos, 128, 0, 10000.0, freq_scale=0.25, ext_factor=1.0, attn_factor=1.0, n_ctx_orig=2048)
    sx = rng.standard_normal((6, 96)).astype(np.float32) * 4
    sm = np.zeros((6, 96), np.float16)
    sm[:, 80:] = -np.inf
    sm[2, :10] = -np.inf
    out["sm_x"], out["sm_mask"] = sx, sm
    out["sm_y"] = R.ref_soft_max(sx, sm, 0.125)
    g_, u_ = rng.standard_normal(1000).astype(np.float32) * 3, rng.standard_normal(1000).astype(np.float32)
    out["silu_g"], out["silu_u"] = g_, u_
    out["silu_y"] = R.ref_silu_mul(g_, u_)
    for name, D, H, Hkv, n_q, n_kv, kvt in FA_CASES:
        q, kb, vb, mask = fa_inputs(rng, D, H, Hkv, n_q, n_kv, kvt)
        out["fa_q_" + name], out["fa_k_" + name], out["fa_v_" + name], out["fa_m_" + name] = q, kb, vb, mask
        out["fa_y_" + name] = R.ref_flash_attn(q, kb, vb, mask, D, n_kv, Hkv, kvt, kvt, 1.0 / np.sqrt(D))
    # the long f16 case goes to a file of its own: every fixture stays under 1 MB
    long = {k: out.pop(k) for k in list(out) if k.endswith("_f16_d128_long")}
    for name, arrays in (("ops_golden.npz", out), ("ops_golden_fa_long.npz", long)):
        path = os.path.join(HERE, name)
        np.savez_compressed(path, **arrays)
        print("wrote", path, "%.1f KB" % (os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()
