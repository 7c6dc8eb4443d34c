"""KV-cache maintenance graphs (SURVEY.md 8 f2): the op sequences llama.cpp emits for a context shift and for defragmentation
stay on the device and match the reference CPU backend.
  * K-shift  -- llama_context::build_rope_shift / build_kv_self_shift (llama-context.cpp:464-588): f16 K is re-rotated IN PLACE by
                ROPE on f16 with an I32 per-cell shift; quantised K goes CPY(q -> f32), ROPE(f32, in place), CPY(f32 -> q);
  * defrag   -- build_kv_self_defrag (llama-context.cpp:590-...): runs of cache rows moved by same-type CPY between 2-D views.
The expected K-shift bytes are the same graph computed by the oracle, whose dequantisers, rope and quantisers are pinned bit for bit
to the reference (tests/test_oracle_pin.py); where oracle/_ref is built they are also checked against the reference's CPU backend."""
import numpy as np
import pytest

import reflib as R
from util import dev_bytes, to_dev

pytestmark = pytest.mark.gpu


def quant_rows(t, x):
    return R.orc_quantize_act(t, x.reshape(-1, x.shape[-1]))


D, HKV, CELLS = 128, 8, 160
ROPE = dict(n_rot=128, mode=0, freq_base=500000.0, freq_scale=1.0, n_ctx_orig=8192)


def k_shift_ops(b200, kd, kt, shift_d, tmp_d):
    row = R.row_size(kt, D)
    kview = b200.tensor(kd.data_ptr(), kt, [D, HKV, CELLS], nb=[R.BLOCK[kt][1], row, row * HKV, row * HKV * CELLS])
    sh = b200.tensor(shift_d.data_ptr(), b200.I32, [CELLS])
    params = [0, ROPE["n_rot"], ROPE["mode"], 0, ROPE["n_ctx_orig"], ROPE["freq_base"], ROPE["freq_scale"], 0.0, 1.0, 32.0, 1.0]
    if kt == R.F16:
        return [b200.make_op(b200.OP_ROPE, kview, [kview, sh, None], params)]
    tmp = b200.tensor(tmp_d.data_ptr(), b200.F32, [D, HKV, CELLS])
    return [b200.make_op(b200.OP_CPY, tmp, [kview]), b200.make_op(b200.OP_ROPE, tmp, [tmp, sh, None], params), b200.make_op(b200.OP_CPY, kview, [tmp])]


def oracle_k_shift(kbytes, kt, shift):
    """build_rope_shift on the oracle: f16 K is widened, roped in f32 and rounded back (ggml-cpu rope_f16); quantised K goes
    dequantise -> rope -> quantise (ggml_cast, ggml_rope_ext_inplace, ggml_cpy)"""
    k = kbytes.view(np.float16).astype(np.float32) if kt == R.F16 else R.orc_dequantize(kt, kbytes, D)
    k = R.orc_rope(k.reshape(CELLS, HKV, D), shift, ROPE["n_rot"], ROPE["mode"], ROPE["freq_base"], freq_scale=ROPE["freq_scale"],
                   n_ctx_orig=ROPE["n_ctx_orig"])
    return k.astype(np.float16).view(np.uint8).reshape(-1) if kt == R.F16 else quant_rows(kt, k).reshape(-1)


@pytest.mark.parametrize("exact", [1, 0])
@pytest.mark.parametrize("kt", [R.F16, R.Q8_0, R.Q4_0])
def test_k_shift_graph_matches_reference(b200, ctx, kt, exact):
    rng = np.random.default_rng(40 + kt)
    k = rng.standard_normal((CELLS * HKV, D)).astype(np.float32)
    kb = k.astype(np.float16).view(np.uint8).reshape(-1) if kt == R.F16 else quant_rows(kt, k).reshape(-1)
    shift = rng.integers(-64, 65, CELLS).astype(np.int32)
    shift[::7] = 0
    want = oracle_k_shift(kb, kt, shift)
    if R.have_ref():
        assert np.array_equal(want, R.ref_k_shift(kb, kt, D, HKV, CELLS, shift, **ROPE))
    kd, sd, tmp = to_dev(kb), to_dev(shift), dev_bytes(CELLS * HKV * D * 4)
    ops = k_shift_ops(b200, kd, kt, sd, tmp)
    for o in ops:
        assert b200.supports(o), "K-shift op %d would fall back to the CPU backend" % o.op
    ctx.set_option("cpu_exact", exact)
    try:
        ctx.compute(ops)
        ctx.sync()
    finally:
        ctx.set_option("cpu_exact", 0)
    got = kd.cpu().numpy()
    if exact:
        assert np.array_equal(got, want), "cpu-exact mode: K-shift bytes must equal the reference CPU arithmetic's"
    else:
        # fast mode: CUDA sincosf instead of glibc's; a value may land one rounding step away
        if kt == R.F16:
            a, b = got.view(np.float16).astype(np.float32), want.view(np.float16).astype(np.float32)
            assert np.abs(a - b).max() <= 4e-3 and (got.view(np.uint16) != want.view(np.uint16)).mean() <= 0.02
        else:
            a, b = R.orc_dequantize(kt, got, D), R.orc_dequantize(kt, want, D)
            assert np.abs(a - b).max() <= 0.08 and (got != want).mean() <= 0.02
    # unshifted cells are bit-identical in either mode (rotation by zero is the identity: cos 0 = 1, sin 0 = 0)
    row = R.row_size(kt, D) * HKV
    keep = np.nonzero(shift == 0)[0]
    if kt == R.F16:
        assert all(np.array_equal(got[c * row:(c + 1) * row], kb[c * row:(c + 1) * row]) for c in keep)


@pytest.mark.parametrize("kt", [R.F16, R.Q8_0, R.Q4_0])
def test_defrag_row_moves(b200, ctx, kt):
    """runs of cells moved towards the front of the cache, K and (flash-attention layout) V alike: CPY between 2-D views of one buffer"""
    rng = np.random.default_rng(50 + kt)
    E = D * HKV
    row = R.row_size(kt, E)
    cache = rng.integers(0, 256, CELLS * row).astype(np.uint8)
    kd = to_dev(cache)
    moves = [(100, 10, 6), (130, 16, 20), (59, 50, 1)]           # (src cell, dst cell, run length), non-overlapping
    ops = []
    for src, dst, nm in moves:
        vs = b200.tensor(kd.data_ptr() + src * row, kt, [E, nm], nb=[R.BLOCK[kt][1], row, row * nm, row * nm])
        vd = b200.tensor(kd.data_ptr() + dst * row, kt, [E, nm], nb=[R.BLOCK[kt][1], row, row * nm, row * nm])
        ops.append(b200.make_op(b200.OP_CPY, vd, [vs]))
        assert b200.supports(ops[-1])
    ctx.compute(ops)
    ctx.sync()
    want = cache.copy()
    for src, dst, nm in moves:
        want[dst * row:(dst + nm) * row] = cache[src * row:(src + nm) * row]
    assert np.array_equal(kd.cpu().numpy(), want)
