"""CPU tests: the C oracle (oracle/oracle.c) against (a) golden vectors produced by the reference itself and
(b) the reference libraries directly when oracle/_ref is present.  Bit-exact for every integer/byte result."""
import os

import numpy as np
import pytest

import reflib as R

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "hotpath_golden.npz"))


@pytest.mark.parametrize("ta", [R.Q8_0, R.Q8_K, R.Q4_0])
def test_act_quantisers_match_golden(ta):
    got = R.orc_quantize_act(ta, G["act_x"])
    want = G["act_" + R.TYPE_NAMES[ta]]
    assert got.shape == want.shape
    assert np.array_equal(got, want), "quantiser %s differs from the reference bytes" % R.TYPE_NAMES[ta]


@pytest.mark.parametrize("K", [256, 1280])
@pytest.mark.parametrize("t", R.QUANT_TYPES)
def test_dequant_and_matmul_match_golden(t, K):
    name = "%s_%d" % (R.TYPE_NAMES[t], K)
    W, x = G["mm_W_" + name], G["mm_x_%d" % K]
    assert np.array_equal(R.orc_dequantize(t, W, K), G["mm_deq_" + name])
    out = R.orc_mul_mat(t, W, x, 12, K)
    want = G["mm_out_" + name]
    # the oracle's vec_dot follows the summation order of the reference's AVX2 build: bit-identical
    assert np.array_equal(out, want), np.abs(out - want).max()


def test_fp16_roundtrip_exhaustive():
    o = R.oracle()
    h = np.arange(65536, dtype=np.uint16)
    f = h.view(np.float16).astype(np.float32)
    for v in list(range(0, 65536, 97)) + [0, 1, 0x3ff, 0x400, 0x7bff, 0x7c00, 0x8000, 0xfbff]:
        got = o.orc_f16_to_f32(v)
        if np.isnan(f[v]):
            assert np.isnan(got)
        else:
            assert got == f[v]
            assert o.orc_f32_to_f16(float(f[v])) == v or f[v] == 0
    rng = np.random.default_rng(3)
    xs = np.concatenate([rng.standard_normal(2000) * 10.0 ** rng.integers(-8, 5, 2000), [65504.0, 65519.9, 65520.0, 1e-8, 6e-8]]).astype(np.float32)
    want = xs.astype(np.float16).view(np.uint16)
    got = np.array([o.orc_f32_to_f16(float(v)) for v in xs], np.uint16)
    assert np.array_equal(got, want)


@pytest.mark.skipif(not R.have_ref(), reason="oracle/_ref not built")
@pytest.mark.parametrize("t", R.QUANT_TYPES)
def test_block_sums_consistent_with_reference_vec_dot(t):
    """exact integer sums recombined in float must reproduce the reference vec_dot to float-order noise"""
    rng = np.random.default_rng(11 + t)
    r = R.ref()
    K, N = 2048, 4
    w = (rng.standard_normal((N, K)) * 0.05).astype(np.float32)
    x = rng.standard_normal((1, K)).astype(np.float32)
    W = r.quantize_weights(t, w).reshape(N, -1)
    ta = R.act_type(t)
    a_ref = r.quantize_act(ta, x)
    a_orc = R.orc_quantize_act(ta, x)
    assert np.array_equal(a_ref, a_orc)
    for n in range(N):
        want = r.vec_dot(t, W[n], a_ref[0], K)
        got = R.oracle().orc_vec_dot(t, W[n].ctypes.data, a_orc[0].ctypes.data, K)
        # the oracle restates the reference build's SIMD lane layout and FMA order: identical float, not just close
        assert np.float32(got) == np.float32(want), (got, want)


@pytest.mark.skipif(not R.have_ref(), reason="oracle/_ref not built")
def test_reference_own_quantize_tests_pass():
    """the reference's test-quantize-fns (dot error <= 0.02 etc.) passes on the oracle build"""
    import subprocess
    exe = os.path.join(R.REF_DIR, "test-quantize-fns")
    if not os.path.exists(exe):
        pytest.skip("tool not built")
    p = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stdout[-2000:]


# ----------------------------------------------------------------------------- glue ops + flash attention (tests/golden/ops_golden*.npz)
OPS = dict(np.load(os.path.join(os.path.dirname(__file__), "golden", "ops_golden.npz")))
OPS.update(np.load(os.path.join(os.path.dirname(__file__), "golden", "ops_golden_fa_long.npz")))


def _close(got, want, tol):
    return np.abs(got - want).max() <= tol * max(np.abs(want).max(), 1e-30)


def test_rms_norm_matches_reference_golden():
    assert np.array_equal(R.orc_rms_norm(OPS["rms_x"], 1e-5), OPS["rms_y"])


@pytest.mark.parametrize("name,kw", [
    ("rope_norm", dict(mode=0, freq_base=10000.0)), ("rope_neox", dict(mode=2, freq_base=10000.0)),
    ("rope_l3_ff", dict(mode=0, freq_base=500000.0, n_ctx_orig=8192, ff=True)),
    ("rope_yarn", dict(mode=0, freq_base=10000.0, freq_scale=0.25, ext_factor=1.0, n_ctx_orig=2048))])
def test_rope_matches_reference_golden(name, kw):
    kw = dict(kw)
    ff = OPS["rope_ff"] if kw.pop("ff", False) else None
    mode = kw.pop("mode")
    fb = kw.pop("freq_base")
    got = R.orc_rope(OPS["rope_x"], OPS["rope_pos"], 128, mode, fb, freq_factors=ff, **kw)
    # same libm on both sides, same multiplicative theta recurrence, no fp contraction in either build: bit-identical
    assert np.array_equal(got, OPS[name]), np.abs(got - OPS[name]).max()


def test_soft_max_matches_reference_golden():
    """bit-exact: ggml_v_expf on full groups of 8 whose horizontal sum enters the double accumulator as one float, expf on leftovers"""
    got = R.orc_soft_max(OPS["sm_x"], OPS["sm_mask"], 0.125)
    assert np.array_equal(got, OPS["sm_y"]), np.abs(got - OPS["sm_y"]).max()
    if R.have_ref():
        rng = np.random.default_rng(5)
        for n in (8, 13, 4, 100):                        # MoE router widths, leftovers only, mixed
            x = (rng.standard_normal((7, n)) * 3).astype(np.float32)
            assert np.array_equal(R.orc_soft_max(x, None, 1.0), R.ref_soft_max(x, None, 1.0)), n


def test_f32_weight_matmul_matches_live_reference():
    """the MoE router (F32 weights): ggml_vec_dot_f32's 4 x 8 FMA lanes + reduce tree + float leftovers, bit for bit"""
    if not R.have_ref():
        pytest.skip("oracle/_ref not built")
    rng = np.random.default_rng(6)
    for K, N, M in ((512, 8, 5), (4096, 8, 3), (100, 4, 2)):
        w = (rng.standard_normal((N, K)) * 0.05).astype(np.float32)
        x = rng.standard_normal((M, K)).astype(np.float32)
        assert np.array_equal(R.orc_mul_mat(R.F32, w.view(np.uint8).reshape(-1), x, N, K), R.ref_mul_mat_f32(w, x)), (K, N, M)


def test_silu_mul_matches_reference_golden():
    """bit-exact: the oracle restates the reference's polynomial ggml_v_expf, not libm's expf"""
    assert np.array_equal(R.orc_silu_mul(OPS["silu_g"], OPS["silu_u"]), OPS["silu_y"])
    big = np.array([-200, -130, -100, -90, -88, -20, 0, 1e-8, 20, 88, 90, 100, 130, 200, -0.0, 7.5], np.float32)
    if R.have_ref():
        assert np.array_equal(R.orc_silu_mul(big, np.ones_like(big)), R.ref_silu_mul(big, np.ones_like(big)))


FA_GOLD = [("f16_d128", 128, 8, 2, 3, 256, R.F16), ("q8_0_d128", 128, 8, 2, 3, 256, R.Q8_0), ("q4_0_d128", 128, 4, 4, 2, 128, R.Q4_0),
           ("f16_d64", 64, 4, 1, 1, 192, R.F16), ("f16_d128_long", 128, 2, 1, 1, 1024, R.F16)]


@pytest.mark.parametrize("name,D,H,Hkv,n_q,n_kv,kvt", FA_GOLD)
def test_flash_attn_matches_reference_golden(name, D, H, Hkv, n_q, n_kv, kvt):
    """the oracle restates the reference's SIMD summation order (K.Q through vec_dot), its FP16 accumulator for f16 V and its
    fused multiply-adds for quantised V: it must agree with the reference to the last bit for every cache type"""
    rs = R.row_size(kvt, D)
    got = R.orc_flash_attn(OPS["fa_q_" + name], OPS["fa_k_" + name].reshape(Hkv, n_kv, rs), OPS["fa_v_" + name].reshape(Hkv, n_kv, rs),
                           OPS["fa_m_" + name], D, n_kv, Hkv, kvt, kvt, 1.0 / np.sqrt(D))
    want = OPS["fa_y_" + name]
    assert np.array_equal(got, want), (np.abs(got - want).max(), np.abs(want).max())


@pytest.mark.skipif(not R.have_ref(), reason="oracle/_ref not built")
def test_flash_attn_oracle_vs_reference_live_random_shapes():
    rng = np.random.default_rng(77)
    for D, H, Hkv, n_q, n_kv, kvt in [(128, 4, 2, 2, 128, R.F16), (64, 2, 2, 3, 64, R.F16), (128, 4, 1, 1, 96, R.Q8_0)]:
        q = rng.standard_normal((H, n_q, D)).astype(np.float32)
        kf = rng.standard_normal((Hkv * n_kv, D)).astype(np.float32)
        vf = rng.standard_normal((Hkv * n_kv, D)).astype(np.float32)
        if kvt == R.F16:
            kb, vb = kf.astype(np.float16).view(np.uint8).reshape(-1), vf.astype(np.float16).view(np.uint8).reshape(-1)
        else:
            kb, vb = R.ref().quantize_weights(kvt, kf), R.ref().quantize_weights(kvt, vf)
        mask = np.zeros((64, n_kv), np.float16)
        mask[:, n_kv - 7:] = -np.inf
        rs = R.row_size(kvt, D)
        want = R.ref_flash_attn(q, kb, vb, mask, D, n_kv, Hkv, kvt, kvt, 0.09)
        got = R.orc_flash_attn(q, kb.reshape(Hkv, n_kv, rs), vb.reshape(Hkv, n_kv, rs), mask, D, n_kv, Hkv, kvt, kvt, 0.09)
        assert np.array_equal(got, want)
