"""Stage references for the fused decode layers (graph.cu fuse()), for tests (no GPU).

A fused launch keeps intermediates the test cannot observe: rms_norm(x) * w and h = silu(gate) * up before their matmul's
activation quantisation, the roped k and the v before the KV store.  The device's value of such an intermediate differs from the
reference's by summation order only, but a q8 / f16 rounding of it flips where the reference value sits within that difference of a
rounding boundary.  The bounds here admit exactly those flips and nothing else:

- `flip_bound`: per output row of a matmul over a quantised intermediate, 3e-6 * max|want| plus d_block * |W| summed over the
  ambiguous elements (one quantisation step each);
- `kv_bytes_ok`: KV-cache bytes must be the rounding of SOME value within `delta` of the reference, i.e. identical except where the
  reference is ambiguous, and there one step off.

Everything is built from reflib (the C oracle); the float64 product `mm_f64` stands in for orc_mul_mat where a whole vector feeds a
later stage (q / k / v, gate / up)."""
import numpy as np

import reflib as R

REL = 3e-6                     # the fast GEMV's bound against the oracle (tests/test_gpu_mulmat.py)


def norm_mul(x, w, eps):
    """RMS_NORM then MUL by the norm weight, as ggml rounds it: x [T, E] f32, w [E] -> f32 (two f32 multiplies)"""
    return (R.orc_rms_norm(x, eps) * np.asarray(w, np.float32)).astype(np.float32)


def decode_act(ta, blocks, K):
    """quantised activation rows (orc_quantize_act output, ta = Q8_0 / Q8_K) -> (values float64 [rows, K], step float64 [rows, K]):
    the dequantised value and the size of one quantisation step of every element"""
    blocks = np.ascontiguousarray(blocks, np.uint8)
    rows = blocks.shape[0]
    if ta == R.Q8_0:
        b = blocks.reshape(rows, K // 32, 34)
        d = b[:, :, 0:2].copy().view(np.float16).astype(np.float64)            # [rows, nb, 1]
        q = b[:, :, 2:34].view(np.int8).astype(np.float64)
    else:
        b = blocks.reshape(rows, K // 256, 292)
        d = b[:, :, 0:4].copy().view(np.float32).astype(np.float64)
        q = b[:, :, 4:260].view(np.int8).astype(np.float64)
    step = np.broadcast_to(np.abs(d), q.shape)
    return (q * d).reshape(rows, K), np.ascontiguousarray(step).reshape(rows, K)


def quant_act(t_w, x):
    """x f32 [T, K] quantised to the weight type's activation format: (values, steps) float64 [T, K]"""
    ta = R.act_type(t_w)
    return decode_act(ta, R.orc_quantize_act(ta, x), x.shape[1])


def dequant_rows(t, W, K, rows=None, chunk=2048):
    """float64 [len(rows), K] of the selected rows of W (uint8 bytes of N rows); all rows when rows is None"""
    rb = R.row_size(t, K)
    Wr = np.ascontiguousarray(W, np.uint8).reshape(-1, rb)
    if rows is not None:
        Wr = Wr[rows]
    out = np.empty((Wr.shape[0], K), np.float64)
    for r0 in range(0, Wr.shape[0], chunk):
        out[r0:r0 + chunk] = R.orc_dequantize(t, Wr[r0:r0 + chunk].reshape(-1), K)
    return out


def mm_f64(t, W, x, K, rows=None, chunk=2048):
    """float64 product of orc_dequantize(W) (rows selected, or all) and the decoded orc_quantize_act blocks of x [T, K] -> [T, rows]"""
    xa, _ = quant_act(t, x)
    rb = R.row_size(t, K)
    Wr = np.ascontiguousarray(W, np.uint8).reshape(-1, rb)
    if rows is not None:
        Wr = Wr[rows]
    out = np.empty((x.shape[0], Wr.shape[0]), np.float64)
    for r0 in range(0, Wr.shape[0], chunk):
        wd = R.orc_dequantize(t, Wr[r0:r0 + chunk].reshape(-1), K).astype(np.float64)
        out[:, r0:r0 + chunk] = xa @ wd.T
    return out


def ambiguous(h, t_w, eps, per_element=False):
    """elements of h [T, K] whose activation quantisation (quantize_row_q8_K_ref / quantize_row_q8_0 scale rule) may flip when h
    moves by eps * max|h| of its column: |frac(|h_k * iscale|) - 1/2| < eps * iscale * max|h|.  per_element: h_k moves by at most
    eps * |h_k| instead (a value rounded a few times on its own, like rms_norm(x) * w).  Returns (mask, step)."""
    h = np.asarray(h, np.float32)
    T, K = h.shape
    be = 32 if R.act_type(t_w) == R.Q8_0 else 256
    amax = np.abs(h).reshape(T, K // be, be).max(2, keepdims=True).astype(np.float64)
    iscale = np.where(amax > 0, 127.0 / np.where(amax > 0, amax, 1.0), 0.0)
    iscale = np.broadcast_to(iscale, (T, K // be, be)).reshape(T, K)
    u = np.abs(h.astype(np.float64)) * iscale
    mag = np.abs(h).astype(np.float64) if per_element else np.abs(h).max(1, keepdims=True).astype(np.float64)
    win = eps * iscale * mag
    mask = np.abs(u - np.floor(u) - 0.5) < win
    _, step = quant_act(t_w, h)
    return mask, step


def flip_bound(h_ref, act_type, W_deq, eps, scale=None, per_element=False):
    """tolerance [T, rows] of a matmul W_deq [rows, K] (weight type `act_type`'s activation format) over an intermediate h whose
    device value is within eps * max|h| of h_ref [T, K]: 3e-6 * scale (default max|want|) plus, per row, d_block(k) * |W[n, k]|
    summed over the ambiguous k (each may round one step the other way)"""
    h_ref = np.asarray(h_ref, np.float32)
    W_deq = np.asarray(W_deq, np.float64)
    if scale is None:
        xa, _ = quant_act(act_type, h_ref)
        scale = float(np.abs(xa @ W_deq.T).max())
    mask, step = ambiguous(h_ref, act_type, eps, per_element)
    return REL * scale + (mask * step) @ np.abs(W_deq).T


def _f16(x):
    return np.asarray(x, np.float64).astype(np.float32).astype(np.float16)


def kv_bytes_ok(got, x_ref, kvt, delta):
    """KV-store bytes `got` (uint8 [rows, row_size(kvt, n)]) of rows x_ref [rows, n] f32: True per element where the stored element
    is the rounding (f16 RNE / quantize_row_q8_0 / quantize_row_q4_0_ref) of some value within delta [rows, 1] of the reference,
    with the block scale taken from some block maximum within delta as well.  delta = 0 demands the reference bytes exactly; an
    all-zero block must store d = 0 and zero quants."""
    x = np.asarray(x_ref, np.float64)
    rows, n = x.shape
    dl = np.broadcast_to(np.asarray(delta, np.float64).reshape(-1, 1), (rows, 1))
    got = np.ascontiguousarray(got, np.uint8).reshape(rows, -1)
    if kvt == R.F16:
        g = got.view(np.float16).astype(np.float64)
        lo, hi = _f16(x - dl).astype(np.float64), _f16(x + dl).astype(np.float64)
        return (g >= lo) & (g <= hi)
    nb = n // 32
    xb = x.reshape(rows, nb, 32)
    db = np.broadcast_to(dl.reshape(rows, 1, 1), xb.shape)
    blk = got.reshape(rows, nb, -1)
    d = blk[:, :, 0:2].copy().view(np.float16).astype(np.float64)           # [rows, nb, 1]
    if kvt == R.Q8_0:
        amax = np.abs(xb).max(2, keepdims=True)
        m_lo, m_hi = np.maximum(amax - db[:, :, :1], 0.0), amax + db[:, :, :1]
        d_ok = (d >= _f16(m_lo / 127)) & (d <= _f16(m_hi / 127))
        q = blk[:, :, 2:34].view(np.int8).astype(np.float64)
        with np.errstate(divide="ignore", invalid="ignore"):
            c = [(xb + s) * 127.0 / m for s in (-db, db) for m in (np.where(m_lo > 0, m_lo, np.inf), np.where(m_hi > 0, m_hi, np.inf))]
        lo, hi = np.minimum.reduce(c), np.maximum.reduce(c)
        ok = (q >= np.ceil(lo - 0.5)) & (q <= np.floor(hi + 0.5))          # either rounding of a tie
        return (ok & d_ok).reshape(rows, n)
    # Q4_0: m = the element of largest magnitude (signed), d = m / -8, q = min(15, (int)(x / d + 8.5)), nibbles [j] | [j + 16] << 4
    idx = np.abs(xb).argmax(2)[:, :, None]
    m = np.take_along_axis(xb, idx, 2)
    sg = np.where(m < 0, -1.0, 1.0)
    m_lo, m_hi = m - sg * np.minimum(db[:, :, :1], np.abs(m)), m + sg * db[:, :, :1]        # same sign, |m| -/+ delta
    dd = np.sort(np.concatenate([_f16(m_lo / -8.0), _f16(m_hi / -8.0)], 2).astype(np.float64), 2)
    d_ok = (d >= dd[:, :, :1]) & (d <= dd[:, :, 1:])
    nib = blk[:, :, 2:18]
    q = np.concatenate([nib & 15, nib >> 4], 2).astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        c = [(xb + s) * -8.0 / mm for s in (-db, db) for mm in (np.where(m_lo != 0, m_lo, np.inf), np.where(m_hi != 0, m_hi, np.inf))]
    lo, hi = np.minimum.reduce(c), np.maximum.reduce(c)
    ok = (q >= np.minimum(15, np.floor(lo + 8.5))) & (q <= np.minimum(15, np.floor(hi + 8.5)))
    return (ok & d_ok).reshape(rows, n)
