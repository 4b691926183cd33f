"""Float64 references, per-element bounds and a dispatch mirror for K2 (csrc/gemm.cu), K4 (csrc/head.cu) and the fused
output layer + head (csrc/gemm_head.cu).  CPU only: NumPy, and torch on the host for the 16-bit conversions.

GEMM.  ``gemm_ref`` works from the kernel's own operand planes (bf16 / fp16 values read back from the device), so
operand rounding is not part of the tolerance.  It sums in float64 exactly the products the kernel sums
(gemm.cu:165-168): A_hi.W_hi; + A_hi.W_lo + A_lo.W_hi for NNAM_SPLIT_AW (no A_lo.W_lo term); + A_lo.W_hi for
NNAM_SPLIT_A; + A_hi.W_lo for NNAM_SPLIT_W; then the bias, then the activation (sigmoid as Chainer's
tanh(x/2)/2 + 1/2, gemm.cu:64).  Products of two bf16 or two fp16 values are exact in fp32, so what is left is
  * fp32 accumulation in the tensor core: tau * 2^-24 * S_ij, S = float64 sum of |products| over all passes,
    tau = TAU_SCALE * sqrt(passes * ceil(K / 16)) + TAU_BASE;
  * the bias add: 2^-23 * |z_ij| (z = value before the activation);
  * the activation: the bound above times the activation's largest slope (1, or 1/4 for sigmoid), plus 2 ulp of
    tanhf for sigmoid and tanh.
16-bit outputs are checked exactly against the same kernel's f32 output at the same tile width: bf16 / fp16 =
round-to-nearest-even of that value, fp16 saturating at +-65504 (cvt.rn.satfinite, ptx.cuh:292-296), and the split
output hi = bf16_rn(v), lo = bf16_rn(v - hi) (gemm.cu:293-299).

Head.  ``head_ref`` is the nnam_head formula in float64 (head.cu:108-215): the weighted ensemble, pre_normalize,
RPL4 with a real logaddexp, prior_scale * prior, the final log-softmax; ``map_rows`` applies the row-map semantics
(-1 drops a row, -2 - q zero-fills output row q).  The bound per element is
  HEAD_REL * 2^-24 * (|h| + sum |lse|) + n_lse * ((terms_per_lane + 6) * 2^-24 + HEAD_EXP)
with |h| the magnitude of every term that went into the logit (weighted inputs, their lse when pre-normalised, the
prior term), sum |lse| the row log-sum-exps subtracted on the way, n_lse the number of log-sum-exps computed (one per
pre-normalised input, one for RPL4, one final), terms_per_lane = 4 * NV4 (fast kernel) or NV (generic kernel), and
HEAD_EXP = 2^-21 for the error of ex2.approx / expf and logf.

Fused.  ``fused_bound`` = the GEMM bound of the element + the largest GEMM bound of its row (that error reaches the
log-sum-exp) + the head bound with terms_per_lane = 128 + 2 * cluster (a thread's online sum over its half-tile plus
the exchanged partials, gemm_head.cu:314-352).

Measured on an NVIDIA B200 (1000 W power limit), with TAU_SCALE = TAU_BASE = 8, HEAD_REL = 4 and HEAD_EXP = 2^-21,
the worst element of each check, as a fraction of its bound:
  * f32 GEMM outputs: 0.31 (single-CTA kernel, NNAM_SPLIT_AW) and 0.24 (pair kernel, NNAM_SPLIT_AW); 0.07 - 0.18 in
    the other modes;
  * head float32 rows 0.44, scores (nll) 0.33, compact row_ref 0.22 (every fast and generic instance);
  * fused rows 0.14, scores 0.12;
  * 16-bit GEMM outputs at the f32 launch's tile width: 0 differing elements (exact).
Two checks reach 0.9 - 1.0 by construction, because a half ulp of 16-bit rounding dominates their allowance: the
compact fp16 format (bound + half an fp16 ulp of |y - max|) and 16-bit GEMM outputs whose tile width differs from the
f32 launch's (bound + half an ulp of the output type).  A planted mistake is still rejected by at least 56 times its
bound (tests/test_gemm_reference_cpu.py).

Kernel models.  ``simulate_gemm`` accumulates in float32 per k-step of 16, by k-block of 64, tile by tile, pair
halves included; ``simulate_output`` stores 16-bit outputs; ``simulate_head_fast`` models the lanes and 4-wide
chunks of head_fast_kernel with its ragged end and its realignment of output rows; ``simulate_head_generic`` the
generic kernel's ensemble / RPL4 path.  Each takes ``mistake=`` to plant one error (tests/test_gemm_reference_cpu.py).
"""
from __future__ import annotations

import math

import numpy as np
import torch

# ----------------------------------------------------------------------------------------------------- constants
BM, BK, UK, MAX_BN = 128, 64, 16, 256          # gemm.cu:32-35
SM_COUNT = 148                                 # B200
OUT_BF16, OUT_BF16_SPLIT, OUT_F32, OUT_F16 = 0, 1, 2, 3
SPLIT_NONE, SPLIT_A, SPLIT_AW, SPLIT_W = 1, 2, 3, 4
OUT_NAMES = {OUT_F32: "f32", OUT_BF16: "bf16", OUT_F16: "f16", OUT_BF16_SPLIT: "split"}
# precision mode -> (nsplit, fp16 operands)
MODES = {"bf16": (SPLIT_NONE, False), "fp16": (SPLIT_NONE, True), "split_a": (SPLIT_A, False),
         "split_aw": (SPLIT_AW, False), "split_w": (SPLIT_W, False)}
ACTS = ("identity", "relu", "sigmoid", "tanh")
F16_MAX = 65504.0

TAU_SCALE, TAU_BASE = 8.0, 8.0
HEAD_REL, HEAD_EXP = 4.0, 2.0 ** -21
U24 = 2.0 ** -24


# ----------------------------------------------------------------------------------------------------- dispatch mirror
def pick_bn(n, box_cols):
    """gemm.cu:589-598 (without the NNAM_GEMM_BN tuning switch)."""
    tiles = (n + MAX_BN - 1) // MAX_BN
    bn = (n + tiles - 1) // tiles
    return (bn + box_cols - 1) // box_cols * box_cols


def use_2sm(M, N, K):
    """gemm.cu:614-628 with the default NNAM_GEMM_2SM / NNAM_GEMM_2SM_MINK."""
    return M >= 4096 and N >= 128 and K >= 384


def gemm_instance(M, N, K, out_kind, sm_count=SM_COUNT):
    """gemm.cu:684-735: the kernel, its tile width and tile counts and the grid of nnam_linear_bias_act."""
    box = 32 if out_kind == OUT_F32 else 64
    pair = use_2sm(M, N, K)
    bn = pick_bn(N, box)
    tiles_m = -(-M // (2 * BM)) if pair else -(-M // BM)
    tiles_n = -(-N // bn)
    total = tiles_m * tiles_n
    grid = 2 * min(total, sm_count // 2) if pair else min(total, sm_count)
    return dict(kernel="gemm_bias_act_2sm_kernel" if pair else "gemm_bias_act_kernel", pair=pair, bn=bn, box=box,
                tiles_m=tiles_m, tiles_n=tiles_n, tiles=total, grid=grid, k_blocks=-(-K // BK),
                ctas_per_tile=2 if pair else 1)


def head_instance(n_inputs, pre_normalize, rpl, ld_in, C, ld16=None, score=False):
    """head.cu:436-487 for 16-byte aligned buffers: ('fast', NV4, SCORE) or ('generic', NV, MULTI, SCORE)."""
    fast_ok = (n_inputs == 1 and not pre_normalize and not rpl and ld_in % 4 == 0 and C + 3 <= 2048
               and (ld16 is None or ld16 <= 2048))
    if fast_ok:
        need = C + 3
        nv4 = 1 if need <= 128 else 4 if need <= 512 else 8 if need <= 1024 else 15 if need <= 1920 else 16
        return ("fast", nv4, bool(score))
    nv = 4 if C <= 128 else 32 if C <= 1024 else 64
    return ("generic", nv, bool(n_inputs > 1 or pre_normalize), bool(score))


def head_terms_per_lane(inst):
    return 4 * inst[1] if inst[0] == "fast" else inst[1]


def head_kernel_name(inst):
    if inst[0] == "fast":
        return f"head_fast_kernel<{inst[1]}, {str(inst[2]).lower()}>"
    return f"head_kernel<{inst[1]}, {str(inst[2]).lower()}, {str(inst[3]).lower()}>"


def fused_cluster(N):
    """gemm_head.cu:578: one CTA per 256-column tile."""
    return -(-N // 256)


# ----------------------------------------------------------------------------------------------------- rounding
def bf16_rn(x):
    return torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(torch.bfloat16).float().numpy()


def f16_rn_sat(x):
    """cvt.rn.satfinite.f16.f32: round to nearest even, finite results clamp to +-65504 (NaN stays NaN)."""
    x = np.clip(np.asarray(x, np.float32), -F16_MAX, F16_MAX)
    return torch.from_numpy(np.ascontiguousarray(x)).to(torch.float16).float().numpy()


def bf16_trunc(x):
    b = np.ascontiguousarray(x, np.float32).view(np.uint32) & np.uint32(0xFFFF0000)
    return b.view(np.float32)


def f16_trunc(x):
    x = np.asarray(x, np.float32)
    r = x.astype(np.float16)
    over = np.abs(r.astype(np.float32)) > np.abs(x)
    r[over] = np.nextafter(r[over], np.float16(0))
    return r.astype(np.float32)


def ulp16(v, kind):
    """ulp of a bf16 / fp16 value at |v| (normal range)."""
    bits = 7 if kind == "bf16" else 10
    e = np.floor(np.log2(np.maximum(np.abs(v), 2.0 ** -14)))
    return 2.0 ** (e - bits)


# ----------------------------------------------------------------------------------------------------- operands
def make_gemm_operands(seed, M, N, K, mode, scale_z=1.0):
    """Seeded fp32 A (M, K), W (N, K), bias (N,) and the planes the kernel reads for ``mode``: a dict of float32
    arrays a_hi, a_lo, w_hi, w_lo (lo planes bf16, zero when the mode has none) and the 16-bit dtype."""
    rng = np.random.default_rng(seed)
    a = rng.standard_normal((M, K)).astype(np.float32)
    w = (scale_z * rng.standard_normal((N, K)) / math.sqrt(K)).astype(np.float32)
    b = rng.standard_normal(N).astype(np.float32)
    nsplit, f16 = MODES[mode]
    if f16:
        a_hi, w_hi = f16_rn_sat(a), f16_rn_sat(w)
    else:
        a_hi, w_hi = bf16_rn(a), bf16_rn(w)
    a_lo = bf16_rn(a - a_hi) if nsplit in (SPLIT_A, SPLIT_AW) else np.zeros_like(a)
    w_lo = bf16_rn(w - w_hi) if nsplit in (SPLIT_W, SPLIT_AW) else np.zeros_like(w)
    return dict(a_hi=a_hi, a_lo=a_lo, w_hi=w_hi, w_lo=w_lo, bias=b, nsplit=nsplit, f16=f16)


def pass_planes(nsplit):
    """(A plane, W plane) of each tensor pass, gemm.cu:165-168."""
    return {SPLIT_NONE: [("a_hi", "w_hi")], SPLIT_A: [("a_hi", "w_hi"), ("a_lo", "w_hi")],
            SPLIT_W: [("a_hi", "w_hi"), ("a_hi", "w_lo")],
            SPLIT_AW: [("a_hi", "w_hi"), ("a_hi", "w_lo"), ("a_lo", "w_hi")]}[nsplit]


# ----------------------------------------------------------------------------------------------------- GEMM reference
def act64(z, act):
    if act == "relu":
        return np.maximum(z, 0.0)
    if act == "sigmoid":
        return np.tanh(z * 0.5) * 0.5 + 0.5
    if act == "tanh":
        return np.tanh(z)
    return z


def gemm_products(planes, nsplit):
    """(float64 sum of products over the passes, float64 sum of |products|) for every element."""
    acc = S = None
    for ap, wp in pass_planes(nsplit):
        a = planes[ap].astype(np.float64)
        w = planes[wp].astype(np.float64)
        p, s = a @ w.T, np.abs(a) @ np.abs(w).T
        acc, S = (p, s) if acc is None else (acc + p, S + s)
    return acc, S


def gemm_ref(planes, bias, act, nsplit, products=None):
    """(y, z, S): y = act(z), z = sum of the pass products + bias, S = sum of |products|; all float64."""
    acc, S = products if products is not None else gemm_products(planes, nsplit)
    z = acc + (0.0 if bias is None else np.asarray(bias, np.float64)[None, :])
    return act64(z, act), z, S


def tau(K, nsplit):
    return TAU_SCALE * math.sqrt(len(pass_planes(nsplit)) * -(-K // UK)) + TAU_BASE


def gemm_bound(y, z, S, K, nsplit, act):
    """Per-element bound of an f32 GEMM output (module docstring)."""
    bz = tau(K, nsplit) * U24 * S + 2.0 ** -23 * np.abs(z)
    if act == "sigmoid":
        return 0.25 * bz + 2.0 ** -22 * np.abs(y) + U24
    if act == "tanh":
        return bz + 2.0 ** -22 * np.abs(y) + 2.0 ** -149
    return bz


def ratio(got, want, bound):
    """|got - want| / bound; non-finite results count as infinitely wrong."""
    got = np.asarray(got, np.float64)
    r = np.abs(got - want) / bound
    r[~np.isfinite(got)] = np.inf
    return r


def check_16bit(v32, hi, lo, out_kind):
    """Elements of a 16-bit output that differ from the exact conversion of the same kernel's f32 output ``v32``."""
    v32 = np.asarray(v32, np.float32)
    if out_kind == OUT_F16:
        bad = hi != f16_rn_sat(v32)
        return int(np.count_nonzero(bad | ~np.isfinite(hi)))
    want_hi = bf16_rn(v32)
    bad = hi != want_hi
    if out_kind == OUT_BF16_SPLIT:
        bad |= lo != bf16_rn((v32 - want_hi).astype(np.float32))
    return int(np.count_nonzero(bad))


# ----------------------------------------------------------------------------------------------------- GEMM model
def _bias_matrix(bias, M, N, inst, mistake):
    bias = np.asarray(bias, np.float32)
    if mistake not in ("bias_other_parity", "bias_shift_box"):
        return np.broadcast_to(bias[None, :], (M, N))
    bn, tiles_n, grid = inst["bn"], inst["tiles_n"], inst["grid"]
    per_tile_rows = BM * inst["ctas_per_tile"]
    n_units = grid // inst["ctas_per_tile"]
    out = np.zeros((M, N), np.float32)
    for t in range(inst["tiles"]):
        mb, nb = divmod(t, tiles_n)
        r0, c0 = mb * per_tile_rows, nb * bn
        cols = np.arange(c0, min(c0 + bn, N))
        if mistake == "bias_other_parity":  # the slice of this CTA's previous tile (zeros before its first tile)
            prev = t - n_units
            src = cols - c0 + (prev % tiles_n) * bn if prev >= 0 else None
            vals = np.zeros(len(cols), np.float32) if src is None else np.where(src < N, bias[np.minimum(src, N - 1)], 0)
        else:  # one store box to the right
            src = cols + inst["box"]
            vals = np.where((src < c0 + bn) & (src < N), bias[np.minimum(src, N - 1)], 0)
        out[r0:r0 + per_tile_rows, c0:c0 + len(cols)] = vals
    return out


def simulate_gemm(planes, M, N, K, act, out_kind=OUT_F32, mistake=None, padded=None):
    """float32 model of gemm_bias_act(_2sm)_kernel: per tile, k-step-of-16 partial products added to a float32
    accumulator in k order, pass after pass; then bias and activation in float32.  ``padded``: the A hi plane with its
    padding columns (NaN), read by the "read_padding" mistake."""
    nsplit = planes["nsplit"]
    inst = gemm_instance(M, N, K, out_kind)
    kb = inst["k_blocks"]
    a_idx, w_idx = np.arange(M), np.arange(N)
    if mistake == "follower_leader_rows":
        assert inst["pair"]
        a_idx = np.where((a_idx // BM) % 2 == 1, a_idx - BM, a_idx)
    if mistake == "same_w_half":
        assert inst["pair"]
        half = inst["bn"] // 2
        w_idx = np.where((w_idx % inst["bn"]) >= half, w_idx - half, w_idx)
    passes = list(pass_planes(nsplit))
    if mistake == "split_a_wlo":
        assert nsplit == SPLIT_A
        passes[1] = ("a_lo", "w_lo")
    if mistake == "aw_drop_hi_wlo":
        assert nsplit == SPLIT_AW
        passes.remove(("a_hi", "w_lo"))
    k_end = K
    if mistake == "drop_ragged_kblock":
        assert K % BK
        k_end = (kb - 1) * BK
    acc = np.zeros((M, N), np.float32)
    for ap, wp in passes:
        a = planes[ap].astype(np.float64)[a_idx]
        if mistake == "read_padding" and ap == "a_hi":
            a = np.concatenate((a, padded[:M, K:kb * BK].astype(np.float64)), axis=1)
        w = planes[wp].astype(np.float64)[w_idx]
        if a.shape[1] > w.shape[1]:
            w = np.concatenate((w, np.ones((N, a.shape[1] - w.shape[1]))), axis=1)
        kk = a.shape[1] if mistake == "read_padding" and ap == "a_hi" else k_end
        for k0 in range(0, kk, UK):
            acc = (acc + (a[:, k0:k0 + UK] @ w[:, k0:k0 + UK].T).astype(np.float32)).astype(np.float32)
    bias = _bias_matrix(planes["bias"], M, N, inst, mistake) if planes.get("bias") is not None else None
    v = acc
    if mistake == "act_before_bias":
        v = act32(v, act)
        return (v + bias).astype(np.float32) if bias is not None else v
    if bias is not None:
        v = (v + bias).astype(np.float32)
    if mistake == "sigmoid_tanh_x":
        return (np.tanh(v) * np.float32(0.5) + np.float32(0.5)).astype(np.float32)
    return act32(v, act)


def act32(v, act):
    v = np.asarray(v, np.float32)
    if act == "relu":
        return np.maximum(v, np.float32(0))
    if act == "sigmoid":
        return (np.tanh(v * np.float32(0.5)) * np.float32(0.5) + np.float32(0.5)).astype(np.float32)
    if act == "tanh":
        return np.tanh(v).astype(np.float32)
    return v


def simulate_output(v32, out_kind, mistake=None):
    """The epilogue's 16-bit stores of the f32 values ``v32``: (hi, lo) as float32 arrays."""
    v32 = np.asarray(v32, np.float32)
    if out_kind == OUT_F16:
        if mistake == "truncate":
            return f16_trunc(np.clip(v32, -F16_MAX, F16_MAX)), None
        if mistake == "f16_inf":
            return torch.from_numpy(np.ascontiguousarray(v32)).to(torch.float16).float().numpy(), None
        return f16_rn_sat(v32), None
    hi = bf16_trunc(v32) if mistake == "truncate" else bf16_rn(v32)
    if out_kind != OUT_BF16_SPLIT:
        return hi, None
    base = bf16_trunc(v32) if mistake == "split_lo_trunc_hi" else hi
    return hi, bf16_rn((v32 - base).astype(np.float32))


# ----------------------------------------------------------------------------------------------------- head reference
def _lse64(x):
    m = x.max(axis=1, keepdims=True)
    return (m + np.log(np.exp(x - m).sum(axis=1, keepdims=True)))[:, 0]


def head_ref(inputs, C, weights=None, pre_normalize=False, rpl=None, prior=None, prior_scale=1.0,
             final_normalize=True):
    """nnam_head in float64 over the logits rows (row map not applied).  Returns (y, mag, lse_sum, n_lse): the output,
    the magnitude of the terms in each logit, the sum of |lse| subtracted per row and the number of log-sum-exps."""
    xs = [np.asarray(x, np.float64)[:, :C] for x in inputs]
    k = len(xs)
    w = [1.0 / k] * k if weights is None else [float(np.float32(v)) for v in weights]
    h = np.zeros_like(xs[0])
    mag = np.zeros_like(xs[0])
    lse_sum = np.zeros(xs[0].shape[0])
    n_lse = 0
    for wk, x in zip(w, xs):
        lse = _lse64(x) if pre_normalize else np.zeros(x.shape[0])
        if pre_normalize:
            n_lse += 1
        h += wk * (x - lse[:, None])
        mag += abs(wk) * (np.abs(x) + np.abs(lse)[:, None])
    if rpl is not None:
        rw, rb, rlb = (np.asarray(t, np.float64)[:C] for t in rpl)
        lse = _lse64(h)
        n_lse += 1
        lse_sum += np.abs(lse)
        x = h - lse[:, None]
        g = x + x * rw + rb
        h = np.logaddexp(g, rlb)
        mag = (mag + np.abs(lse)[:, None]) * (1 + np.abs(rw)) + np.abs(rb) + np.abs(h)
    if prior is not None:
        pt = float(np.float32(prior_scale)) * np.asarray(prior, np.float64)[:C]
        h = h - pt
        mag = mag + np.abs(pt)
    if not final_normalize:
        return h, mag, lse_sum, n_lse
    lse = _lse64(h)
    n_lse += 1
    lse_sum += np.abs(lse)
    return h - lse[:, None], mag, lse_sum, n_lse


def head_bound(mag, lse_sum, n_lse, terms_per_lane):
    return HEAD_REL * U24 * (mag + lse_sum[:, None]) + n_lse * ((terms_per_lane + 6) * U24 + HEAD_EXP)


def map_rows(y, row_map, rows_out, fill=np.nan):
    """Row-map semantics of nnam_head_scatter: out[map[r]] = y[r]; -1 drops row r; -2 - q zero-fills row q.  Rows no
    entry names keep ``fill``.  Returns (out, written, zeroed)."""
    out = np.full((rows_out,) + y.shape[1:], fill)
    written = np.zeros(rows_out, bool)
    zeroed = np.zeros(rows_out, bool)
    for r, q in enumerate(row_map):
        if q >= 0:
            out[q] = y[r]
            written[q] = True
        elif q <= -2:
            out[-2 - q] = 0.0
            zeroed[-2 - q] = True
    return out, written, zeroed


def score_ref(y, bound, targets):
    """(nll, pred candidates): nll[r] = -y[r, t] (0 for t < 0) with its bound, and the float64 argmax with a flag
    telling whether the gap to the runner-up exceeds twice the bound (pred must then equal it)."""
    rows = np.arange(y.shape[0])
    t = np.maximum(targets, 0)
    nll = np.where(targets >= 0, -y[rows, t], 0.0)
    nb = np.where(targets >= 0, bound[rows, t], 0.0)
    order = np.argsort(-y, axis=1, kind="stable")
    top = order[:, 0]
    if y.shape[1] > 1:
        gap = y[rows, top] - y[rows, order[:, 1]]
        sure = gap > 2 * (bound[rows, top] + bound[rows, order[:, 1]])
    else:
        sure = np.ones(y.shape[0], bool)
    return nll, nb, top, sure


def fused_bound(gb, hbound):
    """GEMM bound of the element + largest GEMM bound of its row + head bound."""
    return gb + gb.max(axis=1, keepdims=True) + hbound


# ----------------------------------------------------------------------------------------------------- head models
LOG2E = np.float32(1.4426950408889634)


def _warp_sum(lane_vals):
    """xor-butterfly sum over the last axis (32 lanes) in float32."""
    v = lane_vals.astype(np.float32)
    for o in (16, 8, 4, 2, 1):
        v = (v + v[..., np.arange(32) ^ o]).astype(np.float32)
    return v[..., 0]


def simulate_head_fast(x, C, nv4, w0=1.0, prior=None, prior_scale=1.0, ld_out=None, mistake=None):
    """float32 model of head_fast_kernel (float32 rows form) for rows of ``x`` (rows, >= C).  Chunk k = lane + 32 i
    holds columns 4k .. 4k+3; columns >= C are -inf (head.cu:279-288).  ``ld_out``: pitch of the output rows, for the
    realignment of rows that start off a 16-byte boundary."""
    rows = x.shape[0]
    width = 128 * nv4
    v = np.full((rows, width), np.float32(0.0) if mistake == "ragged_zero" else -np.inf, np.float32)
    v[:, :C] = np.asarray(x, np.float32)[:, :C]
    if w0 != 1.0 and mistake != "ignore_weight":
        v[:, :C] = v[:, :C] * np.float32(w0)
    if prior is not None:
        ps = np.float32(1.0 if mistake == "ignore_prior_scale" else prior_scale)
        v[:, :C] = (v[:, :C] - (ps * np.asarray(prior, np.float32)[:C]).astype(np.float32)).astype(np.float32)
    mx = v.max(axis=1)
    with np.errstate(over="ignore", invalid="ignore"):
        if mistake == "no_max_sub":
            e = np.exp2(v * LOG2E).astype(np.float32)
        else:
            e = np.exp2((v * LOG2E - (mx * LOG2E)[:, None]).astype(np.float32)).astype(np.float32)
        e4 = e.reshape(rows, nv4, 32, 4)  # [row, i, lane, element]
        s0 = np.zeros((rows, 32), np.float32)
        s1 = np.zeros((rows, 32), np.float32)
        for i in range(nv4):
            s0 = (s0 + (e4[:, i, :, 0] + e4[:, i, :, 1]).astype(np.float32)).astype(np.float32)
            s1 = (s1 + (e4[:, i, :, 2] + e4[:, i, :, 3]).astype(np.float32)).astype(np.float32)
        s = _warp_sum((s0 + s1).astype(np.float32))
        lse = (np.log(s) if mistake == "no_max_sub" else mx + np.log(s)).astype(np.float32)
        y = (v[:, :C] - lse[:, None]).astype(np.float32)
    if mistake == "realign_wrong_neighbour":
        # the first `a` columns of each aligned output chunk come from the right neighbour's chunk instead of the left
        y2 = y.copy()
        for r in range(rows):
            a = (r * ld_out) % 4
            for c in range(C):
                if (c + a) % 4 < a:
                    y2[r, c] = y[r, c + 8] if c + 8 < C else 0.0
        y = y2
    return y


def simulate_head_generic(inputs, C, weights, pre_normalize=False, rpl=None, prior=None, prior_scale=1.0,
                          final_normalize=True, mistake=None):
    """float32 model of head_kernel<NV, MULTI, false> (ensemble, pre_normalize, RPL4, prior, final log-softmax)."""
    f = np.float32

    def lse32(x):
        m = x.max(axis=1, keepdims=True)
        return (m + np.log(np.exp(x - m).sum(axis=1, keepdims=True, dtype=f))).astype(f)

    h = np.zeros((inputs[0].shape[0], C), f)
    for wk, x in zip(weights, inputs):
        t = np.asarray(x, f)[:, :C]
        lse = lse32(t) if pre_normalize and mistake != "skip_pre_normalize" else f(0)
        h = (h + f(wk) * (t - lse)).astype(f)
    if rpl is not None:
        rw, rb, rlb = (np.asarray(a, f)[:C] for a in rpl)
        x = (h - lse32(h)).astype(f)
        g = (x + x * rw + rb).astype(f)
        mx, mn = np.maximum(g, rlb), np.minimum(g, rlb)
        h = mx if mistake == "rpl_max" else (mx + np.log(f(1) + np.exp(mn - mx))).astype(f)
    if prior is not None:
        h = (h - f(prior_scale) * np.asarray(prior, f)[:C]).astype(f)
    return (h - lse32(h)).astype(f) if final_normalize else h


# ----------------------------------------------------------------------------------------------------- head data
def make_head_logits(seed, rows, C, n_inputs=1, scale=3.0):
    """Seeded logits rows: every 7th row shifted so that its maximum is negative (about -40), every 11th so that its
    maximum is about +200; the rest standard normal times ``scale``."""
    rng = np.random.default_rng(seed)
    xs = []
    for _ in range(n_inputs):
        x = scale * rng.standard_normal((rows, C))
        r = np.arange(rows)
        x[r % 7 == 3] -= x[r % 7 == 3].max(axis=1, keepdims=True) + 40.0
        x[r % 11 == 5] += 200.0 - x[r % 11 == 5].max(axis=1, keepdims=True)
        xs.append(x.astype(np.float32))
    return xs


def make_head_extras(seed, C):
    """prior (log-priors around -3) and RPL4 parameters (W, b around 0, lb = -6)."""
    rng = np.random.default_rng(seed + 1)
    prior = (-3.0 + rng.standard_normal(C)).astype(np.float32)
    rpl = ((0.1 * rng.standard_normal(C)).astype(np.float32), (0.1 * rng.standard_normal(C)).astype(np.float32),
           np.full(C, -6.0, np.float32))
    return prior, rpl
