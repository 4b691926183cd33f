"""torch-tensor front ends of the C-ABI ops.  PyTorch is plumbing only: it owns device memory and
streams; all arithmetic happens in libnnam_b200.so."""
from __future__ import annotations

import ctypes

import torch

from . import _native
from ._native import NnamError, check

ACT = {"identity": 0, "none": 0, None: 0, "relu": 1, "sigmoid": 2, "tanh": 3}
OUT_BF16, OUT_BF16_SPLIT, OUT_F32, OUT_F16 = 0, 1, 2, 3   # NNAM_OUT_*
ELEM_BF16, ELEM_F16 = 0, 1                                # NNAM_ELEM_*
SPLIT_NONE, SPLIT_A, SPLIT_AW, SPLIT_W = 1, 2, 3, 4       # NNAM_SPLIT_* (operand passes of K2)
E16 = {ELEM_BF16: torch.bfloat16, ELEM_F16: torch.float16}


def out_dtype(out_kind):
    """torch dtype of the (hi) output buffer of a kernel asked for ``out_kind``."""
    return {OUT_F32: torch.float32, OUT_F16: torch.float16}.get(out_kind, torch.bfloat16)


# launch accounting (bench.py: gpu_launches, per-kernel CUDA-event timing for the roofline block)
LAUNCHES = {"splice": 0, "convert": 0, "gemm": 0, "head": 0, "rnn": 0, "cell": 0}
PROFILE = None  # set to a list to record (kernel, start_event, end_event, work) per launch


class _Prof:
    def __init__(self, name, work):
        self.name, self.work = name, work

    def __enter__(self):
        LAUNCHES[self.name] += 1
        if PROFILE is not None:
            self.s = torch.cuda.Event(enable_timing=True)
            self.e = torch.cuda.Event(enable_timing=True)
            self.s.record()
        return self

    def __exit__(self, *exc):
        if PROFILE is not None:
            self.e.record()
            PROFILE.append((self.name, self.s, self.e, self.work))
        return False


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _req(t, dtype, name):
    if t is None:
        return
    if not t.is_cuda:
        raise NnamError(f"{name}: expected a CUDA tensor (there is no CPU path)")
    if t.dtype != dtype:
        raise NnamError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if t.dim() == 2 and t.stride(1) != 1:
        raise NnamError(f"{name}: rows must be contiguous")


def round_up(v, m):
    return (v + m - 1) // m * m


def splice_transform(x, n_total, splice, add_shift=None, rescale=None, ivec=None, f0=0, f1=None, x_row0=0,
                     out_kind=OUT_F32, ldo=None, out=None):
    """K1.  x: (rows, dim) f32 holding global rows [x_row0, x_row0+rows); returns (out_hi, out_lo)."""
    _req(x, torch.float32, "x")
    _req(ivec, torch.float32, "ivec")
    _req(add_shift, torch.float32, "add_shift")
    _req(rescale, torch.float32, "rescale")
    if not x.is_contiguous() or (ivec is not None and not ivec.is_contiguous()):
        raise NnamError("splice: x and ivec must be contiguous")
    rows, dim = x.shape
    if f1 is None:
        f1 = n_total
    ivec_dim = 0 if ivec is None else ivec.shape[1]
    cols = (2 * splice + 1) * dim + ivec_dim
    if add_shift is not None and add_shift.numel() != (2 * splice + 1) * dim:
        raise NnamError(f"splice: transform has {add_shift.numel()} entries, expected {(2 * splice + 1) * dim}")
    if ivec is not None and ivec.shape[0] < f1 - f0:
        raise NnamError("splice: ivec has fewer rows than the frame range")
    if ldo is None:
        ldo = cols if out_kind == OUT_F32 else round_up(cols, 8)
    n = f1 - f0
    dt = out_dtype(out_kind)
    if out is None:
        hi = torch.empty((n, ldo), dtype=dt, device=x.device)
        lo = torch.empty((n, ldo), dtype=dt, device=x.device) if out_kind == OUT_BF16_SPLIT else None
    else:
        hi, lo = out
    _req(hi, dt, "out")
    work = n * (dim * 4 + ivec_dim * 4 + cols * (2 if out_kind in (OUT_BF16, OUT_F16) else 4))
    with _Prof("splice", work):
        check(_native.lib().nnam_splice_transform(_ptr(x), x_row0, rows, n_total, dim, splice, _ptr(add_shift),
                                              _ptr(rescale), _ptr(ivec), ivec_dim, f0, f1, _ptr(hi), _ptr(lo),
                                                  ldo, out_kind, _stream()))
    return hi, lo


def convert_f32(src, out_kind=OUT_BF16, ldd=None, out=None):
    """fp32 (rows, cols) -> 16-bit hi (bf16 or fp16; and bf16 lo) with zero padding up to ldd columns."""
    _req(src, torch.float32, "src")
    rows, cols = src.shape
    if ldd is None:
        ldd = round_up(cols, 8)
    if out is None:
        hi = torch.empty((rows, ldd), dtype=out_dtype(out_kind), device=src.device)
        lo = torch.empty((rows, ldd), dtype=torch.bfloat16, device=src.device) if out_kind == OUT_BF16_SPLIT else None
    else:
        hi, lo = out
    _req(hi, out_dtype(out_kind), "out")
    with _Prof("convert", rows * cols * 4):
        check(_native.lib().nnam_convert_f32(_ptr(src), rows, cols, src.stride(0), _ptr(hi), _ptr(lo), ldd,
                                             out_kind, _stream()))
    return hi, lo


def linear_bias_act(a_hi, a_lo, w_hi, w_lo, bias, M, N, K, act="identity", out_kind=OUT_BF16, nsplit=1, out=None,
                    ldo=None, elem=ELEM_BF16):
    """K2.  out = act(A . W^T + bias).  a_*: (>=M, lda), w_*: (>=N, ldw) K-major; hi planes in ``elem`` (bf16 / fp16),
    lo planes bf16.  ``nsplit``: SPLIT_* operand passes."""
    for t, n in ((a_hi, "a_hi"), (w_hi, "w_hi")):
        _req(t, E16[elem], n)
    for t, n in ((a_lo, "a_lo"), (w_lo, "w_lo")):
        _req(t, torch.bfloat16, n)
    _req(bias, torch.float32, "bias")
    if nsplit in (SPLIT_NONE, SPLIT_W):
        a_lo = None
    if nsplit in (SPLIT_NONE, SPLIT_A):
        w_lo = None
    if ldo is None:
        ldo = round_up(N, 16) if out is None else out[0].stride(0)
    dt = out_dtype(out_kind)
    if out is None:
        hi = torch.empty((M, ldo), dtype=dt, device=a_hi.device)
        lo = torch.empty((M, ldo), dtype=dt, device=a_hi.device) if out_kind == OUT_BF16_SPLIT else None
    else:
        hi, lo = out
    _req(hi, dt, "out")
    with _Prof("gemm", 2.0 * M * N * K):  # ALGORITHMIC flops (one pass, unpadded), whatever nsplit is
        check(_native.lib().nnam_linear_bias_act(_ptr(a_hi), _ptr(a_lo), a_hi.stride(0), _ptr(w_hi), _ptr(w_lo),
                                                 w_hi.stride(0), _ptr(bias), _ptr(hi), _ptr(lo), ldo, M, N, K,
                                                 ACT[act], out_kind, nsplit, elem, _stream()))
    return hi, lo


FUSED_HEAD_MAX_CLASSES = 2048  # eight 256-column tiles: one thread-block cluster spans a row


def _req_score(score):
    targets, nll, pred = score
    _req(targets, torch.int32, "targets")
    _req(nll, torch.float32, "nll")
    _req(pred, torch.int32, "pred")
    if targets is None or nll is None or pred is None:
        raise NnamError("scoring needs targets, nll and pred tensors")
    return targets, nll, pred


def linear_logsoftmax(a_hi, a_lo, w_hi, w_lo, bias, M, N, K, prior=None, prior_scale=1.0, nsplit=1, elem=ELEM_BF16,
                      out=None, out16=None, out_row_map=None, score=None):
    """K2 + K4 fused for one net without RPL: log_softmax(A . W^T + bias - prior_scale * prior) straight from the
    accumulators (the float32 logits never go to HBM).  ``out``: float32 (rows_out, >= N) tensor, or ``out16`` = (fp16
    (rows_out, ld16), f32 (rows_out,)) for the compact transfer format; ``out_row_map`` as in :func:`head`.
    ``score`` = (int32 targets, f32 nll, int32 pred), each indexed by output row, scores the rows the float32 form would
    write instead of writing them (nnam_linear_logsoftmax_score); returns that tuple."""
    for t, n in ((a_hi, "a_hi"), (w_hi, "w_hi")):
        _req(t, E16[elem], n)
    for t, n in ((a_lo, "a_lo"), (w_lo, "w_lo")):
        _req(t, torch.bfloat16, n)
    _req(bias, torch.float32, "bias")
    _req(prior, torch.float32, "prior")
    _req(out_row_map, torch.int32, "out_row_map")
    if nsplit in (SPLIT_NONE, SPLIT_W):
        a_lo = None
    if nsplit in (SPLIT_NONE, SPLIT_A):
        w_lo = None
    if score is not None:
        targets, nll, pred = _req_score(score)
        with _Prof("gemm", 2.0 * M * N * K):
            check(_native.lib().nnam_linear_logsoftmax_score(
                _ptr(a_hi), _ptr(a_lo), a_hi.stride(0), _ptr(w_hi), _ptr(w_lo), w_hi.stride(0), _ptr(bias), _ptr(prior),
                float(prior_scale), _ptr(targets), _ptr(nll), _ptr(pred), _ptr(out_row_map), M, N, K, nsplit, elem,
                _stream()))
        return score
    o16 = ref = None
    if out16 is not None:
        o16, ref = out16
        _req(o16, torch.float16, "out16")
        _req(ref, torch.float32, "row_ref")
        out = None
    else:
        if out is None:
            out = torch.empty((M, N), dtype=torch.float32, device=a_hi.device)
        _req(out, torch.float32, "out")
    with _Prof("gemm", 2.0 * M * N * K):
        check(_native.lib().nnam_linear_logsoftmax(_ptr(a_hi), _ptr(a_lo), a_hi.stride(0), _ptr(w_hi), _ptr(w_lo),
                                                   w_hi.stride(0), _ptr(bias), _ptr(prior), float(prior_scale), _ptr(out),
                                                   0 if out is None else out.stride(0), _ptr(o16),
                                                   0 if o16 is None else o16.stride(0), _ptr(ref), _ptr(out_row_map),
                                                   M, N, K, nsplit, elem, _stream()))
    return out16 if out16 is not None else out


def head(logits, n_classes, rows=None, weights=None, pre_normalize=False, rpl=None, prior=None, prior_scale=1.0,
         final_normalize=True, out=None, out_row_map=None, out16=None):
    """K4.  logits: one (rows, ld) f32 tensor or a list of them (ensemble).  ``out16`` = (fp16 (rows_out, ld16), f32
    (rows_out,)) selects the compact transfer format (nnam_head_f16) instead of the float32 ``out``."""
    if isinstance(logits, torch.Tensor):
        logits = [logits]
    for t in logits:
        _req(t, torch.float32, "logits")
    ld_in = logits[0].stride(0)
    if any(t.stride(0) != ld_in for t in logits):
        raise NnamError("head: all inputs must share one leading dimension")
    if rows is None:
        rows = logits[0].shape[0]
    if out16 is not None:
        o16, ref = out16
        _req(o16, torch.float16, "out16")
        _req(ref, torch.float32, "row_ref")
    elif out is None:
        out = torch.empty((rows, n_classes), dtype=torch.float32, device=logits[0].device)
    _req(out, torch.float32, "out")
    k = len(logits)
    ptrs = (ctypes.c_void_p * k)(*[t.data_ptr() for t in logits])
    wts = None if weights is None else (ctypes.c_float * k)(*[float(w) for w in weights])
    rw = rb = rlb = None
    if rpl is not None:
        rw, rb, rlb = rpl
        for t in (rw, rb, rlb):
            _req(t, torch.float32, "rpl")
    _req(prior, torch.float32, "prior")
    _req(out_row_map, torch.int32, "out_row_map")
    if out16 is not None:
        with _Prof("head", rows * n_classes * (4 * k + 2)):
            check(_native.lib().nnam_head_f16(ptrs, wts, k, ld_in, int(bool(pre_normalize)), _ptr(rw), _ptr(rb),
                                              _ptr(rlb), _ptr(prior), float(prior_scale), int(bool(final_normalize)),
                                              _ptr(o16), o16.stride(0), _ptr(ref), rows, n_classes, _ptr(out_row_map),
                                              _stream()))
        return out16
    with _Prof("head", rows * n_classes * 4 * (k + 1)):
        if out_row_map is None:
            check(_native.lib().nnam_head(ptrs, wts, k, ld_in, int(bool(pre_normalize)), _ptr(rw), _ptr(rb),
                                          _ptr(rlb), _ptr(prior), float(prior_scale), int(bool(final_normalize)),
                                          _ptr(out), out.stride(0), rows, n_classes, _stream()))
        else:
            check(_native.lib().nnam_head_scatter(ptrs, wts, k, ld_in, int(bool(pre_normalize)), _ptr(rw), _ptr(rb),
                                                  _ptr(rlb), _ptr(prior), float(prior_scale),
                                                  int(bool(final_normalize)), _ptr(out), out.stride(0), rows,
                                                  n_classes, _ptr(out_row_map), _stream()))
    return out


def head_score(logits, n_classes, targets, nll, pred, rows=None, weights=None, pre_normalize=False, rpl=None, prior=None,
               prior_scale=1.0, final_normalize=True, out_row_map=None):
    """K4 scored against frame targets (nnam_head_score): the rows :func:`head` would write are reduced to nll[q] =
    -y[q][targets[q]] (0 for target -1) and pred[q] = argmax_c y[q][c] (lowest column on ties); a zero-fill map entry
    -2 - q gives nll 0, pred -1.  ``targets`` / ``nll`` / ``pred``: int32 / f32 / int32, indexed by output row."""
    if isinstance(logits, torch.Tensor):
        logits = [logits]
    for t in logits:
        _req(t, torch.float32, "logits")
    ld_in = logits[0].stride(0)
    if any(t.stride(0) != ld_in for t in logits):
        raise NnamError("head: all inputs must share one leading dimension")
    if rows is None:
        rows = logits[0].shape[0]
    targets, nll, pred = _req_score((targets, nll, pred))
    k = len(logits)
    ptrs = (ctypes.c_void_p * k)(*[t.data_ptr() for t in logits])
    wts = None if weights is None else (ctypes.c_float * k)(*[float(w) for w in weights])
    rw = rb = rlb = None
    if rpl is not None:
        rw, rb, rlb = rpl
        for t in (rw, rb, rlb):
            _req(t, torch.float32, "rpl")
    _req(prior, torch.float32, "prior")
    _req(out_row_map, torch.int32, "out_row_map")
    with _Prof("head", rows * (n_classes * 4 * k + 12)):
        check(_native.lib().nnam_head_score(ptrs, wts, k, ld_in, int(bool(pre_normalize)), _ptr(rw), _ptr(rb), _ptr(rlb),
                                            _ptr(prior), float(prior_scale), int(bool(final_normalize)), _ptr(targets),
                                            _ptr(nll), _ptr(pred), rows, n_classes, _ptr(out_row_map), _stream()))
    return nll, pred


def widen_f16_host(src16, row_ref, dst, threads=1, dst_rows=None):
    """HOST op: dst[r] = float(src16[r, :C]) + row_ref[r] for the rows of the compact transfer format (see ``head``).
    src16: (rows, ld16) fp16 host tensor / array, row_ref: (rows,) f32, dst: (rows, C) f32 C-contiguous NumPy array --
    or, with ``dst_rows`` (int64 array of ``len(dst_rows)`` destination row indices), the WHOLE output array, of which
    row dst_rows[r] receives source row r."""
    import numpy as np
    rows, cols = (len(dst_rows) if dst_rows is not None else dst.shape[0]), dst.shape[1]
    if rows == 0:
        return dst
    if dst_rows is not None:
        dst_rows = np.ascontiguousarray(dst_rows, dtype=np.int64)
        if dst_rows.min() < 0 or dst_rows.max() >= dst.shape[0]:
            raise NnamError("widen: destination row outside the output array")
    if src16.shape[0] < rows or row_ref.shape[0] < rows or dst.strides[1] != 4:
        raise NnamError("widen: shape mismatch")
    sp = src16.data_ptr() if isinstance(src16, torch.Tensor) else src16.ctypes.data
    rp = row_ref.data_ptr() if isinstance(row_ref, torch.Tensor) else row_ref.ctypes.data
    ld16 = src16.stride(0) if isinstance(src16, torch.Tensor) else src16.strides[0] // 2
    check(_native.lib().nnam_widen_f16_host(sp, ld16, rp, dst.ctypes.data, dst.strides[0] // 4,
                                            None if dst_rows is None else dst_rows.ctypes.data, rows, cols, int(threads)))
    return dst


def gather_transform(x, row_map, add_shift=None, rescale=None, ivec=None, out_kind=OUT_BF16, ldo=None, out=None):
    """Recurrent-path feature prep: out[r] = transform(x[row_map[r]]) ++ ivec[row_map[r]]."""
    _req(x, torch.float32, "x")
    _req(ivec, torch.float32, "ivec")
    _req(row_map, torch.int32, "row_map")
    if not x.is_contiguous() or (ivec is not None and not ivec.is_contiguous()):
        raise NnamError("gather: x and ivec must be contiguous")
    n_src, dim = x.shape
    ivec_dim = 0 if ivec is None else ivec.shape[1]
    n_rows = row_map.numel()
    if ldo is None:
        ldo = round_up(dim + ivec_dim, 8)
    dt = out_dtype(out_kind)
    if out is None:
        hi = torch.empty((n_rows, ldo), dtype=dt, device=x.device)
        lo = torch.empty((n_rows, ldo), dtype=dt, device=x.device) if out_kind == OUT_BF16_SPLIT else None
    else:
        hi, lo = out
    _req(hi, dt, "out")
    with _Prof("splice", n_rows * ((dim + ivec_dim) * 4 + (dim + ivec_dim) * (2 if out_kind in (OUT_BF16, OUT_F16) else 4))):
        check(_native.lib().nnam_gather_transform(_ptr(x), n_src, dim, _ptr(add_shift), _ptr(rescale), _ptr(ivec),
                                                  ivec_dim, _ptr(row_map), n_rows, _ptr(hi), _ptr(lo), ldo, out_kind,
                                                  _stream()))
    return hi, lo


def rnn_plan(cell, hidden, batch, nsplit):
    """(CTAs per group, max concurrent groups on the current device, SM cycles per stream step, streams per group)
    for a recurrent cell configuration with ``batch`` utterance slots per stream."""
    g, m, c, s = ctypes.c_int(0), ctypes.c_int(0), ctypes.c_int(0), ctypes.c_int(0)
    check(_native.lib().nnam_rnn_plan(cell, hidden, batch, nsplit, ctypes.byref(g), ctypes.byref(m), ctypes.byref(c),
                                      ctypes.byref(s)))
    return g.value, m.value, c.value, s.value


def rnn_solo_step_cycles(cell, hidden, batch, nsplit):
    """SM cycles per step of a stream whose sibling streams in the group are idle (see include/nnam_b200.h)."""
    c = ctypes.c_int(0)
    check(_native.lib().nnam_rnn_solo_step_cycles(cell, hidden, batch, nsplit, ctypes.byref(c)))
    return c.value


def rnn_seq(desc, flops):
    """K3: run one recurrent layer (all batches, one or both directions) described by an RnnDesc."""
    with _Prof("rnn", flops):
        check(_native.lib().nnam_rnn_seq(ctypes.addressof(desc), _stream()))


def peephole_cell(phase, gx, g1, p2, c_prev, c_new, out_hi, out_lo, n, hidden, fast, elem=ELEM_BF16):
    """One phase of the peephole-LSTM gate arithmetic on n packed rows (see include/nnam_b200.h)."""
    _req(out_hi, E16[elem], "out_hi")
    with _Prof("cell", n * hidden * 4 * 8):
        check(_native.lib().nnam_peephole_cell(
            phase, _ptr(gx), gx.stride(0), _ptr(g1), 0 if g1 is None else g1.stride(0), _ptr(p2),
            0 if p2 is None else p2.stride(0), _ptr(c_prev), _ptr(c_new), _ptr(out_hi), _ptr(out_lo), out_hi.stride(0),
            n, hidden, int(bool(fast)), elem, _stream()))
