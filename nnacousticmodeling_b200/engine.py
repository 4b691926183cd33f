"""Device-side planning for the hot path: weight packing, workspaces, the chunked
splice -> GEMM stack -> head pipeline with overlapped D2H, and utterance sharding.

HBM layout (per device)
  raw features      fp32 (rows, dim)            uploaded once per shard, with a +-splice halo
  layer inputs      bf16 (chunk, ld)  [+ lo]    ld = roundup(K, 8); hi/lo pair in 'fp32' (bf16x3) mode
  weights           bf16 (N, roundup(K, 8)) [+ lo], bias fp32 (N)   Chainer (out, in) layout, K-major
  logits            fp32 (chunk, roundup(C, 16))
  log-likelihoods   fp32 (chunk, C)  double-buffered, copied to the (pinned) host array on a side stream
"""
from __future__ import annotations

import os
import time
import threading

import numpy as np
import torch

from . import ops
from ._native import NnamError
from .ops import (ELEM_BF16, ELEM_F16, OUT_BF16, OUT_BF16_SPLIT, OUT_F16, OUT_F32, SPLIT_A, SPLIT_AW, SPLIT_NONE,
                  SPLIT_W, round_up)

DEFAULT_CHUNK = int(os.environ.get("NNAM_CHUNK_ROWS", "65536"))  # frames per feed-forward chunk (tuning aid)


class Precision:
    """Parsed ``model.precision``.

    ``"fp32"``  bf16x3 error-compensated tensor-core GEMMs (<= 1e-3 of the fp32 reference), every operand as a bf16
                hi/lo pair;
    ``"bf16"``  single-pass bf16 operands (8-bit significand);
    ``"fp16"``  single-pass IEEE fp16 operands (11-bit significand, saturating conversions): same tensor-pipe rate as
                bf16 with an 8x smaller rounding error per operand -- the single-pass mode that meets north_star's
                >= 99.5 % frame-argmax agreement on the flat logits of random-init nets (DESIGN.md section 3);
    ``"bf16+a[:layers][+w[:layers]]"``  (MLP only) bf16 with the ACTIVATIONS (``a``) and / or WEIGHTS (``w``) of the
                listed Linear layers carried as hi/lo pairs, i.e. one extra tensor pass each -- the per-layer parity study
                of DESIGN.md.  Layers are numbered 0..L-1 (hidden) and L or -1 (output), separated by ',' or '/';
                no list = every layer.
    """

    def __init__(self, spec):
        parts = str(spec).split("+")
        self.spec, self.base = str(spec), parts[0]
        if self.base not in ("fp32", "bf16", "fp16"):
            raise NnamError(f"precision must be 'fp32', 'bf16', 'fp16' or 'bf16+a[:l,..][+w[:l,..]]' (got {spec!r})")
        self.split = self.base == "fp32"
        self.elem = ELEM_F16 if self.base == "fp16" else ELEM_BF16
        self.tdt = ops.E16[self.elem]
        self.out16 = OUT_F16 if self.base == "fp16" else OUT_BF16
        self.act_kind = OUT_BF16_SPLIT if self.split else self.out16
        self.fast_math = not self.split  # MUFU tanh in the 16-bit modes, tanhf in the fp32-accurate mode
        self._sel = {}
        for part in parts[1:]:
            which, _, arg = part.partition(":")
            if self.base != "bf16" or which not in ("a", "w"):
                raise NnamError(f"precision {spec!r}: per-layer splits are '+a[:layers]' / '+w[:layers]' on 'bf16'")
            self._sel[which] = None if arg in ("", "all") else frozenset(int(t) for t in arg.replace("/", ",").split(","))
        self.per_layer = bool(self._sel)

    def _has(self, which, l, n_linear):
        if which not in self._sel:
            return False
        sel = self._sel[which]
        return sel is None or l in sel or (l - n_linear) in sel

    def a_split(self, l, n_linear):
        """Does Linear layer ``l`` (of ``n_linear``, the last one being the output layer) read split activations?"""
        return self.split or self._has("a", l, n_linear)

    def w_split(self, l, n_linear):
        return self.split or self._has("w", l, n_linear)

    def nsplit(self, l, n_linear):
        a, w = self.a_split(l, n_linear), self.w_split(l, n_linear)
        return SPLIT_AW if (a and w) else (SPLIT_A if a else (SPLIT_W if w else SPLIT_NONE))

    def in_kind(self, l, n_linear):
        """Output kind the PRODUCER of layer ``l``'s input must emit."""
        return OUT_BF16_SPLIT if self.a_split(l, n_linear) else self.out16


def _device(dev):
    if isinstance(dev, torch.device):
        return dev
    if dev is None:
        dev = 0
    if int(dev) < 0:
        raise NnamError("gpu < 0 (CPU) is not supported: nnacousticmodeling_b200 has no CPU path")
    return torch.device("cuda", int(dev))


def empty_pinned(shape, dtype=np.float32):
    """Page-locked host array (NumPy view of a pinned torch tensor) for H2D/D2H at PCIe speed."""
    tdt = {np.dtype(np.float32): torch.float32, np.dtype(np.int32): torch.int32}[np.dtype(dtype)]
    return torch.empty(tuple(shape), dtype=tdt, pin_memory=True).numpy()


def _as_host_tensor(a):
    """NumPy array -> torch CPU tensor sharing memory (pinned-ness is preserved)."""
    if isinstance(a, torch.Tensor):
        return a
    return torch.from_numpy(a)


# ------------------------------------------------------------------------------------------
# packed parameters
# ------------------------------------------------------------------------------------------
class LinearDev:
    """One Linear layer on a device: 16-bit (hi[, bf16 lo]) K-major weights + fp32 bias."""

    def __init__(self, w, b, device, split, elem=ELEM_BF16):
        w = np.ascontiguousarray(w, dtype=np.float32)
        self.n, self.k = w.shape
        kind = OUT_BF16_SPLIT if split else (OUT_F16 if elem == ELEM_F16 else OUT_BF16)
        wd = torch.from_numpy(w).to(device)
        self.w_hi, self.w_lo = ops.convert_f32(wd, kind)
        self.bias = None if b is None else torch.from_numpy(np.ascontiguousarray(b, dtype=np.float32)).to(device)
        self.split, self.elem = split, elem

    def __call__(self, a_hi, a_lo, rows, act, out_kind, out=None, nsplit=None):
        if nsplit is None:
            nsplit = SPLIT_AW if self.split else SPLIT_NONE
        return ops.linear_bias_act(a_hi, a_lo, self.w_hi, self.w_lo, self.bias, rows, self.n, self.k, act=act,
                                   out_kind=out_kind, nsplit=nsplit, out=out, elem=self.elem)


    def logsoftmax(self, a_hi, a_lo, rows, prior=None, prior_scale=1.0, nsplit=None, out=None, out16=None,
                   out_row_map=None, score=None):
        """This layer as the output layer of a single net, fused with the head (ops.linear_logsoftmax); ``score`` =
        (targets, nll, pred) scores the rows instead of writing them."""
        if nsplit is None:
            nsplit = SPLIT_AW if self.split else SPLIT_NONE
        return ops.linear_logsoftmax(a_hi, a_lo, self.w_hi, self.w_lo, self.bias, rows, self.n, self.k, prior=prior,
                                     prior_scale=prior_scale, nsplit=nsplit, elem=self.elem, out=out, out16=out16,
                                     out_row_map=out_row_map, score=score)


FUSED_HEAD_MAX_K = 1024


def fused_head_ok(models, head, k):
    """Run the output layer (fan-in ``k``) and the head as ONE kernel (ops.linear_logsoftmax) when the head is plain -- a
    single net, no RPL, weight 1, final log-softmax, 512..2048 classes -- and the layer is short: up to K = 1024 the fused
    kernel beats the unfused pair by 6-20 % (its epilogue, not its main loop, sets the pace, and the logits round trip it
    saves is a third of the pair's time); at K = 2048 its 15 resident clusters (120 of 148 SMs) cost what the fusion
    saves, and the feed-forward engine hides the unfused head under the next chunk's GEMMs anyway
    (profiles/r02_fused_head.md).  NNAM_FUSED_HEAD=0 switches it off, =force takes every eligible layer."""
    env = os.environ.get("NNAM_FUSED_HEAD", "1")
    if env == "0" or len(models) != 1 or head.rpl is not None or head.pre_normalize or not head.final_normalize:
        return False
    if head.weights is not None and [float(w) for w in head.weights] != [1.0]:
        return False
    n = models[0].n_out
    if models[0].network == "tdnn" or n > ops.FUSED_HEAD_MAX_CLASSES:
        return False
    return env == "force" or (n >= 512 and k <= FUSED_HEAD_MAX_K)


class Workspace:
    """Grow-only named device buffers (the kernels never allocate).

    Debug aid: with ``NNAM_REDZONE=<bytes>`` in the environment every buffer gets that many guard bytes in front and
    behind, filled with 0xA5; :meth:`check_redzones` raises if a kernel wrote into one (tests/test_gpu_redzones.py).
    """

    GUARD_BYTE = 0xA5

    def __init__(self, device):
        self.device = device
        self.buf = {}
        self.redzone = int(os.environ.get("NNAM_REDZONE", "0")) // 256 * 256
        self._raw = {}

    def get(self, name, rows, cols, dtype):
        t = self.buf.get(name)
        need = rows * cols
        if t is None or t.numel() < need or t.dtype != dtype:
            if self.redzone:
                nbytes = need * torch.empty((), dtype=dtype).element_size()
                raw = torch.full((2 * self.redzone + round_up(nbytes, 256),), self.GUARD_BYTE, dtype=torch.uint8,
                                 device=self.device)
                self._raw[name] = (raw, nbytes)
                t = raw[self.redzone:self.redzone + nbytes].view(dtype)
            else:
                t = torch.empty(need, dtype=dtype, device=self.device)
            self.buf[name] = t
        return t[:need].view(rows, cols)

    def check_redzones(self):
        """Raise NnamError naming the first buffer whose guard bytes changed; returns the number of buffers checked."""
        for name, (raw, nbytes) in self._raw.items():
            front = raw[:self.redzone]
            back = raw[self.redzone + nbytes:]
            for where, g in (("before", front), ("after", back)):
                bad = (g != self.GUARD_BYTE).nonzero()
                if bad.numel():
                    raise NnamError(f"workspace buffer '{name}' ({nbytes} bytes): {bad.numel()} guard bytes "
                                    f"{where} it were overwritten, first at offset {int(bad[0])}")
        return len(self._raw)


class Plan:
    """Per (model, device, precision) packed parameters."""

    def __init__(self, model, device):
        self.device = device
        self.prec = prec = Precision(model.precision)
        self.split = prec.split          # every operand is a bf16 hi/lo pair (fp32-accurate mode)
        self.elem, self.tdt = prec.elem, prec.tdt
        self.act_kind = prec.act_kind    # what producers of GEMM operands emit (first-layer input: see in_kind)
        self.in_kind = prec.act_kind
        self.ws = Workspace(device)
        p = model.params
        if prec.per_layer and model.network != "ff":
            raise NnamError(f"precision {prec.spec!r}: per-layer splits are implemented for the MLP ('ff') only")
        with torch.cuda.device(device):
            if model.network == "ff":
                n_lin = model.layers + 1
                self.in_kind = prec.in_kind(0, n_lin)
                self.layers = [LinearDev(p[f"layer_{l}/W"], p[f"layer_{l}/b"], device, prec.w_split(l, n_lin), prec.elem)
                               for l in range(model.layers)]
                self.out = LinearDev(p["out/W"], p["out/b"], device, prec.w_split(model.layers, n_lin), prec.elem)
            elif model.network == "tdnn":
                from . import tdnn_engine
                tdnn_engine.build_plan(self, model)
            else:
                from . import recurrent_engine
                recurrent_engine.build_plan(self, model)
            torch.cuda.current_stream().synchronize()


_plan_lock = threading.Lock()


def get_plan(model, device):
    """Packed parameters of ``model`` on ``device`` (built on first use).  run_sharded() calls this from one host
    thread per device on the same model: creation and the cache update happen under a lock, so no thread can drop
    another device's freshly built plan or iterate the dict while it changes."""
    device = _device(device)
    key = (device.index, model.precision, model._version)
    plan = model._plans.get(key)
    if plan is not None:
        return plan
    with _plan_lock:
        plan = model._plans.get(key)
        if plan is None:
            if not model.params:
                raise NnamError(f"{type(model).__name__} has no parameters: load_npz() or init_params() first")
            plan = Plan(model, device)
            plans = {k: v for k, v in model._plans.items() if k[2] == model._version}
            plans[key] = plan
            model._plans = plans
    return plan


# ------------------------------------------------------------------------------------------
# MLP stack on already-staged bf16 inputs
# ------------------------------------------------------------------------------------------
def mlp_hidden(model, plan, a_hi, a_lo, rows, ws=None):
    """Run the hidden Linear stack; returns the operands (hi, lo) of the output layer."""
    ws = ws or plan.ws
    act = model.activation.name
    cap = a_hi.shape[0]
    prec, n_lin = plan.prec, len(plan.layers) + 1
    for l, lin in enumerate(plan.layers):
        ld = round_up(lin.n, 16)
        kind = prec.in_kind(l + 1, n_lin)  # what the NEXT layer reads
        hi = ws.get(f"act.h{l % 2}.hi", cap, ld, plan.tdt)
        lo = ws.get(f"act.h{l % 2}.lo", cap, ld, torch.bfloat16) if kind == OUT_BF16_SPLIT else None
        lin(a_hi, a_lo, rows, act, kind, out=(hi, lo), nsplit=prec.nsplit(l, n_lin))
        a_hi, a_lo = hi, lo
    return a_hi, a_lo


def mlp_logits(model, plan, a_hi, a_lo, rows, tag="mlp", ws=None):
    """Run the Linear stack; returns fp32 logits (rows, roundup(C, 16)) in workspace memory (``ws``: the
    workspace to use -- ensemble members share the first member's activation buffers)."""
    ws = ws or plan.ws
    cap = a_hi.shape[0]
    n_lin = len(plan.layers) + 1
    a_hi, a_lo = mlp_hidden(model, plan, a_hi, a_lo, rows, ws)
    ldc = round_up(plan.out.n, 16)
    logits = ws.get(f"{tag}.logits", cap, ldc, torch.float32)
    plan.out(a_hi, a_lo, rows, "identity", OUT_F32, out=(logits, None), nsplit=plan.prec.nsplit(n_lin - 1, n_lin))
    return logits


def ff_logits(model, plan, a_hi, a_lo, rows, tag, ws=None):
    """Frame-independent nets on staged inputs: MLP Linear stack or TDNN conv-as-GEMM stack."""
    if model.network == "tdnn":
        from . import tdnn_engine
        return tdnn_engine.logits(model, plan, a_hi, a_lo, rows, tag=tag, ws=ws)
    return mlp_logits(model, plan, a_hi, a_lo, rows, tag=tag, ws=ws)


def call_model(model, x):
    """``model(x)``: (B, D_in) float32 -> (B, C) raw logits.  NumPy in -> NumPy out; CUDA tensor in ->
    CUDA tensor out (mirrors Chainer's xp-array behaviour).  Recurrent models are stateful per call."""
    is_np = not isinstance(x, torch.Tensor)
    if hasattr(x, "data") and not isinstance(x, (np.ndarray, torch.Tensor)):  # chainer.Variable-like
        x = x.data
    if is_np:
        xt = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
        device = _device(model._device)
    else:
        xt = x
        device = x.device if x.is_cuda else _device(model._device)
    plan = get_plan(model, device)
    with torch.cuda.device(device):
        xd = xt.to(device, dtype=torch.float32)
        if xd.dim() != 2 or xd.shape[1] != model.in_size:
            raise NnamError(f"model(x): expected (B, {model.in_size}) input, got {tuple(xd.shape)}")
        if model.recurrent:
            from . import recurrent_engine
            logits = recurrent_engine.step(model, plan, xd)
        else:
            rows = xd.shape[0]
            a_hi, a_lo = ops.convert_f32(xd.contiguous(), plan.in_kind)
            logits = ff_logits(model, plan, a_hi, a_lo, rows, "call")
            logits = logits[:rows, :model.n_out].clone()
        if is_np:
            return logits.cpu().numpy()
        return logits


# ------------------------------------------------------------------------------------------
# sharding (SURVEY 8e): contiguous ranges, no collective
# ------------------------------------------------------------------------------------------
def partition_frames(n_frames, parts):
    """Equal contiguous frame ranges for feed-forward nets (per-frame independent given the halo)."""
    cuts = [(n_frames * i) // parts for i in range(parts + 1)]
    return [(cuts[i], cuts[i + 1]) for i in range(parts)]


def partition_utterances(offsets, parts):
    """Contiguous utterance ranges with ~equal frame counts (prefix-sum cut points on ``offsets``)."""
    offsets = np.asarray(offsets, dtype=np.int64)
    n_utt = len(offsets) - 1
    total = int(offsets[-1])
    cuts = [0]
    for i in range(1, parts):
        target = total * i / parts
        u = int(np.searchsorted(offsets, target, side="left"))
        if u > 0 and abs(offsets[u - 1] - target) <= abs(offsets[min(u, n_utt)] - target):
            u -= 1
        cuts.append(min(max(u, cuts[-1]), n_utt))
    cuts.append(n_utt)
    return [(cuts[i], cuts[i + 1]) for i in range(parts)]


# ------------------------------------------------------------------------------------------
# feed-forward frame pipeline: splice -> GEMMs -> head -> D2H
# ------------------------------------------------------------------------------------------
class HeadSpec:
    """What the head applies after the logits (K4 arguments)."""

    def __init__(self, prior=None, prior_scale=1.0, rpl=None, weights=None, pre_normalize=False,
                 final_normalize=True):
        self.prior, self.prior_scale, self.rpl = prior, prior_scale, rpl
        self.weights, self.pre_normalize, self.final_normalize = weights, pre_normalize, final_normalize


def _dev_vec(a, device):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32).reshape(-1)).to(device)


class RowSink:
    """Consumer of finished output rows for callers that do not want the whole (N, C) matrix in host memory at once
    (the predict_folds CLI streams them into the .npy file).  ``write(r0, r1, rows)`` is called from a helper thread,
    once per chunk, in increasing row order for feed-forward nets; ``rows`` is a NumPy view of a pinned staging buffer
    that is reused after the call returns."""

    def write(self, r0, r1, rows):
        raise NotImplementedError


def upload_targets(ws, name, targets, r0, r1):
    """Rows [r0, r1) of the (N,) int32 host targets as a device vector in workspace memory (4 B per frame, once per
    shard)."""
    t = ws.get(name, r1 - r0, 1, torch.int32).view(-1)
    t.copy_(torch.from_numpy(np.ascontiguousarray(targets[r0:r1], dtype=np.int32)))
    return t


def score_buffers(ws, tag, targets, r0, r1):
    """Device (targets, nll, pred) of rows [r0, r1) for a scoring pass, in workspace memory (NNAM_REDZONE guards
    them)."""
    return (upload_targets(ws, f"{tag}.targets", targets, r0, r1), ws.get(f"{tag}.nll", r1 - r0, 1, torch.float32).view(-1),
            ws.get(f"{tag}.pred", r1 - r0, 1, torch.int32).view(-1))


def download_scores(dev, score, r0, r1):
    """Copy the device (nll, pred) of rows [r0, r1) into the host arrays of ``score`` = (targets, nll, pred)."""
    _, nll_h, pred_h = score
    nll_h[r0:r1] = dev[1].cpu().numpy()
    pred_h[r0:r1] = dev[2].cpu().numpy()


def ff_forward_frames(models, x, ft, splice, out, f0=0, f1=None, ivectors=None, device=0, head=None,
                      chunk=None, presliced=False, sink=None, transfer=None, host_threads=None, score=None):
    """Feed-forward hot loop on ONE device for frames [f0, f1) of the whole array ``x``.

    models    : one MLP or a list (ensemble -> logits combined in the head with head.weights)
    x         : (N, dim) float32 raw features, host array or CUDA tensor (already resident) -- or, with
                presliced=True, the already spliced/transformed (N, D_in) matrix (evaluate.py hands such
                data to the model)
    ivectors  : optional (N, I) host array or CUDA tensor, appended after splice + transform
    out       : (N, C) float32; rows [f0, f1) are written.  Host array (pinned => async D2H overlapped
                with the next chunk on a side stream) or CUDA tensor (results stay in HBM).  May be None when
                ``sink`` (a RowSink) is given: every chunk is then copied into one of two pinned staging buffers and
                handed to ``sink.write`` on a helper thread while the next chunk is computed.
    transfer  : how rows reach the host: "f32" = the float32 rows themselves; "f16" = the compact format of
                nnam_head_f16 (fp16 offsets from the row maximum + the maximum: half the PCIe bytes, widened back to
                float32 by ``host_threads`` host threads); None = "f16" in the 16-bit precision modes, "f32" in the
                fp32-accurate mode (see :func:`use_compact_transfer`).
    score     : (targets, nll, pred) host arrays of shape (N,) -- int32 targets in [-1, C), float32 nll, int32 pred --
                to score rows [f0, f1) against their targets instead of writing them (``out`` and ``sink`` are None
                then): nll[f] = -y[f][targets[f]] (0 for target -1), pred[f] = argmax_c y[f][c], with y the row this
                function would have written to a host ``out``.  The targets go up once, the chunk sizes and kernel
                choices are those of a host ``out``, and 8 B per frame come back at the end.
    """
    if not isinstance(models, (list, tuple)):
        models = [models]
    device = _device(device)
    head = head or HeadSpec()
    n_total = x.shape[0]
    f1 = n_total if f1 is None else f1
    if f1 <= f0:
        return out
    n_out = models[0].n_out
    from .dist_util import halo_range
    lo, hi = halo_range(f0, f1, 0 if presliced else splice, n_total)
    with torch.cuda.device(device):
        plans = [get_plan(m, device) for m in models]
        plan0 = plans[0]
        ws = plan0.ws
        t_pass = time.perf_counter()
        if chunk is None:
            # A GEMM launch over 65,536 frames of a 1024-wide layer lasts ~100 us, of which the prologue, the pipeline fill
            # and the last tile's drain are ~8 %: small single nets take chunks of twice the size (cfg1: 66.7 -> 71.9 M
            # frames/s; no effect on cfg2, whose launches last 300-400 us) -- when the rows stay in HBM: with a host
            # destination the pass is bound by PCIe, and the longer first / last chunk costs more than the launches save.
            small = (len(models) == 1 and isinstance(out, torch.Tensor) and out.is_cuda and models[0].network == "ff"
                     and max((lin.n for lin in plan0.layers), default=0) <= 1024)
            chunk = DEFAULT_CHUNK * 2 if (small and "NNAM_CHUNK_ROWS" not in os.environ) else DEFAULT_CHUNK
        main = torch.cuda.current_stream()
        side = plan0.__dict__.setdefault("_side_stream", torch.cuda.Stream(device=device))
        # Host inputs are uploaded chunk by chunk on their own stream (`up`): the GEMMs of chunk 0 start after ~1/18 of
        # the upload instead of all of it, and later uploads overlap the D2H copies (the two directions are full duplex).
        up = plan0.__dict__.setdefault("_up_stream", torch.cuda.Stream(device=device))
        x_host = iv_host = None
        if isinstance(x, torch.Tensor) and x.is_cuda:
            x_dev, lo = x, 0
        else:
            x_dev = ws.get("ff.x", hi - lo, x.shape[1], torch.float32)
            x_host = _as_host_tensor(x)
        iv_dev, iv0 = None, f0
        if ivectors is not None:
            if isinstance(ivectors, torch.Tensor) and ivectors.is_cuda:
                iv_dev, iv0 = ivectors, 0
            else:
                iv_dev = ws.get("ff.iv", f1 - f0, ivectors.shape[1], torch.float32)
                iv_host = _as_host_tensor(ivectors)
        up.wait_stream(main)  # the buffers may still be read by a previous pass
        uploaded = []         # per chunk: event after which its raw rows (+ halo) and i-vector rows are resident
        if x_host is not None or iv_host is not None:
            x_done = lo  # global raw rows [lo, x_done) have been queued
            step = min(chunk, f1 - f0)
            with torch.cuda.stream(up):
                for c0 in range(f0, f1, step):
                    c1 = min(c0 + step, f1)
                    if x_host is not None:
                        need = min(c1 + halo_of(presliced, splice), hi)
                        if need > x_done:
                            x_dev[x_done - lo:need - lo].copy_(x_host[x_done:need], non_blocking=True)
                            x_done = need
                    if iv_host is not None:
                        iv_dev[c0 - f0:c1 - f0].copy_(iv_host[c0:c1], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(up)
                    uploaded.append(ev)
        add = mul = None
        if ft is not None and not presliced:
            add, mul = _dev_vec(ft["addShift"], device), _dev_vec(ft["rescale"], device)
        prior = _dev_vec(head.prior, device)
        rpl = None if head.rpl is None else tuple(_dev_vec(head.rpl[k], device) for k in ("W", "b", "lb"))
        fused = fused_head_ok(models, head, plan0.out.k if hasattr(plan0, "out") else 0)
        n_lin = len(getattr(plan0, "layers", ())) + 1
        out_on_device = isinstance(out, torch.Tensor) and out.is_cuda
        out_h = None if (out_on_device or out is None) else _as_host_tensor(out)
        if score is not None and (out is not None or sink is not None):
            raise NnamError("ff_forward_frames: a scoring pass writes no rows (out and sink must be None)")
        if out is None and sink is None and score is None:
            raise NnamError("ff_forward_frames: give an output array or a RowSink")
        chunk = min(chunk, f1 - f0)
        d_in = models[0].in_size
        if any(m.in_size != d_in or m.n_out != n_out for m in models):
            raise NnamError("ensemble members must share input and output sizes")
        have = x.shape[1] if presliced else (2 * splice + 1) * x.shape[1] + (0 if ivectors is None else ivectors.shape[1])
        if have != d_in:
            raise NnamError(f"model expects {d_in} inputs per frame, the data provides {have}")
        ld_in = round_up(d_in, 8)
        if any(p.prec.spec != plan0.prec.spec for p in plans):
            raise NnamError("ensemble members must use the same precision mode")
        a_bufs = [(ws.get("ff.a.hi", chunk, ld_in, plan0.tdt),
                   ws.get("ff.a.lo", chunk, ld_in, torch.bfloat16) if plan0.in_kind == OUT_BF16_SPLIT else None)]
        out_dev = None if (out_on_device or score is not None) else [ws.get(f"ff.out{i}", chunk, n_out, torch.float32)
                                                                      for i in range(2)]
        sc_dev = None if score is None else score_buffers(ws, "ff", score[0], f0, f1)
        # Host output.  "direct" = D2H straight into the caller's array; otherwise a chunk goes through one of two pinned
        # staging buffers and a helper thread finishes it (widen the compact format and / or feed the sink).  With the
        # compact format and a PINNED destination the chunks are MIXED: PCIe and the widening threads are two servers,
        # compact chunks load both (half the PCIe bytes + host work), float32 chunks only PCIe, so a fraction x of the
        # chunks goes compact such that both finish together (see _TransferStats).
        host_threads = host_threads or default_host_threads()
        mixable = (not out_on_device) and sink is None and out_h is not None and out_h.is_pinned()
        compact = (not out_on_device and score is None) and use_compact_transfer(plan0, transfer, host_threads=host_threads,
                                                                                  mixable=mixable)
        writer = o16_dev = ref_dev = stats = None
        frac_compact = 1.0
        if (compact or sink is not None) and not out_on_device:
            ld16 = round_up(n_out, 8)
            # Compact chunks cross PCIe in PIECES of a few thousand rows through a small ring of pinned buffers (4 x 16 MB
            # for 1909 classes): the widening threads then read a piece while it is still in the last-level cache (the
            # DMA wrote it there or it was just brought in), instead of streaming a 250 MB chunk back from DRAM -- the
            # widening is bound by the host's memory system, and this takes a third of its traffic away.
            piece = max(256, min(chunk, int(os.environ.get("NNAM_PIECE_ROWS", "4096")))) if compact else chunk
            slots = max(2, int(os.environ.get("NNAM_PIECE_SLOTS", "4")))
            key = ("f16" if compact else "f32", piece, n_out, slots)
            cache = plan0.__dict__.setdefault("_stage", {})
            if key not in cache:
                cache.clear()
                if compact:
                    cache[key] = [(torch.empty((piece, ld16), dtype=torch.float16, pin_memory=True),
                                   torch.empty((piece,), dtype=torch.float32, pin_memory=True)) for _ in range(slots)]
                else:
                    cache[key] = [(torch.empty((chunk, n_out), dtype=torch.float32, pin_memory=True), None) for _ in range(2)]
            stage = cache[key]
            if compact:
                o16_dev = [ws.get(f"ff.out16.{i}", chunk, ld16, torch.float16) for i in range(2)]
                ref_dev = [ws.get(f"ff.ref.{i}", chunk, 1, torch.float32).view(-1) for i in range(2)]
                if mixable and (transfer or os.environ.get("NNAM_TRANSFER")) is None:
                    stats = plan0.__dict__.setdefault("_xfer_stats", _TransferStats(host_threads))
                    frac_compact = stats.compact_fraction()
            out_np = out.numpy() if isinstance(out, torch.Tensor) else out
            writer = _ChunkWriter(stage, compact, out_np, sink, n_out, host_threads)
        # Three streams: `main` runs splice + the GEMM stack of chunk i; `aux` runs the HBM-bound head of chunk i-1 in
        # their shadow (the GEMM kernels cap their registers so that one head CTA fits next to a GEMM CTA on every SM);
        # `side` carries the D2H copies.  Logits and head outputs are double-buffered by chunk parity.  (Moving the
        # splice kernel to `aux` as well was measured and dropped: it needs shared memory, cannot co-reside with a
        # GEMM CTA and only delayed the head.)
        aux = plan0.__dict__.setdefault("_aux_stream", torch.cuda.Stream(device=device))
        aux.wait_stream(main)
        a_hi, a_lo = a_bufs[0]
        copied_f, copied_c = [None, None], [None, None]  # D2H of the chunk that last used out_dev[i] / o16_dev[i]
        n_f = n_c = 0
        copies = []                # (start, end, bytes) of every D2H copy, for the transfer statistics
        head_done = [None, None]   # head of the chunk that last used the logits buffers of this parity
        pending = None
        ring = [0]

        def drain(as_compact, via_writer, ob, c0, c1, hd):
            """Queue the device->host copies of a finished chunk (rows [c0, c1)) and hand them to the helper thread."""
            rows = c1 - c0
            side.wait_event(hd)
            ev = None
            if as_compact:
                for p0 in range(0, rows, piece):
                    p1 = min(p0 + piece, rows)
                    slot = ring[0] % len(stage)
                    ring[0] += 1
                    writer.wait_free(slot)  # the helper thread still widens the piece that used this slot
                    with torch.cuda.stream(side):
                        t0 = torch.cuda.Event(enable_timing=True) if stats is not None else None
                        if t0 is not None:
                            t0.record(side)
                        stage[slot][0][:p1 - p0].copy_(o16_dev[ob][p0:p1], non_blocking=True)
                        stage[slot][1][:p1 - p0].copy_(ref_dev[ob][p0:p1], non_blocking=True)
                        ev = torch.cuda.Event(enable_timing=stats is not None)
                        ev.record(side)
                        if stats is not None:
                            copies.append((t0, ev, (p1 - p0) * (o16_dev[ob].stride(0) * 2 + 4)))
                    writer.submit(slot, c0 + p0, c0 + p1, ev)
                copied_c[ob] = ev
                return
            if via_writer:
                writer.wait_free(ob)  # the helper thread still reads the staging buffer of the chunk two before
            with torch.cuda.stream(side):
                t0 = torch.cuda.Event(enable_timing=True) if stats is not None else None
                if t0 is not None:
                    t0.record(side)
                dst = stage[ob][0][:rows] if via_writer else out_h[c0:c1]
                dst.copy_(out_dev[ob][:rows], non_blocking=True)
                ev = torch.cuda.Event(enable_timing=stats is not None)
                ev.record(side)
                if stats is not None:
                    copies.append((t0, ev, rows * n_out * 4))
            copied_f[ob] = ev
            if via_writer:
                writer.submit(ob, c0, c1, ev)

        for ci, c0 in enumerate(range(f0, f1, chunk)):
            c1 = min(c0 + chunk, f1)
            rows = c1 - c0
            buf = ci % 2
            if uploaded:
                main.wait_event(uploaded[ci])
            if presliced:
                ops.convert_f32(x_dev[c0 - lo:c1 - lo], plan0.in_kind, ldd=ld_in, out=(a_hi, a_lo))
            else:
                ops.splice_transform(x_dev, n_total, splice, add, mul,
                                     None if iv_dev is None else iv_dev[c0 - iv0:c1 - iv0], f0=c0, f1=c1, x_row0=lo,
                                     out_kind=plan0.in_kind, ldo=ld_in, out=(a_hi, a_lo))
            # this chunk's transfer format (error diffusion of the compact fraction over the chunk index)
            as_compact = compact and int((ci + 1) * frac_compact + 1e-9) > int(ci * frac_compact + 1e-9)
            via_writer = writer is not None and (as_compact or not compact)
            if as_compact:
                ob, n_c = n_c % 2, n_c + 1   # ring position among the compact chunks / the staging buffers
            else:
                ob, n_f = n_f % 2, n_f + 1   # ring position among the float32 chunks
            last = copied_c if as_compact else copied_f
            if fused:
                # output layer + head as ONE kernel on the main stream (no logits buffer, nothing for `aux` to do)
                h_hi, h_lo = mlp_hidden(models[0], plan0, a_hi, a_lo, rows, ws)
                okw = dict(prior=prior, prior_scale=head.prior_scale, nsplit=plan0.prec.nsplit(n_lin - 1, n_lin))
                if out_on_device:
                    plan0.out.logsoftmax(h_hi, h_lo, rows, out=out[c0:c1], **okw)
                elif sc_dev is not None:
                    plan0.out.logsoftmax(h_hi, h_lo, rows, score=tuple(t[c0 - f0:c1 - f0] for t in sc_dev), **okw)
                else:
                    if last[ob] is not None:
                        main.wait_event(last[ob])  # the side stream still reads this buffer
                    if as_compact:
                        plan0.out.logsoftmax(h_hi, h_lo, rows, out16=(o16_dev[ob], ref_dev[ob]), **okw)
                    else:
                        plan0.out.logsoftmax(h_hi, h_lo, rows, out=out_dev[ob], **okw)
                hd = torch.cuda.Event()
                hd.record(main)
            else:
                if head_done[buf] is not None:
                    main.wait_event(head_done[buf])  # the head of chunk i-2 still reads these logits
                logits = [ff_logits(m, p, a_hi, a_lo, rows, f"ff{k}.{buf}", ws) for k, (m, p) in enumerate(zip(models, plans))]
                gemm_done = torch.cuda.Event()
                gemm_done.record(main)
                hkw = dict(rows=rows, weights=head.weights, pre_normalize=head.pre_normalize, rpl=rpl, prior=prior,
                           prior_scale=head.prior_scale, final_normalize=head.final_normalize)
                aux.wait_event(gemm_done)
                with torch.cuda.stream(aux):
                    if out_on_device:
                        ops.head(logits, n_out, out=out[c0:c1], **hkw)
                    elif sc_dev is not None:
                        ops.head_score(logits, n_out, *(t[c0 - f0:c1 - f0] for t in sc_dev), **hkw)
                    else:
                        if last[ob] is not None:
                            aux.wait_event(last[ob])  # the side stream still reads this buffer
                        if as_compact:
                            ops.head(logits, n_out, out16=(o16_dev[ob], ref_dev[ob]), **hkw)
                        else:
                            ops.head(logits, n_out, out=out_dev[ob], **hkw)
                    hd = torch.cuda.Event()
                    hd.record(aux)
            head_done[buf] = hd
            if out_on_device or sc_dev is not None:
                continue
            # the copies of chunk i are queued one iteration later, after chunk i+1's kernels: queueing them may block on
            # the helper thread (ring slots), and the GPU should have its next chunk by then
            if pending is not None:
                drain(*pending)
            pending = (as_compact, via_writer, ob, c0, c1, hd)
        if pending is not None:
            drain(*pending)
        main.wait_stream(aux)  # callers that time or consume on the current stream see the whole pass
        if sc_dev is not None:
            download_scores(sc_dev, score, f0, f1)
        side.synchronize()
        main.synchronize()
        if writer is not None:
            writer.close()
        if stats is not None:
            stats.update(copies, writer, f1 - f0, time.perf_counter() - t_pass)
    return out


class _TransferStats:
    """What the two servers of the host-bound output path sustain in THIS process, measured on the passes so far: PCIe
    (bytes / duration of the D2H copies, CUDA events) and the widening threads (float32 bytes written / time spent
    in nnam_widen_f16_host).  A compact chunk costs 3,828 B/frame of PCIe plus 7,636 B/frame of widening, a float32
    chunk 7,636 B/frame of PCIe; both servers finish together when the compact fraction is
        x = 1 / (P / W + 0.5)      (P, W in bytes/s; x >= 1 means: everything compact)
    e.g. P = 57, W = 70 GB/s (one GPU, 16 threads) -> x = 0.76; under contention (8 ranks sharing the host's 92 GB/s of
    ingest and 32 cores) both P and W shrink and x follows.  Before the first measurement: P = 55 GB/s, W = 4.4 GB/s per
    thread (what one GPU on this pod shows)."""

    def __init__(self, threads):
        self.pcie, self.widen, self.last_d2h_bytes = 55e9, 4.4e9 * threads, None
        # The two servers are not independent -- the widening threads and the DMA compete for the same DRAM (2 ranks x 12
        # threads pushed a rank's PCIe rate from 54 to 20 GB/s), float32 and compact chunks alternate on one copy stream,
        # and whether the piece ring stays in the last-level cache depends on the box -- so the model's x is only the
        # first guess.  The first passes PROBE: the model's x from the prior rates, 0 (float32 rows only), the model's x
        # from the rates measured meanwhile (or half the first guess if that says the same), the first one again (its
        # first pass was a cold one); afterwards the fraction with the best measured frames/s is kept and its measurement
        # refreshed.  NNAM_TRANSFER_PROBE=0 keeps the model's value.
        self.probe = os.environ.get("NNAM_TRANSFER_PROBE", "1") != "0"
        self.tried = {}      # fraction -> frames/s of whole passes
        self.current = None  # fraction of the pass in flight
        self.cold = True     # the first candidate has only been measured on the first (cold) pass

    def model_fraction(self):
        x = 1.0 / (self.pcie / max(self.widen, 1e6) + 0.5)
        return 1.0 if x > 0.97 else max(x, 0.0)

    def compact_fraction(self):
        x = self.model_fraction()
        if self.probe:
            x = round(x, 2)
            if len(self.tried) == 0:
                self.first = x        # from the prior rates
            elif 0.0 not in self.tried:
                x = 0.0               # float32 rows only
            elif len(self.tried) == 2:
                # the model again, now from the rates measured under this box's contention -- or half the first guess
                # if that says the same
                x = 1.0 if x >= 0.85 else x  # nearly everything compact: take all of it (no alternation of formats)
                x = x if abs(x - self.first) > 0.1 else round(self.first / 2, 2)
            elif self.cold:
                x = self.first        # its first measurement included the one-time allocations of a first pass
            else:
                x = max(self.tried, key=self.tried.get)
        self.current = x
        return x

    def update(self, copies, writer, frames=0, seconds=0.0):
        ms = sum(a.elapsed_time(b) for a, b, _ in copies)
        nbytes = sum(n for _, _, n in copies)
        self.last_d2h_bytes = nbytes
        if ms > 1.0 and nbytes > (64 << 20):  # passes too small to measure keep the previous estimate
            self.pcie = 0.5 * self.pcie + 0.5 * nbytes / (ms * 1e-3)
        if writer is not None and writer.widen_s > 1e-3 and writer.widen_bytes > (64 << 20):
            self.widen = 0.5 * self.widen + 0.5 * writer.widen_bytes / writer.widen_s
        if self.probe and self.current is not None and frames >= 100000 and seconds > 0:
            rate = frames / seconds
            old = self.tried.get(self.current)
            if self.cold and old is not None and self.current == self.first:
                old, self.cold = None, False
            self.tried[self.current] = rate if old is None else 0.5 * old + 0.5 * rate


MIN_WIDEN_THREADS = 12  # host threads a process needs before the compact transfer beats the plain float32 copy


def use_compact_transfer(plan, transfer=None, recurrent=False, host_threads=None, mixable=False):
    """Does a host-bound pass of ``plan`` use the compact (fp16 offsets + row maximum) transfer format?  Explicit
    ``transfer`` ("f16" / "f32") wins, then the environment (NNAM_TRANSFER), then the precision mode and the host: the
    16-bit modes (tolerance 5e-2) take it, the fp32-accurate mode (tolerance 1e-3) keeps float32 rows.  Feed-forward
    path: chunks stream, the host widens chunk i while chunk i+1 crosses PCIe (+22 % to +80 % end to end on cfg2).
    Recurrent path: rows only exist after the last layer of a subset of utterances; each subset is packed into one
    contiguous block, crosses PCIe in pieces and is scattered to its frames by the widening threads (cfg3 8.1 M vs 6.3 M,
    cfg4 6.5 M vs 5.5 M, cfg3t 9.8 M vs 6.5 M frames/s where the piece ring stays in the last-level cache; a tie
    -- +4 % / -1 % / +13 % -- on a box where it does not).  The widening needs host cores: with the 4 threads a rank gets
    when 8 processes share a 32-core box it is the bottleneck (10.4 M against 11.9 M frames/s on 8 GPUs, where plain
    copies already run at 98 % of the box's 92.6 GB/s D2H ceiling), so ALL-compact is only chosen when the process has
    at least MIN_WIDEN_THREADS.  With a pinned destination (``mixable``) the feed-forward path instead sends a measured
    FRACTION of the chunks compact and the rest as float32 rows, which helps with any number of threads
    (_TransferStats; profiles/r02_transfer.md)."""
    threads = host_threads or default_host_threads()
    auto = "f32" if (plan.split or (threads < MIN_WIDEN_THREADS and not (mixable and not recurrent))) else "f16"
    mode = transfer or os.environ.get("NNAM_TRANSFER") or auto
    if mode not in ("f16", "f32"):
        raise NnamError(f"transfer must be 'f16' or 'f32' (got {mode!r})")
    return mode == "f16"


def default_host_threads():
    """Host threads for widening the compact format: the process's share of the CPUs it may run on (torchrun starts
    one process per GPU), at most 16."""
    try:
        cpus = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        cpus = os.cpu_count() or 1
    share = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
    return int(os.environ.get("NNAM_HOST_THREADS", max(1, min(16, cpus // share))))


class _ChunkWriter:
    """Helper thread that finishes chunks in submission order once their D2H copy into a pinned staging buffer has
    completed: widens the compact format into the caller's array (or a scratch block) and / or hands the float32 rows
    to a RowSink."""

    def __init__(self, stage, compact, out, sink, n_out, threads):
        import queue
        self.stage, self.compact, self.out, self.sink, self.n_out, self.threads = stage, compact, out, sink, n_out, threads
        self.scratch = None
        self.widen_s, self.widen_bytes = 0.0, 0
        self.free = [threading.Event() for _ in stage]
        for e in self.free:
            e.set()
        self.q = queue.Queue()
        self.err = None
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _finish(self, buf, r0, r1):
        data, ref = self.stage[buf]
        if isinstance(r1, np.ndarray):  # scattered piece: r1 holds the destination row of every source row
            import time
            t0 = time.perf_counter()
            ops.widen_f16_host(data, ref, self.out, self.threads, dst_rows=r1)
            self.widen_s += time.perf_counter() - t0
            self.widen_bytes += len(r1) * self.n_out * 4
            return
        rows = r1 - r0
        if not self.compact:
            self.sink.write(r0, r1, data[:rows].numpy())
            return
        if self.out is not None:
            dst = self.out[r0:r1]
        else:
            if self.scratch is None or self.scratch.shape[0] < rows:
                self.scratch = np.empty((rows, self.n_out), dtype=np.float32)
            dst = self.scratch[:rows]
        import time
        t0 = time.perf_counter()
        ops.widen_f16_host(data, ref, dst, self.threads)
        self.widen_s += time.perf_counter() - t0
        self.widen_bytes += dst.size * 4
        if self.sink is not None:
            self.sink.write(r0, r1, dst)

    def _run(self):
        while True:
            item = self.q.get()
            if item is None:
                return
            buf, r0, r1, ev = item
            try:
                if self.err is None:
                    ev.synchronize()
                    self._finish(buf, r0, r1)
            except BaseException as e:  # noqa: BLE001  (re-raised on the caller's thread by close())
                self.err = e
            finally:
                self.free[buf].set()

    def wait_free(self, buf):
        self.free[buf].wait()
        self.free[buf].clear()

    def submit(self, buf, r0, r1, ev):
        self.q.put((buf, r0, r1, ev))

    def close(self):
        self.q.put(None)
        self.thread.join()
        if self.err is not None:
            raise self.err


def halo_of(presliced, splice):
    """Raw frames a chunk needs beyond its own range on each side."""
    return 0 if presliced else splice


def run_sharded(fn, shards, devices):
    """Run ``fn(shard, device)`` for every (shard, device) pair, one host thread per device."""
    if len(devices) == 1:
        return [fn(shards[0], devices[0])]
    res, errs = [None] * len(devices), []

    def work(i):
        try:
            res[i] = fn(shards[i], devices[i])
        except BaseException as e:  # noqa: BLE001
            errs.append(e)

    th = [threading.Thread(target=work, args=(i,)) for i in range(len(devices))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    if errs:
        raise errs[0]
    return res
