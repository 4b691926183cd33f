"""Parity of the CUDA kernels (through the C ABI) against the oracle / golden vectors.  -m gpu."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import nnam_oracle as O  # noqa: E402


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ops():
    from nnacousticmodeling_b200 import ops as _ops
    return _ops


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _bf16(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.bfloat16).to(torch.float32).numpy()


# ----------------------------------------------------------------------------------------- K1
def test_splice_golden_bit_exact(ops, dev, golden_dir):
    g = np.load(os.path.join(golden_dir, "splice.npz"))
    ft = O.load_kaldi_feature_transform(os.path.join(golden_dir, "final.feature_transform"))
    x = _t(g["x"], dev)
    add, mul = _t(ft["addShift"], dev), _t(ft["rescale"], dev)
    assert np.array_equal(ops.splice_transform(x, len(x), 5)[0].cpu().numpy(), g["splice11"])
    assert np.array_equal(ops.splice_transform(x, len(x), 5, add, mul)[0].cpu().numpy(), g["splice11_ft"])
    xs = _t(g["x_small"], dev)  # 3 frames: both clamps active in one window
    assert np.array_equal(ops.splice_transform(xs, 3, 5)[0].cpu().numpy(), g["splice11_small"])
    assert np.array_equal(ops.splice_transform(x[:64].contiguous(), 64, 8)[0].cpu().numpy(), g["splice17"])
    assert np.array_equal(ops.splice_transform(x[:8].contiguous(), 8, 0)[0].cpu().numpy(), g["splice1"])


def test_splice_recurrent_middle_block(ops, dev, golden_dir):
    g = np.load(os.path.join(golden_dir, "timedelay.npz"))
    ft = O.select_transform_for_network(
        O.load_kaldi_feature_transform(os.path.join(golden_dir, "final.feature_transform")), "lstm")
    out, _ = ops.splice_transform(_t(g["x"], dev), len(g["x"]), 0, _t(ft["addShift"], dev), _t(ft["rescale"], dev))
    assert np.array_equal(out.cpu().numpy(), g["x_mid_ft"])


@pytest.mark.parametrize("n,dim,splice,ivd", [(1000, 40, 5, 100), (333, 40, 5, 0), (70, 13, 3, 5), (129, 40, 0, 100),
                                              (1, 40, 5, 0), (5000, 40, 5, 100)])
def test_splice_ivectors_shards_and_odd_dims(ops, dev, n, dim, splice, ivd):
    rng = np.random.default_rng(n + dim)
    x = rng.standard_normal((n, dim)).astype(np.float32)
    iv = rng.standard_normal((n, ivd)).astype(np.float32) if ivd else None
    w = 2 * splice + 1
    ft = {"addShift": rng.standard_normal(w * dim).astype(np.float32),
          "rescale": (1 + 0.1 * rng.standard_normal(w * dim)).astype(np.float32)}
    want = O.apply_kaldi_feature_transform(O.splicing(x, range(-splice, splice + 1)), ft)
    if iv is not None:
        want = np.concatenate((want, iv), axis=1)
    add, mul = _t(ft["addShift"], dev), _t(ft["rescale"], dev)
    got = ops.splice_transform(_t(x, dev), n, splice, add, mul, None if iv is None else _t(iv, dev))[0]
    assert np.array_equal(got.cpu().numpy(), want)
    # shards: rows [f0, f1) from a buffer that only holds the halo'd slice, must equal the 1-shot output
    for parts in (2, 3):
        pieces = []
        for i in range(parts):
            f0, f1 = n * i // parts, n * (i + 1) // parts
            if f1 == f0:
                continue
            lo, hi = max(f0 - splice, 0), min(f1 + splice, n)
            o = ops.splice_transform(_t(x[lo:hi], dev), n, splice, add, mul,
                                     None if iv is None else _t(iv[f0:f1], dev), f0=f0, f1=f1, x_row0=lo)[0]
            pieces.append(o.cpu().numpy())
        assert np.array_equal(np.concatenate(pieces), want)
    # bf16 and bf16 hi/lo outputs: hi == bf16(fp32 value), hi + lo ~ fp32 value to 2^-16
    hi, lo = ops.splice_transform(_t(x, dev), n, splice, add, mul, None if iv is None else _t(iv, dev),
                                  out_kind=ops.OUT_BF16_SPLIT)
    cols = want.shape[1]
    assert np.array_equal(hi.float().cpu().numpy()[:, :cols], _bf16(want))
    assert np.all(hi.float().cpu().numpy()[:, cols:] == 0)
    rec = (hi.float() + lo.float()).cpu().numpy()[:, :cols]
    assert np.abs(rec - want).max() <= 2.0 ** -15 * max(1.0, np.abs(want).max())


def test_splice_rejects_bad_arguments(ops, dev):
    from nnacousticmodeling_b200 import NnamError
    x = torch.zeros(10, 40, device=dev)
    with pytest.raises(NnamError):
        ops.splice_transform(x, 100, 5, f0=50, f1=60, x_row0=0)  # buffer does not cover the halo
    with pytest.raises(NnamError):
        ops.splice_transform(torch.zeros(10, 40), 10, 5)  # host tensor: no CPU path
    assert ops.splice_transform(x, 10, 5, f0=4, f1=4)[0].shape[0] == 0  # empty range is a no-op


# ----------------------------------------------------------------------------------------- K4
def test_head_golden(ops, dev, golden_dir):
    h = np.load(os.path.join(golden_dir, "head.npz"))
    ap = np.load(os.path.join(golden_dir, "log_ap_Kaldi1909.npy"))
    y = _t(h["y"], dev)
    assert np.abs(ops.head(y, 1909).cpu().numpy() - h["logsoftmax"]).max() < 1e-4
    got = ops.head(y, 1909, prior=_t(ap.reshape(-1), dev)).cpu().numpy()
    assert np.abs(got - h["head_ap"]).max() < 1e-4
    got = ops.head(y, 1909, prior=_t(ap.reshape(-1), dev), prior_scale=0.5).cpu().numpy()
    assert np.abs(got - O.head(h["y"], np.float32(0.5) * ap)).max() < 1e-4


@pytest.mark.parametrize("c,rows,ld", [(39, 77, 48), (1909, 300, 1920), (1000, 17, 1000), (2048, 9, 2048), (7, 1, 7)])
def test_head_ensembles_rpl_and_shapes(ops, dev, c, rows, ld):
    rng = np.random.default_rng(c)
    ys = [(2 * rng.standard_normal((rows, c))).astype(np.float32) for _ in range(3)]

    def dv(a):
        buf = torch.zeros(rows, ld, device=dev)
        buf[:, :c] = _t(a, dev)
        return buf

    yd = [dv(a) for a in ys]
    assert np.abs(ops.head(yd[0], c).cpu().numpy() - O.log_softmax(ys[0])).max() < 1e-4
    # evaluate.py:35-51 master + folds: (K*master + sum folds) / (2K), then log-softmax
    k = 2
    want = O.log_softmax(O.nn_with_rpl(lambda v: ys[0], [lambda v: ys[1], lambda v: ys[2]], None, None))
    got = ops.head(yd, c, weights=[k / (2 * k), 1 / (2 * k), 1 / (2 * k)]).cpu().numpy()
    assert np.abs(got - want).max() < 1e-4
    # predict_folds dev mode: mean of log-softmax outputs, renormalised
    want = O.log_softmax((O.log_softmax(ys[0]) + O.log_softmax(ys[1]) + O.log_softmax(ys[2])) / np.float32(3))
    got = ops.head(yd, c, pre_normalize=True).cpu().numpy()
    assert np.abs(got - want).max() < 1e-4
    # RPL4 then prior then log-softmax
    prm = {"W": (0.1 * rng.standard_normal((1, c))).astype(np.float32),
           "b": (0.1 * rng.standard_normal((1, c))).astype(np.float32), "lb": np.full((1, c), -6.0, np.float32)}
    ap = (-3 + rng.standard_normal((1, c))).astype(np.float32)
    want = O.head(O.rpl4(prm, ys[1]), ap)
    got = ops.head(yd[1], c, rpl=tuple(_t(prm[n].reshape(-1), dev) for n in ("W", "b", "lb")),
                   prior=_t(ap.reshape(-1), dev)).cpu().numpy()
    assert np.abs(got - want).max() < 1e-4
    # raw (un-normalised) ensemble mean
    got = ops.head(yd[:2], c, final_normalize=False).cpu().numpy()
    assert np.abs(got - (ys[0] + ys[1]) / 2).max() < 1e-5


def test_head_compact_transfer_format(ops, dev):
    """nnam_head_f16 + nnam_widen_f16_host: out = fp16(y - rowmax) + rowmax.  Entries near the row maximum keep float32-like
    resolution (argmax unchanged), the tail keeps 11 bits of its distance from the maximum; scatter map and zero rows
    (quirk Q4) included; single-input fast kernel and the generic ensemble kernel."""
    rng = np.random.default_rng(11)
    rows, c = 1500, 1909
    ys = [(3.0 * rng.standard_normal((rows, c))).astype(np.float32) for _ in range(2)]
    yd = []
    for a in ys:
        buf = torch.zeros(rows, 1920, device=dev)
        buf[:, :c] = _t(a, dev)
        yd.append(buf)
    ap = (-3 + rng.standard_normal(c)).astype(np.float32)
    rmap = rng.permutation(rows).astype(np.int32)
    lost = int(rmap[77])  # no logits row maps to this output row any more: it keeps whatever the buffer held
    rmap[5], rmap[77] = -1, -2 - int(rmap[5])  # row 5 dropped, row 77 zero-fills the output row row 5 would have had
    for logits, want in ((yd[0], O.head(ys[0], ap[None, :])),
                         (yd, O.head((ys[0] + ys[1]) / np.float32(2), ap[None, :]))):
        o16 = torch.full((rows, 1912), 9.0, dtype=torch.float16, device=dev)
        ref = torch.full((rows,), 9.0, device=dev)
        ops.head(logits, c, prior=_t(ap, dev), out16=(o16, ref), out_row_map=_t(rmap, dev))
        got = np.empty((rows, c), np.float32)
        ops.widen_f16_host(o16.cpu(), ref.cpu(), got, threads=3)
        exp = np.zeros_like(got)
        for r in range(rows):
            if rmap[r] >= 0:
                exp[rmap[r]] = want[r]
        keep = np.ones(rows, bool)
        keep[-2 - rmap[77]] = keep[lost] = False
        assert np.all(got[-2 - rmap[77]] == 0) and np.all(got[lost] == 18.0)  # fp16(9) + 9: untouched
        dist = exp[keep].max(axis=1, keepdims=True) - exp[keep]
        assert np.all(np.abs(got[keep] - exp[keep]) <= 2.0 ** -11 * dist + 1e-4)  # 1e-4: the head's own fp32 error
        assert np.array_equal(got[keep].argmax(axis=1), exp[keep].argmax(axis=1))
        top = np.take_along_axis(got[keep] - exp[keep], exp[keep].argmax(axis=1)[:, None], axis=1)
        assert np.abs(top).max() < 1e-4  # the best class keeps float32 resolution (no fp16 rounding at distance 0)


# ----------------------------------------------------------------------------------------- K2
@pytest.mark.parametrize("m,n,k,elem,nsplit", [(1000, 1909, 512, "f16", 1), (4173, 1909, 1024, "f16", 1), (300, 39, 136, "bf16", 1),
                                                (777, 600, 72, "bf16", 1), (129, 2048, 2048, "f16", 1), (1500, 1909, 440, "bf16", 3),
                                                (20000, 1909, 512, "f16", 1)])
def test_linear_logsoftmax_fused(ops, dev, m, n, k, elem, nsplit):
    """nnam_linear_logsoftmax (output layer + head in one kernel, row statistics exchanged across a thread-block cluster)
    against the unfused pair nnam_linear_bias_act -> nnam_head / nnam_head_f16 on the same operands, and against the
    float64 result: plain rows, scatter map with dropped and zero-filled rows, prior, compact format."""
    rng = np.random.default_rng(m + n + k)
    a = rng.standard_normal((m, k)).astype(np.float32)
    w = (3.0 * rng.standard_normal((n, k)) / np.sqrt(k)).astype(np.float32)
    b = rng.standard_normal(n).astype(np.float32)
    ap = (-3 + rng.standard_normal(n)).astype(np.float32)
    e = ops.ELEM_F16 if elem == "f16" else ops.ELEM_BF16
    kind = ops.OUT_BF16_SPLIT if nsplit == 3 else (ops.OUT_F16 if elem == "f16" else ops.OUT_BF16)
    a_hi, a_lo = ops.convert_f32(_t(a, dev), kind)
    w_hi, w_lo = ops.convert_f32(_t(w, dev), kind)
    bd, apd = _t(b, dev), _t(ap, dev)
    logits, _ = ops.linear_bias_act(a_hi, a_lo, w_hi, w_lo, bd, m, n, k, out_kind=ops.OUT_F32, nsplit=nsplit, elem=e)
    for prior, scale in ((None, 1.0), (apd, 0.7)):
        want = ops.head(logits, n, rows=m, prior=prior, prior_scale=scale).cpu().numpy()
        got = ops.linear_logsoftmax(a_hi, a_lo, w_hi, w_lo, bd, m, n, k, prior=prior, prior_scale=scale, nsplit=nsplit,
                                    elem=e).cpu().numpy()
        assert got.shape == (m, n)
        assert np.abs(got - want).max() < 2e-5
        assert np.abs(np.exp(got.astype(np.float64)).sum(axis=1) - 1).max() < 1e-4
    if elem == "f16" and nsplit == 1:  # float64 check on the fp16-rounded operands
        z = a_hi.float().cpu().numpy().astype(np.float64)[:m, :k] @ w_hi.float().cpu().numpy().astype(np.float64)[:n, :k].T + b
        z -= z.max(axis=1, keepdims=True)
        ref = z - np.log(np.exp(z).sum(axis=1, keepdims=True))
        got = ops.linear_logsoftmax(a_hi, a_lo, w_hi, w_lo, bd, m, n, k, elem=e).cpu().numpy()
        assert np.abs(got - ref).max() < 1e-4  # fp32 accumulation over K <= 2048 + approximate exp2
    # scatter map: a permutation with one dropped row and one zero-filled row
    rmap = rng.permutation(m).astype(np.int32)
    lost = int(rmap[min(77, m - 1)])
    rmap[5], rmap[min(77, m - 1)] = -1, -2 - int(rmap[5])
    zrow = -2 - int(rmap[min(77, m - 1)])
    rm = _t(rmap, dev)
    want = torch.full((m, n), 7.0, device=dev)
    ops.head(logits, n, rows=m, prior=apd, out=want, out_row_map=rm)
    got = torch.full((m, n), 7.0, device=dev)
    ops.linear_logsoftmax(a_hi, a_lo, w_hi, w_lo, bd, m, n, k, prior=apd, nsplit=nsplit, elem=e, out=got, out_row_map=rm)
    want, got = want.cpu().numpy(), got.cpu().numpy()
    assert np.all(got[zrow] == 0) and np.all(got[lost] == 7.0)
    assert np.abs(got - want).max() < 2e-5
    # compact transfer format
    ld16 = (n + 7) // 8 * 8
    o16w = torch.full((m, ld16), 9.0, dtype=torch.float16, device=dev)
    refw = torch.full((m,), 9.0, device=dev)
    ops.head(logits, n, rows=m, prior=apd, out16=(o16w, refw), out_row_map=rm)
    o16 = torch.full((m, ld16), 9.0, dtype=torch.float16, device=dev)
    ref = torch.full((m,), 9.0, device=dev)
    ops.linear_logsoftmax(a_hi, a_lo, w_hi, w_lo, bd, m, n, k, prior=apd, nsplit=nsplit, elem=e, out16=(o16, ref),
                          out_row_map=rm)
    assert np.abs(ref.cpu().numpy() - refw.cpu().numpy()).max() < 2e-5
    d = (o16.float() - o16w.float()).abs().cpu().numpy()[:, :n]
    scale_ = np.maximum(o16w.float().abs().cpu().numpy()[:, :n], 1.0)
    assert (d <= 2.0 ** -10 * scale_ + 2e-5).all()  # one fp16 ulp: the two paths round v - max from slightly different v
    assert np.all(o16.cpu().numpy()[:, n:] == 9.0)  # padding columns untouched


@pytest.mark.parametrize("m,n,k", [(128, 256, 64), (1, 16, 8), (300, 1024, 544), (1000, 1909, 440), (77, 40, 40),
                                   (2048, 2048, 2048), (513, 2048, 140), (129, 1909, 1024),
                                   # M >= 4096 with K >= 384 runs the CTA-pair (cta_group::2) kernel: ragged M, ragged N
                                   (4096, 2048, 2048), (4173, 1909, 1024), (5000, 512, 544),
                                   # single-CTA kernel at large M: K = 72 < 384 keeps it off the pair kernel
                                   (4100, 128, 72)])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_linear_bias_act(ops, dev, m, n, k, mode):
    rng = np.random.default_rng(m * 7 + n)
    a = rng.standard_normal((m, k)).astype(np.float32)
    w = (rng.standard_normal((n, k)) / np.sqrt(k)).astype(np.float32)
    b = rng.standard_normal(n).astype(np.float32)
    split = mode == "fp32"
    kind = ops.OUT_BF16_SPLIT if split else ops.OUT_BF16
    a_hi, a_lo = ops.convert_f32(_t(a, dev), kind)
    w_hi, w_lo = ops.convert_f32(_t(w, dev), kind)
    for act in ("relu", "identity"):
        got, _ = ops.linear_bias_act(a_hi, a_lo, w_hi, w_lo, _t(b, dev), m, n, k, act=act, out_kind=ops.OUT_F32,
                                     nsplit=3 if split else 1)
        got = got.cpu().numpy()[:, :n]
        if split:
            ref = a.astype(np.float64) @ w.astype(np.float64).T + b
            tol = 2e-4  # bf16x3: 16 mantissa bits per operand
        else:
            ref = _bf16(a).astype(np.float64) @ _bf16(w).astype(np.float64).T + b
            tol = 5e-5  # exact products of bf16 inputs, fp32 accumulation
        ref = O.activation(act)(ref)
        assert np.abs(got - ref).max() < tol * max(1.0, np.abs(ref).max())
    # bf16 / split outputs of the hidden layers
    hi, lo = ops.linear_bias_act(a_hi, a_lo, w_hi, w_lo, _t(b, dev), m, n, k, act="relu", out_kind=kind,
                                 nsplit=3 if split else 1)
    rec = hi.float() if lo is None else hi.float() + lo.float()
    assert np.abs(rec.cpu().numpy()[:, :n] - ref * (ref > 0)).max() < (2e-4 if split else 2e-2) * max(1.0, np.abs(ref).max())


def _f16(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.float16).to(torch.float32).numpy()


@pytest.mark.parametrize("m,n,k", [(128, 256, 64), (300, 1024, 544), (1000, 1909, 440), (4173, 1909, 1024),
                                   (5000, 512, 544)])
def test_linear_fp16_operands(ops, dev, m, n, k):
    """NNAM_ELEM_F16: exact products of fp16 inputs, fp32 accumulation, fp32 / fp16 outputs (1-CTA and pair kernels)."""
    rng = np.random.default_rng(m + n + k)
    a = rng.standard_normal((m, k)).astype(np.float32)
    w = (rng.standard_normal((n, k)) / np.sqrt(k)).astype(np.float32)
    b = rng.standard_normal(n).astype(np.float32)
    a_hi, _ = ops.convert_f32(_t(a, dev), ops.OUT_F16)
    w_hi, _ = ops.convert_f32(_t(w, dev), ops.OUT_F16)
    assert a_hi.dtype == torch.float16 and np.array_equal(a_hi.float().cpu().numpy()[:, :k], _f16(a))
    ref = _f16(a).astype(np.float64) @ _f16(w).astype(np.float64).T + b
    got, _ = ops.linear_bias_act(a_hi, None, w_hi, None, _t(b, dev), m, n, k, act="identity", out_kind=ops.OUT_F32,
                                 elem=ops.ELEM_F16)
    assert np.abs(got.cpu().numpy()[:, :n] - ref).max() < 5e-5 * max(1.0, np.abs(ref).max())
    hi, _ = ops.linear_bias_act(a_hi, None, w_hi, None, _t(b, dev), m, n, k, act="relu", out_kind=ops.OUT_F16,
                                elem=ops.ELEM_F16)
    assert hi.dtype == torch.float16
    assert np.abs(hi.float().cpu().numpy()[:, :n] - ref * (ref > 0)).max() < 2e-3 * max(1.0, np.abs(ref).max())


def test_fp16_conversions_saturate(ops, dev):
    big = torch.tensor([[1e6, -1e6, 65504.0, 7e4, 1.0, -2.0, 0.0, 3e-8]], device=dev)
    hi, _ = ops.convert_f32(big, ops.OUT_F16)
    got = hi.float().cpu().numpy()[0]
    assert np.isfinite(got).all() and got[0] == 65504.0 and got[1] == -65504.0 and got[3] == 65504.0 and got[4] == 1.0


@pytest.mark.parametrize("nsplit", [2, 4])
@pytest.mark.parametrize("m", [300, 4200])
def test_linear_partial_split_passes(ops, dev, nsplit, m):
    """NNAM_SPLIT_A (activations as hi/lo pairs) and NNAM_SPLIT_W (weights): the split operand carries 16 mantissa bits,
    the other one stays plain bf16."""
    n, k = 520, 544
    rng = np.random.default_rng(nsplit + m)
    a = rng.standard_normal((m, k)).astype(np.float32)
    w = (rng.standard_normal((n, k)) / np.sqrt(k)).astype(np.float32)
    a_hi, a_lo = ops.convert_f32(_t(a, dev), ops.OUT_BF16_SPLIT)
    w_hi, w_lo = ops.convert_f32(_t(w, dev), ops.OUT_BF16_SPLIT)
    got, _ = ops.linear_bias_act(a_hi, a_lo, w_hi, w_lo, None, m, n, k, out_kind=ops.OUT_F32, nsplit=nsplit)
    a_eff = a if nsplit == ops.SPLIT_A else _bf16(a)
    w_eff = w if nsplit == ops.SPLIT_W else _bf16(w)
    ref = a_eff.astype(np.float64) @ w_eff.astype(np.float64).T
    assert np.abs(got.cpu().numpy()[:, :n] - ref).max() < 2e-4 * max(1.0, np.abs(ref).max())
    plain = _bf16(a).astype(np.float64) @ _bf16(w).astype(np.float64).T
    assert np.abs(plain - ref).max() > 1e-3  # the pass really changes the result


def test_splice_and_gather_fp16_output(ops, dev, golden_dir):
    """K1 with NNAM_OUT_F16: the fp32 result of the bit-exact path rounded once to fp16."""
    rng = np.random.default_rng(5)
    x = rng.standard_normal((700, 40)).astype(np.float32)
    iv = rng.standard_normal((700, 100)).astype(np.float32)
    ft = O.load_kaldi_feature_transform(os.path.join(golden_dir, "final.feature_transform"))
    want = np.concatenate((O.apply_kaldi_feature_transform(O.splicing(x, range(-5, 6)), ft), iv), axis=1)
    hi, _ = ops.splice_transform(_t(x, dev), 700, 5, _t(ft["addShift"], dev), _t(ft["rescale"], dev), _t(iv, dev),
                                 out_kind=ops.OUT_F16)
    assert hi.dtype == torch.float16 and np.array_equal(hi.float().cpu().numpy()[:, :540], _f16(want))
    ftm = O.select_transform_for_network(ft, "lstm")
    rmap = torch.from_numpy(rng.integers(0, 700, 333).astype(np.int32)).to(dev)
    hi, _ = ops.gather_transform(_t(x, dev), rmap, _t(ftm["addShift"], dev), _t(ftm["rescale"], dev), _t(iv, dev),
                                 out_kind=ops.OUT_F16)
    sel = rmap.cpu().numpy()
    wantg = np.concatenate((O.apply_kaldi_feature_transform(x[sel], ftm), iv[sel]), axis=1)
    assert np.array_equal(hi.float().cpu().numpy()[:, :140], _f16(wantg))


def test_linear_activations_match_chainer_formulation(ops, dev):
    rng = np.random.default_rng(3)
    a = rng.standard_normal((256, 512)).astype(np.float32)
    w = (rng.standard_normal((512, 512)) / np.sqrt(512)).astype(np.float32)
    a_hi, a_lo = ops.convert_f32(_t(a, dev), ops.OUT_BF16_SPLIT)
    w_hi, w_lo = ops.convert_f32(_t(w, dev), ops.OUT_BF16_SPLIT)
    for act in ("sigmoid", "tanh"):
        got, _ = ops.linear_bias_act(a_hi, a_lo, w_hi, w_lo, None, 256, 512, 512, act=act, out_kind=ops.OUT_F32, nsplit=3)
        ref = O.activation(act)((a.astype(np.float64) @ w.astype(np.float64).T).astype(np.float32))
        assert np.abs(got.cpu().numpy() - ref).max() < 1e-4


def test_linear_rejects_bad_arguments(ops, dev):
    from nnacousticmodeling_b200 import NnamError
    a = torch.zeros(16, 24, dtype=torch.bfloat16, device=dev)
    w = torch.zeros(16, 24, dtype=torch.bfloat16, device=dev)
    with pytest.raises(NnamError):
        ops.linear_bias_act(a, None, w, None, None, 16, 16, 24, nsplit=3)  # missing lo operands
    with pytest.raises(NnamError):
        ops.linear_bias_act(a, None, w, None, None, 16, 16, 24, nsplit=2)  # SPLIT_A without a_lo
    with pytest.raises(NnamError):
        ops.linear_bias_act(a, None, w, None, None, 16, 16, 24, nsplit=5)  # not a NNAM_SPLIT_* code
    with pytest.raises(NnamError):  # the hi/lo split passes are defined for bf16 operands only
        h = torch.zeros(16, 24, dtype=torch.float16, device=dev)
        ops.linear_bias_act(h, a, h, a, None, 16, 16, 24, nsplit=3, elem=ops.ELEM_F16)
    with pytest.raises(NnamError):  # element type / buffer dtype mismatch is caught on the host side
        ops.linear_bias_act(a, None, w, None, None, 16, 16, 24, elem=ops.ELEM_F16)
    with pytest.raises(NnamError):
        a20 = torch.zeros(16, 20, dtype=torch.bfloat16, device=dev)
        ops.linear_bias_act(a20, None, w, None, None, 16, 16, 20)  # lda = 20 elements: rows not 16-byte aligned
