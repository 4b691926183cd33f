"""K2 / K4 element by element: every GEMM, head and fused output-layer instance against the float64 references of
tests/gemm_reference.py, at the tile and dispatch edges.  -m gpu.

Operands are built with torch, not convert_f32: columns [K, lda), rows past M of A and rows past N of W are NaN, and
some cases pass A as a column slice at an offset of 8 or 24 elements with NaN on both sides.  Outputs are column
slices of wider buffers filled with a sentinel; everything outside [0, M) x [0, N) must keep it.  f32 GEMM outputs are
checked against the per-element bound; 16-bit outputs exactly against the same kernel's f32 output where both use the
same tile width (gemm_reference.check_16bit), else against the bound plus half an ulp of the output type.

Instances reached on a 148-SM B200 (tests/gemm_reference.py mirrors the dispatch: gemm_instance, head_instance,
fused_cluster; tests/test_gemm_reference_cpu.py checks every case's label against it):

  kernel                                    tile / template            case ids
  gemm_bias_act_kernel<OUT, 4, 2>           bn 32 .. 256, 1 CTA/tile   g1-* (M < 4096, or N < 128, or K < 384)
      bn 32 (f32) / 64 (16-bit)                                        g1-1-1-8, g1-127-31-16, g1-128-32-56
      bn 64                                                            g1-129-33-64, g1-4095-64-72
      bn 96 (f32) / 128 (16-bit)                                       g1-5000-65-72, g1-127-65-72-off24
      bn 256                                                           g1-x (cross product), g1-128-255-2056,
                                                                       g1-127-256-16
      bn 160 (f32) / 192 (16-bit), 2 column tiles                      g1-129-257-72, g1-129-257-56-off8
      bn 256, 288 tiles > 148 CTAs                                     g1-4095-2049-72
      fp16 output saturation                                           g1-sat
  gemm_bias_act_2sm_kernel<OUT>             256 x bn per CTA pair      g2-* (M >= 4096, N >= 128, K >= 384)
      bn 128 (halves of 64 rows)                                       g2-4096-128-384
      fp16 output saturation                                           g2-sat
      bn 160 (f32) / 192 (16-bit)                                      g2-4097-160-392, g2-4225-320-384
      bn 192                                                           g2-4224-192-1032, g2-4097-192-392-off8
      bn 224 (f32) / 256 (16-bit)                                      g2-4225-224-384
      bn 256                                                           g2-x (cross product), g2-4351-256-392
      bn 256, 153 tiles > 74 pairs                                     g2-4351-2049-392
  head_fast_kernel<1, *>                    C + 3 <= 128               h-fast-1, h-fast-125
  head_fast_kernel<4, *>                    C + 3 in (128, 512]        h-fast-126, h-fast-509, h-fast-126-grid
  head_fast_kernel<8, *>                    C + 3 in (512, 1024]       h-fast-510, h-fast-1021
  head_fast_kernel<15, *>                   C + 3 in (1024, 1920]      h-fast-1022, h-fast-1917
  head_fast_kernel<16, *>                   C + 3 in (1920, 2048]      h-fast-1918, h-fast-1919, h-fast-2045
  head_kernel<4, false, *>                  C <= 128, one input        h-gen4-ld
  head_kernel<4, true, *>                   ensembles                  h-gen4-ens2, h-gen4-ens2-grid
  head_kernel<32, false, *>                 C <= 1024                  h-gen32-rpl
  head_kernel<32, true, *>                                             h-gen32-ens5-prenorm, h-gen32-prenorm-raw
  head_kernel<64, false, *>                 C > 1024                   h-gen64-2046, h-gen64-2048, h-gen64-ld
  head_kernel<64, true, *>                                             h-gen64-ens2-rpl
  gemm_logsoftmax_kernel<MODE>              cluster of ceil(N / 256)   f-256-* (1), f-257-* (2), f-1000-* (4),
                                                                       f-1100-* (5), f-1400-* (6), f-1700-* (7),
                                                                       f-1909-* (8)

The head's float32 rows, compact and scoring forms run for every head case (``*`` = SCORE false / true); the fast
kernel's compact form uses ld16 > 128 * NV4 where that keeps ld16 <= 2048.  Row maps with a dropped and a zero-filled
row are checked row by row.

Each case prints ``K2|K4|K2K4 <case> worst=<e> bound=<b> of-bound=<r>`` (run with -s): the error and the bound at the
element with the largest ratio r, which must not exceed 1.  Exact checks print the number of differing elements."""
import os
import re
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import gemm_reference as G  # noqa: E402

NAN = float("nan")
SENT = -7.25  # exact in every output type


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from nnacousticmodeling_b200 import ops as _ops
    return _ops


def _round_up(v, m):
    return (v + m - 1) // m * m


# ----------------------------------------------------------------------------------------------------- case tables
ALL_OUTS = (G.OUT_F32, G.OUT_BF16, G.OUT_F16, G.OUT_BF16_SPLIT)
ALL_MODES = tuple(G.MODES)


def _g(cid, M, N, K, kernel, bn, modes=("bf16",), acts=("identity",), outs=(G.OUT_F32,), bias=True, a_off=0,
       scale_z=1.0):
    return dict(id=cid, M=M, N=N, K=K, kernel=kernel, bn=bn, modes=modes, acts=acts, outs=outs, bias=bias, a_off=a_off,
                scale_z=scale_z)


# kernel: "1cta" / "pair"; bn: the f32-output tile width the case claims
GEMM_CASES = [
    _g("g1-x", 129, 255, 72, "1cta", 256, ALL_MODES, G.ACTS, ALL_OUTS),
    _g("g1-1-1-8", 1, 1, 8, "1cta", 32, ("bf16", "split_aw"), ("relu",), (G.OUT_F32, G.OUT_BF16)),
    _g("g1-127-31-16", 127, 31, 16, "1cta", 32, ("fp16",), ("sigmoid",), (G.OUT_F32, G.OUT_F16), bias=False),
    _g("g1-128-32-56", 128, 32, 56, "1cta", 32, ("split_a",), ("tanh",), (G.OUT_F32, G.OUT_BF16_SPLIT)),
    _g("g1-129-33-64", 129, 33, 64, "1cta", 64, ("split_w", "bf16"), ("relu",), ALL_OUTS),
    _g("g1-4095-64-72", 4095, 64, 72, "1cta", 64, ("fp16",), ("identity",), (G.OUT_F32, G.OUT_F16)),
    _g("g1-5000-65-72", 5000, 65, 72, "1cta", 96, ("split_aw",), ("sigmoid",), (G.OUT_F32, G.OUT_BF16_SPLIT)),
    _g("g1-127-65-72-off24", 127, 65, 72, "1cta", 96, ("bf16",), ("tanh",), (G.OUT_F32, G.OUT_BF16), a_off=24),
    _g("g1-128-255-2056", 128, 255, 2056, "1cta", 256, ("bf16", "split_aw"), ("identity",), (G.OUT_F32, G.OUT_BF16)),
    _g("g1-127-256-16", 127, 256, 16, "1cta", 256, ("split_w",), ("relu",), (G.OUT_F32, G.OUT_BF16_SPLIT)),
    _g("g1-129-257-72", 129, 257, 72, "1cta", 160, ("fp16", "split_a"), ("sigmoid",), (G.OUT_F32, G.OUT_F16)),
    _g("g1-129-257-56-off8", 129, 257, 56, "1cta", 160, ("bf16",), ("relu",), (G.OUT_F32, G.OUT_BF16), a_off=8),
    _g("g1-4095-2049-72", 4095, 2049, 72, "1cta", 256, ("bf16",), ("relu",), (G.OUT_F32, G.OUT_BF16)),
    _g("g1-sat", 128, 64, 64, "1cta", 64, ("fp16",), ("identity",), (G.OUT_F32, G.OUT_F16), scale_z=3e5),
    _g("g2-sat", 4096, 128, 384, "pair", 128, ("fp16",), ("identity",), (G.OUT_F32, G.OUT_F16), scale_z=3e5),
    _g("g2-x", 4225, 256, 392, "pair", 256, ALL_MODES, G.ACTS, ALL_OUTS),
    _g("g2-4096-128-384", 4096, 128, 384, "pair", 128, ("bf16", "split_a"), ("relu",), ALL_OUTS, bias=False),
    _g("g2-4097-160-392", 4097, 160, 392, "pair", 160, ("fp16", "split_w"), ("tanh",), (G.OUT_F32, G.OUT_F16)),
    _g("g2-4225-320-384", 4225, 320, 384, "pair", 160, ("bf16",), ("sigmoid",), (G.OUT_F32, G.OUT_BF16)),
    _g("g2-4224-192-1032", 4224, 192, 1032, "pair", 192, ("split_aw", "fp16"), ("identity",), ALL_OUTS),
    _g("g2-4097-192-392-off8", 4097, 192, 392, "pair", 192, ("bf16",), ("relu",), (G.OUT_F32, G.OUT_BF16), a_off=8),
    _g("g2-4225-224-384", 4225, 224, 384, "pair", 224, ("split_a",), ("sigmoid",), (G.OUT_F32, G.OUT_BF16_SPLIT)),
    _g("g2-4351-256-392", 4351, 256, 392, "pair", 256, ("split_w",), ("tanh",), (G.OUT_F32, G.OUT_BF16)),
    _g("g2-4351-2049-392", 4351, 2049, 392, "pair", 256, ("bf16",), ("relu",), (G.OUT_F32, G.OUT_BF16)),
]


def _h(cid, C, inst, rows=300, n_inputs=1, pre_normalize=False, rpl=False, ld_in=None, ld_out=None, w0=1.0,
       prior=True, final_normalize=True, forms=("rows", "map", "compact", "score")):
    return dict(id=cid, C=C, inst=inst, rows=rows, n_inputs=n_inputs, pre_normalize=pre_normalize, rpl=rpl,
                ld_in=_round_up(C, 4) if ld_in is None else ld_in, ld_out=C if ld_out is None else ld_out, w0=w0,
                prior=prior, final_normalize=final_normalize, forms=forms)


# inst: ("fast", NV4) or ("generic", NV, MULTI)
HEAD_CASES = [
    _h("h-fast-1", 1, ("fast", 1), ld_out=5),
    _h("h-fast-125", 125, ("fast", 1), w0=0.9),
    _h("h-fast-126", 126, ("fast", 4), ld_out=131),
    _h("h-fast-509", 509, ("fast", 4), w0=0.9),
    _h("h-fast-126-grid", 126, ("fast", 4), rows=10000, forms=("rows", "score")),
    _h("h-fast-510", 510, ("fast", 8)),
    _h("h-fast-1021", 1021, ("fast", 8), w0=1.25),
    _h("h-fast-1022", 1022, ("fast", 15)),
    _h("h-fast-1917", 1917, ("fast", 15), ld_out=1921),
    _h("h-fast-1918", 1918, ("fast", 16)),
    _h("h-fast-1919", 1919, ("fast", 16)),  # odd pitch: row starts at a = 3, whose last columns need NV4 = 16
    _h("h-fast-2045", 2045, ("fast", 16), w0=0.9),
    _h("h-gen64-2046", 2046, ("generic", 64, False)),
    _h("h-gen64-2048", 2048, ("generic", 64, False), ld_out=2051),
    _h("h-gen4-ld", 100, ("generic", 4, False), ld_in=101, ld_out=103, w0=0.9),
    _h("h-gen4-ens2", 127, ("generic", 4, True), n_inputs=2),
    _h("h-gen4-ens2-grid", 99, ("generic", 4, True), rows=10000, n_inputs=2, forms=("rows", "score")),
    _h("h-gen32-rpl", 1000, ("generic", 32, False), rpl=True, ld_out=1003),
    _h("h-gen32-ens5-prenorm", 1001, ("generic", 32, True), n_inputs=5, pre_normalize=True),
    _h("h-gen32-prenorm-raw", 999, ("generic", 32, True), n_inputs=2, pre_normalize=True, prior=False,
       final_normalize=False, forms=("rows",)),
    _h("h-gen64-ld", 1909, ("generic", 64, False), ld_in=1909),
    _h("h-gen64-ens2-rpl", 1909, ("generic", 64, True), n_inputs=2, rpl=True),
]


def _f(cid, M, N, K, mode, forms=("rows", "compact", "score"), row_map=False):
    return dict(id=cid, M=M, N=N, K=K, mode=mode, forms=forms, row_map=row_map, cluster=G.fused_cluster(N))


FUSED_CASES = [
    _f("f-256-1", 1, 256, 136, "bf16"),
    _f("f-257-127", 127, 257, 136, "fp16", row_map=True),
    _f("f-1000-128", 128, 1000, 72, "split_a"),
    _f("f-1100-129", 129, 1100, 136, "split_aw", row_map=True),
    _f("f-1400-129", 129, 1400, 392, "split_w"),
    _f("f-1700-128", 128, 1700, 136, "fp16"),
    _f("f-1909-4173", 4173, 1909, 136, "bf16", row_map=True),
    _f("f-1909-129", 129, 1909, 1032, "split_aw"),
]


def gemm_case_instance(case, out_kind):
    return G.gemm_instance(case["M"], case["N"], case["K"], out_kind)


def head_case_instance(case, form):
    ld16 = compact_ld16(case) if form == "compact" else None
    return G.head_instance(case["n_inputs"], case["pre_normalize"], case["rpl"], case["ld_in"], case["C"], ld16,
                           form == "score")


def compact_ld16(case):
    C = case["C"]
    inst = G.head_instance(case["n_inputs"], case["pre_normalize"], case["rpl"], case["ld_in"], C)
    if inst[0] == "fast":
        return min(128 * inst[1] + 8, 2048)
    return _round_up(C, 8) + 8


# ----------------------------------------------------------------------------------------------------- GEMM
def _dev_plane(vals, dtype, rows_pad, off):
    """(rows + rows_pad, off + lda) NaN buffer holding ``vals`` at column ``off``; returns the view from ``off``."""
    rows, K = vals.shape
    lda = _round_up(K, 8) + 8
    buf = torch.full((rows + rows_pad, off + lda), NAN, dtype=dtype, device="cuda")
    buf[:rows, off:off + K] = torch.from_numpy(np.ascontiguousarray(vals)).to(dtype).cuda()
    return buf[:, off:]


def _device_operands(P, a_off):
    e16 = torch.float16 if P["f16"] else torch.bfloat16
    d = {"a_hi": _dev_plane(P["a_hi"], e16, 5, a_off), "w_hi": _dev_plane(P["w_hi"], e16, 7, 0),
         "a_lo": None, "w_lo": None}
    if P["nsplit"] in (G.SPLIT_A, G.SPLIT_AW):
        d["a_lo"] = _dev_plane(P["a_lo"], torch.bfloat16, 5, a_off)
    if P["nsplit"] in (G.SPLIT_W, G.SPLIT_AW):
        d["w_lo"] = _dev_plane(P["w_lo"], torch.bfloat16, 7, 0)
    return d


def _run_gemm(ops, D, P, bias_t, M, N, K, act, out_kind):
    dt = ops.out_dtype(out_kind)
    off = 4 if out_kind == G.OUT_F32 else 8
    width = off + _round_up(N, 16) + 16
    bufs = [torch.full((M + 2, width), SENT, dtype=dt, device="cuda")
            for _ in range(2 if out_kind == G.OUT_BF16_SPLIT else 1)]
    out = (bufs[0][:M, off:off + N], bufs[1][:M, off:off + N] if len(bufs) == 2 else None)
    ops.linear_bias_act(D["a_hi"], D["a_lo"], D["w_hi"], D["w_lo"], bias_t, M, N, K, act=act, out_kind=out_kind,
                        nsplit=P["nsplit"], out=out, elem=ops.ELEM_F16 if P["f16"] else ops.ELEM_BF16)
    torch.cuda.synchronize()
    res = []
    for b in bufs:
        h = b.float().cpu().numpy()
        keep = h.copy()
        keep[:M, off:off + N] = SENT
        assert np.all(keep == SENT), "GEMM output: a store landed outside [0, M) x [0, N) of the slice"
        res.append(h[:M, off:off + N])
    return res[0], (res[1] if len(res) == 2 else None)


def _report(tag, name, err, bound):
    r = np.abs(err) / bound
    r[~np.isfinite(err)] = np.inf
    i = np.unravel_index(int(np.argmax(r)), r.shape)
    print(f"{tag} {name} worst={float(np.abs(err)[i]):.3g} bound={float(bound[i]):.3g} of-bound={float(r[i]):.3g}")
    assert r[i] <= 1.0, f"{tag} {name}: element {tuple(int(v) for v in i)} error {float(err[i])!r} bound {float(bound[i])!r}"
    return float(r[i])


def run_gemm_case(ops, case):
    M, N, K = case["M"], case["N"], case["K"]
    for mode in case["modes"]:
        seed = M * 131 + N * 7 + K + len(mode)
        P = G.make_gemm_operands(seed, M, N, K, mode, case["scale_z"])
        D = _device_operands(P, case["a_off"])
        bias = P["bias"] if case["bias"] else None
        bias_t = None
        if bias is not None:
            bbuf = torch.full((N + 64,), NAN, device="cuda")
            bbuf[:N] = torch.from_numpy(bias).cuda()
            bias_t = bbuf[:N]
        prods = G.gemm_products(P, P["nsplit"])
        for act in case["acts"]:
            y, z, S = G.gemm_ref(P, bias, act, P["nsplit"], prods)
            if case["scale_z"] > G.F16_MAX:  # the saturation case: a good share of |z| lies beyond the fp16 range
                assert (np.abs(z) > 65520).mean() > 0.1
            bound = G.gemm_bound(y, z, S, K, P["nsplit"], act)
            v32, _ = _run_gemm(ops, D, P, bias_t, M, N, K, act, G.OUT_F32)
            name = f"{case['id']} {mode} {act} f32"
            _report("K2", name, v32 - y, bound)
            bn32 = gemm_case_instance(case, G.OUT_F32)["bn"]
            for out_kind in case["outs"]:
                if out_kind == G.OUT_F32:
                    continue
                hi, lo = _run_gemm(ops, D, P, bias_t, M, N, K, act, out_kind)
                name = f"{case['id']} {mode} {act} {G.OUT_NAMES[out_kind]}"
                assert np.isfinite(hi).all(), f"K2 {name}: non-finite 16-bit output (an fp16 store overflowed to inf?)"
                if gemm_case_instance(case, out_kind)["bn"] == bn32:
                    bad = G.check_16bit(v32, hi, lo, out_kind)
                    print(f"K2 {name} exact: {bad} of {hi.size} elements differ from the rounded f32 output")
                    assert bad == 0, f"K2 {name}: {bad} elements are not the rounding of the f32 output"
                else:
                    kind = "f16" if out_kind == G.OUT_F16 else "bf16"
                    got = hi if lo is None else hi.astype(np.float64) + lo
                    half = 0.5 * G.ulp16(y, kind) if lo is None else 2.0 ** -17 * np.abs(y)
                    want = np.clip(y, -G.F16_MAX, G.F16_MAX) if out_kind == G.OUT_F16 else y
                    _report("K2", name, got - want, bound + half)


@pytest.mark.parametrize("case", GEMM_CASES, ids=[c["id"] for c in GEMM_CASES])
def test_gemm_instance(ops, case):
    run_gemm_case(ops, case)


# ----------------------------------------------------------------------------------------------------- head
def _row_map(rows, seed):
    rng = np.random.default_rng(seed)
    perm = rng.permutation(rows).astype(np.int32)
    rmap = perm.copy()
    if rows >= 3:
        rmap[1] = -1
        rmap[2] = -2 - int(perm[1])
    return rmap


def _head_inputs(case):
    C, rows, k = case["C"], case["rows"], case["n_inputs"]
    xs = G.make_head_logits(C * 3 + rows + k, rows, C, k)
    prior, rpl = G.make_head_extras(C, C)
    dev = []
    for x in xs:
        buf = torch.full((rows, case["ld_in"]), NAN, device="cuda")
        buf[:, :C] = torch.from_numpy(x).cuda()
        dev.append(buf[:, :C])
    weights = [case["w0"]] if k == 1 else [float(np.float32(v)) for v in np.linspace(0.5, 1.5, k) / k]
    return xs, dev, weights, prior, rpl


def run_head_case(ops, case):
    C, rows = case["C"], case["rows"]
    xs, dev, weights, prior, rpl = _head_inputs(case)
    prior_t = torch.from_numpy(prior).cuda() if case["prior"] else None
    rpl_t = tuple(torch.from_numpy(a).cuda() for a in rpl) if case["rpl"] else None
    ps = 0.7
    y, mag, lse_sum, n_lse = G.head_ref(xs, C, weights, case["pre_normalize"], rpl if case["rpl"] else None,
                                        prior if case["prior"] else None, ps, case["final_normalize"])
    kw = dict(weights=weights, pre_normalize=case["pre_normalize"], rpl=rpl_t, prior=prior_t, prior_scale=ps,
              final_normalize=case["final_normalize"])
    rmap = _row_map(rows, C)
    rmap_t = torch.from_numpy(rmap).cuda()
    worst = 0.0
    for form in case["forms"]:
        inst = head_case_instance(case, form)
        bound = G.head_bound(mag, lse_sum, n_lse, G.head_terms_per_lane(inst))
        name = f"{case['id']} {form} {G.head_kernel_name(inst)}"
        if form in ("rows", "map"):
            buf = torch.full((rows, case["ld_out"]), SENT, device="cuda")
            out = buf[:, :C]
            ops.head(dev, C, out=out, out_row_map=rmap_t if form == "map" else None, **kw)
            got = buf.cpu().numpy()
            assert np.all(got[:, C:] == SENT), f"K4 {name}: pitch columns overwritten"
            got = got[:, :C]
            if form == "rows":
                worst = max(worst, _report("K4", name, got - y, bound))
                continue
            want, written, zeroed = G.map_rows(y, rmap, rows)
            bmap, _, _ = G.map_rows(bound, rmap, rows)
            assert np.all(got[zeroed] == 0) and np.all(got[~written & ~zeroed] == SENT), f"K4 {name}: row map"
            worst = max(worst, _report("K4", name, got[written] - want[written], bmap[written]))
        elif form == "compact":
            ld16 = compact_ld16(case)
            o16 = torch.full((rows, ld16), SENT, dtype=torch.float16, device="cuda")
            ref = torch.full((rows,), SENT, device="cuda")
            ops.head(dev, C, out16=(o16, ref), out_row_map=rmap_t, **kw)
            g16_all = o16.float().cpu().numpy()
            g16 = g16_all[:, :C].astype(np.float64)
            gref = ref.cpu().numpy().astype(np.float64)
            want, written, zeroed = G.map_rows(y, rmap, rows)
            bmap, _, _ = G.map_rows(bound, rmap, rows)
            # pitch [C, ld16): the generic kernel leaves it alone; the fast kernel's 8-byte chunk stores cover columns up
            # to 128 * NV4 with fp16(-inf - max), saturated (0 in zero-filled rows), and leave the rest alone
            pitch = g16_all[:, C:]
            n_w = min(ld16, 128 * inst[1]) - C if inst[0] == "fast" else 0
            assert np.all(pitch[:, n_w:] == SENT) and np.all(pitch[~written & ~zeroed] == SENT), f"K4 {name}: pitch"
            assert np.all(pitch[written, :n_w] <= -G.F16_MAX) and np.all(pitch[zeroed, :n_w] == 0), f"K4 {name}: pitch"
            assert np.all(g16[zeroed] == 0) and np.all(gref[zeroed] == 0), f"K4 {name}: zero-filled row"
            assert np.all(gref[~written & ~zeroed] == SENT), f"K4 {name}: a row no map entry names was written"
            w, b = want[written], bmap[written]
            top = w.max(axis=1, keepdims=True)
            # fp16 rounding of the offset from the row maximum: half an ulp of |y - max|
            allow = 2 * b + 2.0 ** -11 * (np.abs(w - top) + 2 * b)
            worst = max(worst, _report("K4", name, g16[written] + gref[written, None] - w, allow))
            _report("K4", name + " row_ref", gref[written] - top[:, 0], b.max(axis=1))
        else:  # score
            rng = np.random.default_rng(C + 1)
            targets = rng.integers(0, C, rows).astype(np.int32)
            targets[::13] = -1
            nll = torch.full((rows,), SENT, device="cuda")
            pred = torch.full((rows,), -5, dtype=torch.int32, device="cuda")
            ops.head(dev, C, out_row_map=rmap_t, score=(torch.from_numpy(targets).cuda(), nll, pred), **kw)
            gn, gp = nll.cpu().numpy(), pred.cpu().numpy()
            want, written, zeroed = G.map_rows(y, rmap, rows)
            bmap, _, _ = G.map_rows(bound, rmap, rows)
            assert np.all(gn[zeroed] == 0) and np.all(gp[zeroed] == -1), f"K4 {name}: zero-filled row"
            assert np.all(gn[~written & ~zeroed] == SENT) and np.all(gp[~written & ~zeroed] == -5), f"K4 {name}: map"
            n_ref, n_b, top, sure = G.score_ref(want[written], bmap[written], targets[written])
            worst = max(worst, _report("K4", name + " nll", gn[written] - n_ref, n_b + 1e-30))
            assert np.array_equal(gp[written][sure], top[sure]), f"K4 {name}: pred differs from the float64 argmax"
            assert sure.mean() > 0.5
    return worst


@pytest.mark.parametrize("case", HEAD_CASES, ids=[c["id"] for c in HEAD_CASES])
def test_head_instance(ops, case):
    run_head_case(ops, case)


# ----------------------------------------------------------------------------------------------------- fused
def run_fused_case(ops, case):
    M, N, K, mode = case["M"], case["N"], case["K"], case["mode"]
    P = G.make_gemm_operands(M * 17 + N + K, M, N, K, mode, scale_z=3.0)
    D = _device_operands(P, 0)
    prior, _ = G.make_head_extras(N, N)
    ps = 0.7
    bias_t, prior_t = torch.from_numpy(P["bias"]).cuda(), torch.from_numpy(prior).cuda()
    _, z, S = G.gemm_ref(P, P["bias"], "identity", P["nsplit"])
    gb = G.gemm_bound(z, z, S, K, P["nsplit"], "identity")
    y, mag, lse_sum, n_lse = G.head_ref([z], N, [1.0], prior=prior, prior_scale=ps)
    bound = G.fused_bound(gb, G.head_bound(mag, lse_sum, n_lse, 128 + 2 * case["cluster"]))
    rmap = _row_map(M, N) if case["row_map"] else np.arange(M, dtype=np.int32)
    rmap_t = torch.from_numpy(rmap).cuda() if case["row_map"] else None
    want, written, zeroed = G.map_rows(y, rmap, M)
    bmap, _, _ = G.map_rows(bound, rmap, M)
    kw = dict(prior=prior_t, prior_scale=ps, nsplit=P["nsplit"], elem=ops.ELEM_F16 if P["f16"] else ops.ELEM_BF16,
              out_row_map=rmap_t)
    args = (D["a_hi"], D["a_lo"], D["w_hi"], D["w_lo"], bias_t, M, N, K)
    for form in case["forms"]:
        name = f"{case['id']} {mode} {form} cluster={case['cluster']}"
        if form == "rows":
            buf = torch.full((M + 1, N + 3), SENT, device="cuda")
            ops.linear_logsoftmax(*args, out=buf[:M, :N], **kw)
            got = buf.cpu().numpy()
            assert np.all(got[:, N:] == SENT) and np.all(got[M:] == SENT), f"K2K4 {name}: pitch or rows past M written"
            got = got[:M, :N]
            assert np.all(got[zeroed] == 0) and np.all(got[~written & ~zeroed] == SENT), f"K2K4 {name}: row map"
            _report("K2K4", name, got[written] - want[written], bmap[written])
        elif form == "compact":
            ld16 = _round_up(N + 1, 8)  # at least one pitch column, which must keep the sentinel
            o16 = torch.full((M, ld16), SENT, dtype=torch.float16, device="cuda")
            ref = torch.full((M,), SENT, device="cuda")
            ops.linear_logsoftmax(*args, out16=(o16, ref), **kw)
            g16_all = o16.float().cpu().numpy()
            assert np.all(g16_all[:, N:] == SENT), f"K2K4 {name}: compact pitch columns written"
            g16 = g16_all[:, :N].astype(np.float64)
            gref = ref.cpu().numpy().astype(np.float64)
            assert np.all(g16[zeroed] == 0) and np.all(gref[zeroed] == 0)
            assert np.all(gref[~written & ~zeroed] == SENT)
            w, b = want[written], bmap[written]
            top = w.max(axis=1, keepdims=True)
            allow = 2 * b + 2.0 ** -11 * (np.abs(w - top) + 2 * b)
            _report("K2K4", name, g16[written] + gref[written, None] - w, allow)
        else:
            rng = np.random.default_rng(N)
            targets = rng.integers(0, N, M).astype(np.int32)
            targets[::13] = -1
            nll = torch.full((M,), SENT, device="cuda")
            pred = torch.full((M,), -5, dtype=torch.int32, device="cuda")
            ops.linear_logsoftmax(*args, score=(torch.from_numpy(targets).cuda(), nll, pred), **kw)
            gn, gp = nll.cpu().numpy(), pred.cpu().numpy()
            assert np.all(gn[zeroed] == 0) and np.all(gp[zeroed] == -1)
            assert np.all(gn[~written & ~zeroed] == SENT) and np.all(gp[~written & ~zeroed] == -5)
            n_ref, n_b, top, sure = G.score_ref(want[written], bmap[written], targets[written])
            _report("K2K4", name + " nll", gn[written] - n_ref, n_b + 1e-30)
            assert np.array_equal(gp[written][sure], top[sure]), f"K2K4 {name}: pred differs from the float64 argmax"


@pytest.mark.parametrize("case", FUSED_CASES, ids=[c["id"] for c in FUSED_CASES])
def test_fused_instance(ops, case):
    run_fused_case(ops, case)


# ----------------------------------------------------------------------------------------------------- which kernel ran
def _kernel_names(prof):
    evs = [e for e in prof.events() if getattr(e, "device_type", None) == torch.autograd.DeviceType.CUDA]
    evs.sort(key=lambda e: e.time_range.start)
    return [e.name for e in evs if "nnam::" in e.name]


def test_profiler_confirms_instances(ops):
    """One launch per table row under torch.profiler: the kernel names and template arguments the profiler records
    are the ones the dispatch mirror names.  No kernel recorded is a failure, not a skip."""
    from torch.profiler import ProfilerActivity, profile
    expected, launches = [], []
    for case in GEMM_CASES:
        P = G.make_gemm_operands(1, case["M"], case["N"], case["K"], "bf16")
        D = _device_operands(P, case["a_off"])
        for out_kind in (G.OUT_F32, G.OUT_BF16):
            inst = gemm_case_instance(case, out_kind)
            assert inst["kernel"] == ("gemm_bias_act_2sm_kernel" if case["kernel"] == "pair" else "gemm_bias_act_kernel")
            expected.append(rf"{inst['kernel']}<{out_kind}(, 4, 2)?>" if not inst["pair"]
                            else rf"{inst['kernel']}<{out_kind}>")
            launches.append(lambda D=D, P=P, c=case, o=out_kind: _run_gemm(ops, D, P, None, c["M"], c["N"], c["K"],
                                                                           "identity", o))
    for case in HEAD_CASES:
        _, dev, weights, prior, rpl = _head_inputs(dict(case, rows=64))
        for form in ("rows", "score"):
            if form not in case["forms"]:
                continue
            inst = head_case_instance(case, form)
            expected.append(re.escape(G.head_kernel_name(inst)))

            def run(dev=dev, weights=weights, case=case, form=form, rpl=rpl):
                C = case["C"]
                kw = dict(weights=weights, pre_normalize=case["pre_normalize"],
                          rpl=tuple(torch.from_numpy(a).cuda() for a in rpl) if case["rpl"] else None,
                          final_normalize=case["final_normalize"])
                if form == "rows":
                    ops.head(dev, C, out=torch.empty((64, C), device="cuda"), **kw)
                else:
                    t = torch.zeros(64, dtype=torch.int32, device="cuda")
                    ops.head(dev, C, score=(t, torch.empty(64, device="cuda"), torch.empty_like(t)), **kw)
            launches.append(run)
    for case in FUSED_CASES:
        P = G.make_gemm_operands(1, case["M"], case["N"], case["K"], "bf16")
        D = _device_operands(P, 0)
        expected.append(r"gemm_logsoftmax_kernel<0>")
        launches.append(lambda D=D, c=case: ops.linear_logsoftmax(D["a_hi"], None, D["w_hi"], None, None, c["M"], c["N"],
                                                                  c["K"]))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for f in launches:
            f()
        torch.cuda.synchronize()
    names = _kernel_names(prof)
    assert names, "the profiler recorded no nnam kernels"
    assert len(names) == len(expected), (len(names), len(expected), names[:5])
    for got, want in zip(names, expected):
        assert re.search(r"nnam::(fused::)?" + want + r"\(", got), (want, got)
