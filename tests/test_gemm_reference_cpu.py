"""The references of tests/gemm_reference.py are tight enough to catch the mistakes the K2 / K4 kernels would make.

Models of the kernels (``simulate_gemm``, ``simulate_output``, ``simulate_head_fast``, ``simulate_head_generic``) play
the kernels with one planted mistake at a time; the comparisons used by tests/test_gpu_gemm_head_kernels.py must
reject each by at least REJECT_MARGIN times its bound (exact checks: at least REJECT_MARGIN differing elements), at
the seeds and scales of the GPU cases.  The unplanted models must stay within half of the bound, and every GPU case
must be labelled with the instance the dispatch mirror picks for it.  CPU only."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import gemm_reference as G  # noqa: E402
import test_gpu_gemm_head_kernels as T  # noqa: E402

REJECT_MARGIN = 5.0


def _gemm_score(M, N, K, mode, act, mistake=None, bias=True, scale_z=1.0):
    P = G.make_gemm_operands(M * 131 + N * 7 + K + len(mode), M, N, K, mode, scale_z)
    if not bias:
        P["bias"] = None
    padded = None
    if mistake == "read_padding":
        padded = np.full((M, G.BK * -(-K // G.BK)), np.nan, np.float32)
        padded[:, :K] = P["a_hi"]
    got = G.simulate_gemm(P, M, N, K, act, mistake=mistake, padded=padded)
    y, z, S = G.gemm_ref(P, P["bias"], act, P["nsplit"])
    return float(G.ratio(got, y, G.gemm_bound(y, z, S, K, P["nsplit"], act)).max())


@pytest.mark.parametrize("M,N,K", [(129, 255, 72), (127, 65, 72), (128, 255, 2056), (4225, 256, 392),
                                   (4097, 160, 392), (4224, 192, 1032)])
@pytest.mark.parametrize("mode", list(G.MODES))
def test_unmutated_gemm_model_passes(M, N, K, mode):
    for act in G.ACTS if (M, N, K) == (129, 255, 72) else ("identity",):
        assert _gemm_score(M, N, K, mode, act) <= 0.5


GEMM_MISTAKES = [
    ("drop_ragged_kblock", 129, 257, 72, "bf16", "identity"),
    ("drop_ragged_kblock", 4097, 160, 392, "fp16", "identity"),
    ("read_padding", 129, 257, 72, "bf16", "identity"),
    ("read_padding", 4225, 224, 392, "split_a", "identity"),
    ("bias_other_parity", 4095, 2049, 72, "bf16", "relu"),
    ("bias_other_parity", 4351, 2049, 392, "bf16", "identity"),
    ("bias_shift_box", 129, 255, 72, "bf16", "identity"),
    ("bias_shift_box", 4225, 256, 392, "split_w", "tanh"),
    ("follower_leader_rows", 4225, 256, 392, "bf16", "identity"),
    ("follower_leader_rows", 4225, 224, 384, "split_a", "sigmoid"),
    ("same_w_half", 4096, 128, 384, "bf16", "identity"),
    ("same_w_half", 4097, 160, 392, "fp16", "identity"),
    ("same_w_half", 4224, 192, 1032, "split_aw", "identity"),
    ("same_w_half", 4225, 224, 384, "split_a", "identity"),
    ("same_w_half", 4225, 256, 392, "bf16", "relu"),
    ("split_a_wlo", 129, 255, 72, "split_a", "identity"),
    ("split_a_wlo", 4225, 256, 392, "split_a", "identity"),
    ("aw_drop_hi_wlo", 129, 255, 72, "split_aw", "identity"),
    ("aw_drop_hi_wlo", 4224, 192, 1032, "split_aw", "identity"),
    ("sigmoid_tanh_x", 129, 255, 72, "bf16", "sigmoid"),
    ("sigmoid_tanh_x", 4225, 256, 392, "split_aw", "sigmoid"),
    ("act_before_bias", 129, 255, 72, "bf16", "relu"),
    ("act_before_bias", 129, 255, 72, "split_aw", "tanh"),
    ("act_before_bias", 4225, 256, 392, "fp16", "sigmoid"),
]


@pytest.mark.parametrize("mistake,M,N,K,mode,act", GEMM_MISTAKES)
def test_planted_gemm_mistake_is_rejected(mistake, M, N, K, mode, act):
    assert _gemm_score(M, N, K, mode, act, mistake) >= REJECT_MARGIN


@pytest.mark.parametrize("bn_n", [128, 160, 224, 256])
def test_same_w_half_caught_at_every_pair_width(bn_n):
    assert G.gemm_instance(4096, bn_n, 384, G.OUT_F32)["bn"] == bn_n
    assert _gemm_score(4096, bn_n, 384, "bf16", "identity", "same_w_half") >= REJECT_MARGIN


OUTPUT_MISTAKES = [("truncate", G.OUT_BF16, 1.0), ("truncate", G.OUT_F16, 1.0), ("truncate", G.OUT_BF16_SPLIT, 1.0),
                   ("f16_inf", G.OUT_F16, 3e5), ("split_lo_trunc_hi", G.OUT_BF16_SPLIT, 1.0)]


@pytest.mark.parametrize("out_kind", [G.OUT_BF16, G.OUT_F16, G.OUT_BF16_SPLIT])
@pytest.mark.parametrize("scale_z", [1.0, 3e5])
def test_unmutated_output_model_passes(out_kind, scale_z):
    P = G.make_gemm_operands(3, 128, 64, 64, "fp16", scale_z)
    v = G.simulate_gemm(P, 128, 64, 64, "identity")
    hi, lo = G.simulate_output(v, out_kind)
    assert np.isfinite(hi).all()
    assert G.check_16bit(v, hi, lo, out_kind) == 0


@pytest.mark.parametrize("mistake,out_kind,scale_z", OUTPUT_MISTAKES)
def test_planted_output_mistake_is_rejected(mistake, out_kind, scale_z):
    """The GPU cases check 16-bit outputs exactly: a mistake must change at least REJECT_MARGIN elements."""
    P = G.make_gemm_operands(3, 128, 64, 64, "fp16", scale_z)
    v = G.simulate_gemm(P, 128, 64, 64, "identity")
    hi, lo = G.simulate_output(v, out_kind, mistake)
    assert G.check_16bit(v, hi, lo, out_kind) >= REJECT_MARGIN


# ----------------------------------------------------------------------------------------------------- head
def _head_fast_score(C, mistake=None, w0=1.0, ps=0.7, rows=300, ld_out=None):
    x = G.make_head_logits(C * 3 + rows + 1, rows, C, 1)[0]
    prior, _ = G.make_head_extras(C, C)
    nv4 = G.head_instance(1, False, False, G.BK, C)[1]
    got = G.simulate_head_fast(x, C, nv4, w0, prior, ps, ld_out=C if ld_out is None else ld_out, mistake=mistake)
    y, mag, lse_sum, n_lse = G.head_ref([x], C, [w0], prior=prior, prior_scale=ps)
    return float(G.ratio(got, y, G.head_bound(mag, lse_sum, n_lse, 4 * nv4)).max())


def _head_generic_score(C, n_inputs, pre_normalize, rpl, mistake=None, final_normalize=True, rows=300):
    xs = G.make_head_logits(C * 3 + rows + n_inputs, rows, C, n_inputs)
    prior, rp = G.make_head_extras(C, C)
    rp = rp if rpl else None
    weights = [float(np.float32(v)) for v in np.linspace(0.5, 1.5, n_inputs) / n_inputs] if n_inputs > 1 else [0.9]
    pr = prior if final_normalize else None
    got = G.simulate_head_generic(xs, C, weights, pre_normalize, rp, pr, 0.7, final_normalize, mistake=mistake)
    y, mag, lse_sum, n_lse = G.head_ref(xs, C, weights, pre_normalize, rp, pr, 0.7, final_normalize)
    nv = G.head_instance(n_inputs, pre_normalize, rpl, 1, C)[1]
    return float(G.ratio(got, y, G.head_bound(mag, lse_sum, n_lse, nv)).max())


@pytest.mark.parametrize("C", [1, 125, 126, 509, 510, 1021, 1022, 1917, 1918, 2045])
def test_unmutated_head_fast_model_passes(C):
    assert _head_fast_score(C, w0=0.9) <= 0.5
    assert _head_fast_score(C) <= 0.5


@pytest.mark.parametrize("C,n_inputs,pre_normalize,rpl,final", [(100, 1, False, False, True), (127, 2, False, False, True),
                                                                 (1000, 1, False, True, True), (1001, 5, True, False, True),
                                                                 (999, 2, True, False, False), (1909, 2, False, True, True)])
def test_unmutated_head_generic_model_passes(C, n_inputs, pre_normalize, rpl, final):
    assert _head_generic_score(C, n_inputs, pre_normalize, rpl, final_normalize=final) <= 0.5


@pytest.mark.parametrize("mistake,C,kw", [
    ("ragged_zero", 125, {}), ("ragged_zero", 1917, {}), ("ragged_zero", 509, {}),
    ("ignore_prior_scale", 125, {}), ("ignore_prior_scale", 1918, {}),
    ("ignore_weight", 125, {"w0": 0.9}), ("ignore_weight", 2045, {"w0": 0.9}),
    ("realign_wrong_neighbour", 125, {}), ("realign_wrong_neighbour", 1917, {}), ("realign_wrong_neighbour", 509, {}),
    ("no_max_sub", 126, {}), ("no_max_sub", 1021, {}),
])
def test_planted_head_fast_mistake_is_rejected(mistake, C, kw):
    assert _head_fast_score(C, mistake, **kw) >= REJECT_MARGIN


@pytest.mark.parametrize("mistake,C,n_inputs,pre_normalize,rpl,final", [
    ("rpl_max", 1000, 1, False, True, True), ("rpl_max", 1909, 2, False, True, True),
    ("skip_pre_normalize", 999, 2, True, False, False),
])
def test_planted_head_generic_mistake_is_rejected(mistake, C, n_inputs, pre_normalize, rpl, final):
    """With a final log-softmax a skipped pre_normalize is invisible (it shifts each row by a constant), so that
    mistake is caught on the raw ensemble (final_normalize off), as in the GPU case h-gen32-prenorm-raw."""
    assert _head_generic_score(C, n_inputs, pre_normalize, rpl, mistake, final) >= REJECT_MARGIN


def test_head_data_has_the_hard_rows():
    x = G.make_head_logits(1, 300, 125)[0]
    assert (x.max(axis=1) < 0).sum() >= 20 and (np.abs(x.max(axis=1) - 200) < 1).sum() >= 20


# ----------------------------------------------------------------------------------------------------- instance table
@pytest.mark.parametrize("case", T.GEMM_CASES, ids=[c["id"] for c in T.GEMM_CASES])
def test_gemm_case_labels_match_dispatch(case):
    inst = G.gemm_instance(case["M"], case["N"], case["K"], G.OUT_F32)
    assert inst["kernel"] == ("gemm_bias_act_2sm_kernel" if case["kernel"] == "pair" else "gemm_bias_act_kernel")
    assert inst["bn"] == case["bn"]
    assert case["id"].startswith("g2-" if inst["pair"] else "g1-")


@pytest.mark.parametrize("case", T.HEAD_CASES, ids=[c["id"] for c in T.HEAD_CASES])
def test_head_case_labels_match_dispatch(case):
    for form in case["forms"]:
        inst = T.head_case_instance(case, form)
        assert inst[:len(case["inst"])] == case["inst"], (form, inst)
        if form == "compact" and inst[0] == "fast" and inst[1] < 16:
            assert T.compact_ld16(case) > 128 * inst[1]


def test_fused_cases_cover_every_cluster_size_but_3():
    assert sorted({c["cluster"] for c in T.FUSED_CASES}) == [1, 2, 4, 5, 6, 7, 8]


def test_every_instance_is_reached():
    fast = {T.head_case_instance(c, "rows")[1] for c in T.HEAD_CASES if c["inst"][0] == "fast"}
    gen = {T.head_case_instance(c, "rows")[1:3] for c in T.HEAD_CASES if c["inst"][0] == "generic"}
    assert fast == {1, 4, 8, 15, 16}
    assert gen == {(4, False), (4, True), (32, False), (32, True), (64, False), (64, True)}
    pair_bn = {G.gemm_instance(c["M"], c["N"], c["K"], o)["bn"] for c in T.GEMM_CASES if c["kernel"] == "pair"
               for o in c["outs"] if o == G.OUT_F32}
    assert {128, 160, 192, 224, 256} <= pair_bn
    pair_bn16 = {G.gemm_instance(c["M"], c["N"], c["K"], o)["bn"] for c in T.GEMM_CASES if c["kernel"] == "pair"
                 for o in c["outs"] if o != G.OUT_F32}
    assert {128, 192, 256} <= pair_bn16
    many = [c for c in T.GEMM_CASES if G.gemm_instance(c["M"], c["N"], c["K"], G.OUT_F32)["tiles"] > 148]
    assert {c["kernel"] for c in many} == {"1cta", "pair"}
    rows_grid = {c["inst"][0] for c in T.HEAD_CASES if c["rows"] > G.SM_COUNT * 64}
    assert rows_grid == {"fast", "generic"}
