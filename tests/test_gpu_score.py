"""Frame scoring on the device (nnam_head_score, nnam_linear_logsoftmax_score, score()) against the row outputs it
replaces, bit for bit, and against the NumPy oracle.  -m gpu."""
import importlib
import json

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import nnam_oracle as O  # noqa: E402

SENT_NLL, SENT_PRED = 12345.0, -7  # what rows nobody writes keep


@pytest.fixture(scope="module")
def nn():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import nnacousticmodeling_b200 as _nn
    import nnacousticmodeling_b200.synth  # noqa: F401  (nn.synth)
    return _nn


@pytest.fixture(scope="module")
def ops(nn):
    from nnacousticmodeling_b200 import ops as _ops
    return _ops


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _check_rows(out, targets, nll, pred, written, zero_rows):
    """nll / pred of the scoring kernel against the rows `out` of the row kernel, for output rows `written` (network
    outputs) and `zero_rows` (zero-fill entries); every other row keeps its sentinels."""
    written = np.asarray(sorted(written), dtype=np.int64)
    t = targets[written]
    want_nll = np.where(t >= 0, -out[written, np.maximum(t, 0)], np.float32(0))
    assert np.array_equal(nll[written], want_nll)
    assert np.array_equal(pred[written], out[written].argmax(axis=1))
    zero_rows = np.asarray(sorted(zero_rows), dtype=np.int64)
    assert np.all(nll[zero_rows] == 0) and np.all(pred[zero_rows] == -1)
    rest = np.setdiff1d(np.arange(len(nll)), np.concatenate([written, zero_rows]))
    assert np.all(nll[rest] == SENT_NLL) and np.all(pred[rest] == SENT_PRED)


def _row_map(rng, rows, n_out):
    """A permutation of the logits rows onto output rows [0, rows) with one dropped row and zero-fill entries for the
    output rows `rows` and `rows + 1`; output rows rows + 2 .. n_out - 1 have no source."""
    rm = rng.permutation(rows).astype(np.int32)
    if rows >= 3:
        rm[0], rm[1], rm[2] = -1, -2 - rows, -2 - (rows + 1)
    written = rm[rm >= 0]
    zero = [-2 - int(v) for v in rm if v <= -2]
    return rm, written, zero


# ------------------------------------------------------------------------------------------ K4 scoring head
@pytest.mark.parametrize("c", [39, 1909, 2048])
@pytest.mark.parametrize("case", ["one", "one_unaligned", "three", "three_prenorm", "rpl", "prior"])
@pytest.mark.parametrize("mapped", [False, True])
def test_head_score_form_matches_head_scatter(ops, c, case, mapped):
    rng = np.random.default_rng(c + len(case))
    rows = 333
    k = 3 if case.startswith("three") else 1
    ld = c if (case == "one_unaligned" and c % 4) else ops.round_up(c, 16)  # ld % 4 != 0: the generic kernel
    logits = [_t(3 * rng.standard_normal((rows, ld)).astype(np.float32)) for _ in range(k)]
    kw = dict(rows=rows, weights=[0.5, 0.3, 0.2] if k == 3 else None, pre_normalize=case == "three_prenorm")
    if case == "rpl":
        kw["rpl"] = (_t(0.3 * rng.standard_normal(c).astype(np.float32)), _t(rng.standard_normal(c).astype(np.float32)),
                     _t((-20 + 5 * rng.random(c)).astype(np.float32)))
    if case in ("rpl", "prior"):
        kw["prior"], kw["prior_scale"] = _t(np.log(rng.dirichlet(np.ones(c))).astype(np.float32)), 0.7
    if mapped:
        n_out = rows + 4
        rm, written, zero = _row_map(rng, rows, n_out)
        kw["out_row_map"] = _t(rm)
    else:
        n_out, written, zero = rows, np.arange(rows), []
    targets = rng.integers(-1, c, n_out).astype(np.int32)
    targets[:4] = [0, c - 1, -1, c // 2]
    out = torch.full((n_out, c), 7.0, device="cuda")
    ops.head(logits, c, out=out, **kw)
    nll = torch.full((n_out,), SENT_NLL, device="cuda")
    pred = torch.full((n_out,), SENT_PRED, dtype=torch.int32, device="cuda")
    ops.head(logits, c, score=(_t(targets), nll, pred), **kw)
    torch.cuda.synchronize()
    _check_rows(out.cpu().numpy(), targets, nll.cpu().numpy(), pred.cpu().numpy(), written, zero)


# ------------------------------------------------------------------------------------------ fused output layer
MODES = {"fp16": (3, 1, 1), "bf16": (0, 0, 1), "bf16x3": (1, 0, 3)}  # convert kind, elem, nsplit


def _operands(ops, a, w, mode):
    kind, elem, nsplit = MODES[mode]
    a_hi, a_lo = ops.convert_f32(_t(a), kind)
    w_hi, w_lo = ops.convert_f32(_t(w), kind)
    return (a_hi, a_lo, w_hi, w_lo), dict(nsplit=nsplit, elem=elem)


def _tile_edge_targets(n, count):
    cols = [t for t in (0, 127, 128, 255, 256, 511, 512, 1023, 1024, 1500, 1791, 1792, n - 1, -1) if t < n]
    return np.resize(np.asarray(cols, np.int32), count)


@pytest.mark.parametrize("k", [140, 512, 1024])
@pytest.mark.parametrize("n", [512, 1909, 2048])
@pytest.mark.parametrize("m", [1, 127, 4173])
def test_fused_score_matches_fused_rows(ops, k, n, m):
    rng = np.random.default_rng(k * n + m)
    a = rng.standard_normal((m, k)).astype(np.float32)
    w = (3 * rng.standard_normal((n, k)) / np.sqrt(k)).astype(np.float32)
    b = _t(rng.standard_normal(n).astype(np.float32))
    prior = _t(np.log(rng.dirichlet(np.ones(n))).astype(np.float32))
    for mode in MODES:
        opnds, kw = _operands(ops, a, w, mode)
        for with_extras in (False, True):
            ekw = dict(kw)
            if with_extras:
                n_out = m + 2
                rm, written, zero = _row_map(rng, m, n_out)
                ekw.update(prior=prior, prior_scale=0.9, out_row_map=_t(rm))
            else:
                n_out, written, zero = m, np.arange(m), []
            targets = _tile_edge_targets(n, n_out)
            rng.shuffle(targets)
            out = torch.full((n_out, n), 7.0, device="cuda")
            ops.linear_logsoftmax(*opnds, b, m, n, k, out=out, **ekw)
            nll = torch.full((n_out,), SENT_NLL, device="cuda")
            pred = torch.full((n_out,), SENT_PRED, dtype=torch.int32, device="cuda")
            ops.linear_logsoftmax(*opnds, b, m, n, k, score=(_t(targets), nll, pred), **ekw)
            torch.cuda.synchronize()
            _check_rows(out.cpu().numpy(), targets, nll.cpu().numpy(), pred.cpu().numpy(), written, zero)


@pytest.mark.parametrize("n", [1909, 2048])
@pytest.mark.parametrize("mode", list(MODES))
def test_fused_score_breaks_an_exact_tie_across_ctas_to_the_lower_column(ops, n, mode):
    """Columns 10 (cluster rank 0) and 1500 (rank 5) have the same W row and bias and dominate every row: the written
    values tie exactly, and pred must be the lower column, as np.argmax has it."""
    rng = np.random.default_rng(n)
    m, k = 1000, 512
    a = rng.standard_normal((m, k)).astype(np.float32)
    w = (rng.standard_normal((n, k)) / np.sqrt(k)).astype(np.float32)
    w[1500] = w[10]
    bias = rng.standard_normal(n).astype(np.float32)
    bias[10] = bias[1500] = 60.0
    opnds, kw = _operands(ops, a, w, mode)
    out = torch.empty((m, n), device="cuda")
    ops.linear_logsoftmax(*opnds, _t(bias), m, n, k, out=out, **kw)
    targets = np.full(m, 1500, np.int32)
    nll = torch.empty((m,), device="cuda")
    pred = torch.empty((m,), dtype=torch.int32, device="cuda")
    ops.linear_logsoftmax(*opnds, _t(bias), m, n, k, score=(_t(targets), nll, pred), **kw)
    o = out.cpu().numpy()
    assert np.array_equal(o[:, 10], o[:, 1500])
    assert np.all(pred.cpu().numpy() == 10)
    assert np.array_equal(nll.cpu().numpy(), -o[:, 1500])


# ------------------------------------------------------------------------------------------ score() vs predict()
def _q4_rows(n, offsets, td, fix):
    q4 = np.zeros(n, bool)
    if td and not fix and offsets is not None:
        for u in range(len(offsets) - 1):
            q4[max(int(offsets[u + 1]) - td, int(offsets[u])):int(offsets[u + 1])] = True
    return q4


def _targets(rng, n, c):
    t = rng.integers(0, c, n).astype(np.int32)
    t[rng.random(n) < 0.1] = -1
    return t


def _check_contract(s, out, targets, q4):
    """nll[f] == -out[f, t_f] bit for bit and pred[f] == argmax out[f] on every network-output row; Q4 rows are pred -1,
    nll 0; rows with target -1 have nll 0."""
    net = ~q4
    assert np.all(s.pred[q4] == -1) and np.all(s.nll[q4] == 0)
    assert np.array_equal(s.pred[net], out[net].argmax(axis=1))
    sc = net & (targets >= 0)
    assert np.array_equal(s.nll[sc], -out[sc, targets[sc]])
    assert np.all(s.nll[net & (targets < 0)] == 0)
    assert s.scored == int(sc.sum()) and s.frames == len(targets)
    assert s.correct == int((out[sc].argmax(axis=1) == targets[sc]).sum())
    assert s.loss_sum == float((-out[sc, targets[sc]]).astype(np.float64).sum())


def _case(nn, case, precision, rng):
    """(models, x, offsets, C, network, winlen, timedelay, kwargs) of one path."""
    def net(network, layers, units, c, in_size, seed, ksize=(5,)):
        m = nn.get_nn(network, layers, list(units), c, nn.F.relu, list(ksize))
        m.init_params(in_size, np.random.default_rng(seed))
        for kk in m.params:  # non-zero biases
            if kk.endswith("/b"):
                m.params[kk] = m.params[kk] + 0.1 * np.random.default_rng(seed + 1).standard_normal(
                    m.params[kk].shape).astype(np.float32)
        m._version += 1
        m.precision = precision
        return m
    x, off, iv = nn.synth.synth_set(int(rng.integers(1 << 30)), 40, 40, 100)
    if case == "mlp_fused":
        return net("ff", 3, [512], 1909, 540, 1), x, None, 1909, "ff", 11, 0, dict(ivectors=iv)
    if case == "mlp_wide":
        return net("ff", 2, [2048], 1909, 540, 2), x, None, 1909, "ff", 11, 0, dict(ivectors=iv)
    if case == "tdnn":
        return net("tdnn", 4, [128] * 4, 39, 680, 3, (5, 5, 5, 5)), x, None, 39, "tdnn", 17, 0, {}
    if case.startswith("lstm"):
        # enough utterances for the utterance-subset split of a host output (>= 256 utterances, >= 150k frames)
        x, off, _ = nn.synth.synth_set(int(rng.integers(1 << 30)), 560, 40, 0)
        return (net("lstm", 2, [512], 1909, 40, 4), x, off, 1909, "lstm", 1, 5,
                dict(fix_timedelay_tail=case == "lstm_fix"))
    if case == "blstm_ivec":
        return net("blstm", 2, [256], 1909, 140, 5), x, off, 1909, "blstm", 1, 0, dict(ivectors=iv)
    if case == "mgru":
        return net("mgrurelur", 2, [256], 1909, 40, 6), x, off, 1909, "mgrurelur", 1, 3, {}
    if case == "peephole":
        # H = 768: the lateral and peephole blocks fit no persistent instance in either mode -> the time-step engine
        return net("peepholelstm", 1, [768], 39, 40, 7), x[:off[6]], off[:7], 39, "peepholelstm", 1, 2, {}
    if case == "dev_ensemble":
        folds = [net("ff", 3, [512], 1909, 540, 10 + f) for f in range(3)]
        return folds, x, None, 1909, "ff", 11, 0, dict(ivectors=iv, head=nn.HeadSpec(pre_normalize=True))
    if case == "rpl":
        master, folds = net("ff", 2, [512], 1909, 440, 20), [net("ff", 2, [512], 1909, 440, 21 + f) for f in range(2)]
        rpl = nn.RPL4(1909)
        rpl.load_params({"W": 0.2 * rng.standard_normal(1909), "b": rng.standard_normal(1909),
                         "lb": -20 + 4 * rng.random(1909)})
        model = nn.NNWithRPL(master, folds, rpl)
        ap = np.log(rng.dirichlet(np.ones(1909))).astype(np.float32)
        feats = rng.standard_normal((len(x), 440)).astype(np.float32)
        return model.members, feats, None, 1909, "ff", 1, 0, dict(head=model.head_spec(ap), presliced=True)
    raise AssertionError(case)


CASES = ["mlp_fused", "mlp_wide", "tdnn", "lstm", "lstm_fix", "blstm_ivec", "mgru", "peephole", "dev_ensemble", "rpl"]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_score_matches_predict_bit_for_bit(nn, monkeypatch, case, precision):
    from nnacousticmodeling_b200 import engine, recurrent_engine
    if case.startswith("lstm") and precision == "fp16":
        monkeypatch.setenv("NNAM_RNN_MIXED", "force")  # the long utterances in their own launch
    rng = np.random.default_rng(len(case) + (precision == "fp16"))
    models, x, off, c, network, winlen, td, kw = _case(nn, case, precision, rng)
    targets = _targets(rng, len(x), c)
    out = nn.predict(models, x, off, c, network, 0, winlen, td, None, progress=False, transfer="f32", **kw)
    s = nn.score(models, x, off, targets, c, network, 0, winlen, td, None, **kw)
    _check_contract(s, out, targets, _q4_rows(len(x), off, td, kw.get("fix_timedelay_tail", False)))
    first = models[0] if isinstance(models, list) else models
    plan = next(iter(first._plans.values()))
    if case == "mlp_fused":
        assert engine.fused_head_ok([first], engine.HeadSpec(), plan.out.k)
    if case == "mlp_wide":
        assert not engine.fused_head_ok([first], engine.HeadSpec(), plan.out.k)
    if case == "peephole":
        assert not plan.peep_persistent  # the time-step engine
    if case.startswith("lstm") and precision == "fp16":
        assert any(isinstance(v[0], recurrent_engine.MixedSchedule) for v in plan._sched_cache.values())


# ------------------------------------------------------------------------------------------ oracle
def test_score_matches_the_oracle_cfg1_shape(nn):
    rng = np.random.default_rng(11)
    x, _, _ = nn.synth.synth_set(5, 60, 40, 0)
    p = O.init_mlp(np.random.default_rng(1), 440, 1024, 6, 1909)
    m = nn.get_nn("ff", 6, [1024], 1909, nn.F.relu, [5])
    m.load_params(p)
    m.precision = "fp32"
    want = O.log_softmax(O.mlp_forward(p, O.splicing(x, range(-5, 6)), 6))
    _check_oracle(nn, m, x, None, "ff", 11, 0, want, rng)


def test_score_matches_the_oracle_cfg3_shape(nn):
    rng = np.random.default_rng(12)
    x, off, _ = nn.synth.synth_set(6, 24, 40, 0)
    p = O.init_recurrent(np.random.default_rng(2), "lstm", 40, 512, 4, 1909)
    m = nn.get_nn("lstm", 4, [512], 1909, nn.F.relu, [5])
    m.load_params(p)
    m.precision = "fp32"
    want = O.predict(O.RecurrentNet(p, "lstm", 4), x, off, "lstm", 1, 5, None)
    _check_oracle(nn, m, x, off, "lstm", 1, 5, want, rng)


def _check_oracle(nn, m, x, off, network, winlen, td, want, rng):
    n = len(x)
    t = _targets(rng, n, 1909)
    s = nn.score(m, x, off, t, 1909, network, 0, winlen, td, None)
    sc = (t >= 0) & ~_q4_rows(n, off, td, False)
    assert s.scored == int(sc.sum())
    ce = float(-want[sc, t[sc]].astype(np.float64).mean())
    acc = float((want[sc].argmax(axis=1) == t[sc]).mean())
    assert abs(s.loss - ce) < 1e-3
    got = nn.predict(m, x, off, 1909, network, 0, winlen, td, None, progress=False, transfer="f32")
    differ = float((got[sc].argmax(axis=1) != want[sc].argmax(axis=1)).mean())
    assert abs(s.accuracy - acc) <= differ + 1e-12


# ------------------------------------------------------------------------------------------ two GPUs
@pytest.mark.parametrize("network", ["ff", "lstm"])
def test_two_gpus_score_like_one(nn, network):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    rng = np.random.default_rng(3)
    x, off, _ = nn.synth.synth_set(9, 50, 40, 0)
    m = nn.get_nn(network, 2, [512], 1909, nn.F.relu, [5])
    m.init_params(440 if network == "ff" else 40, np.random.default_rng(4))
    m.precision = "fp16"
    t = _targets(rng, len(x), 1909)
    args = (x, off if network == "lstm" else None, t, 1909, network)
    tail = (11 if network == "ff" else 1, 5 if network == "lstm" else 0, None)
    a = nn.score(m, *args, 0, *tail)
    b = nn.score(m, *args, [0, 1], *tail)
    assert np.array_equal(a.nll, b.nll) and np.array_equal(a.pred, b.pred)


# ------------------------------------------------------------------------------------------ CLI
def test_score_cli_matches_predict_cli(nn, tmp_path, capsys):
    predict_mod = importlib.import_module("nnacousticmodeling_b200.predict")
    score_mod = importlib.import_module("nnacousticmodeling_b200.score")
    for network, extra, in_size, ivd in (("ff", ["--splice", "5", "--layers", "2", "--units", "256"], 440, 0),
                                         ("lstm", ["--layers", "2", "--units", "128", "--timedelay", "5",
                                                   "--ivector-dir", str(tmp_path)], 140, 100)):
        d, md, od = tmp_path / network / "data", tmp_path / network / "models", tmp_path / network / "out"
        for p in (d, md):
            p.mkdir(parents=True)
        rng = np.random.default_rng(len(network))
        for k in range(2):
            x, off, iv = nn.synth.synth_set(40 + k, 12, 40, ivd)
            np.save(d / f"data_{k}.npy", x)
            np.save(d / f"offsets_{k}.npy", off)
            if ivd:
                np.save(d / f"ivectors_{k}.npy", iv)
            np.save(d / f"targets_{k}.npy", _targets(rng, len(x), 39).astype(np.int64))
            m = nn.get_nn(network, 2, [256 if network == "ff" else 128], 39, nn.F.relu, [5])
            m.init_params(in_size, np.random.default_rng(100 + k))
            nn.save_npz(str(md / f"fold_{k}.npz"), nn.Classifier(m))
        flags = ["--network", network, "--fold-data-dir", d, "--fold-model-dir", md, "--fold-output-dir", od,
                 "--precision", "fp32", "--no-progress"] + extra
        predict_mod.main(flags)
        js = tmp_path / network / "score.json"
        score_mod.main(flags + ["--json", js])
        doc = json.loads(js.read_text())
        assert sorted(p.name for p in od.iterdir()) == ["data_0.npy", "data_1.npy"]  # scoring wrote no .npy
        tot = dict(frames=0, scored=0, correct=0, loss_sum=0.0)
        for k in range(2):
            y = np.load(od / f"data_{k}.npy")
            t = np.load(d / f"targets_{k}.npy")
            off = np.load(d / f"offsets_{k}.npy")
            sc = (t >= 0) & ~_q4_rows(len(y), off if network == "lstm" else None, 5 if network == "lstm" else 0, False)
            want = dict(frames=len(y), scored=int(sc.sum()), correct=int((y[sc].argmax(axis=1) == t[sc]).sum()),
                        loss_sum=float((-y[sc, t[sc]]).astype(np.float64).sum()))
            got = doc["folds"][k]
            assert got["fold"] == k
            assert {kk: got[kk] for kk in want} == want
            assert got["loss"] == pytest.approx(want["loss_sum"] / want["scored"], rel=1e-12)
            for kk in tot:
                tot[kk] += want[kk]
        pooled = doc["pooled"]
        assert {kk: pooled[kk] for kk in ("frames", "scored", "correct")} == {kk: tot[kk] for kk in ("frames", "scored", "correct")}
        assert pooled["loss_sum"] == pytest.approx(tot["loss_sum"], rel=1e-12)
        lines = capsys.readouterr().out.splitlines()
        assert any(line.startswith("fold 1: frames") for line in lines) and lines[-1].startswith("pooled: frames")


# ------------------------------------------------------------------------------------------ redzones
def test_score_keeps_inside_its_workspaces(nn, monkeypatch):
    monkeypatch.setenv("NNAM_REDZONE", "16384")
    rng = np.random.default_rng(8)
    x, off, iv = nn.synth.synth_set(13, 30, 40, 100)
    for network, in_size, winlen, td, ivec in (("ff", 540, 11, 0, iv), ("lstm", 40, 1, 3, None)):
        m = nn.get_nn(network, 2, [512], 1909, nn.F.relu, [5])
        m.init_params(in_size, np.random.default_rng(9))
        m.precision = "bf16"
        t = _targets(rng, len(x), 1909)
        s = nn.score(m, x, off if network == "lstm" else None, t, 1909, network, 0, winlen, td, None, ivectors=ivec)
        assert s.scored > 0 and np.isfinite(s.loss)
        n = sum(plan.ws.check_redzones() for plan in m._plans.values())
        assert n > 0, "no guarded workspace buffers were checked"
        names = set().union(*(plan.ws._raw for plan in m._plans.values()))
        assert {"ff.nll", "ff.pred", "ff.targets"} <= names or {"rnn.nll", "rnn.pred", "rnn.targets"} <= names
