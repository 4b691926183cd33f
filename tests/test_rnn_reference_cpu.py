"""The step reference of tests/rnn_reference.py is tight enough to catch the mistakes a recurrence kernel makes.

A model of the kernel (``rnn_reference.simulate``) plays the kernel, with one planted mistake at a time; the
teacher-forced comparison used by tests/test_gpu_rnn_kernel.py must reject each by at least REJECT_MARGIN times its
bound, at the seeds and scales of the GPU cases.  The unplanted model must pass, the recurrent term must matter in the
test data, and the reference without rounding must agree with oracle.RecurrentNet.  CPU only."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import rnn_reference as R  # noqa: E402
from oracle import nnam_oracle as O  # noqa: E402

REJECT_MARGIN = 5.0
# ragged lengths, three batches of 16 in one lane (so items run back to back), a shortest utterance of 3 steps
STEPS = [23, 9, 30, 4, 17, 12, 3, 25, 8, 14, 19, 6, 27, 11, 5, 21] * 2 + [16, 10, 7, 29, 13, 18, 24, 15]


def _case(cell, mode, n_dirs=1, flags=0, nb=16, hidden=64, **kw):
    return R.Case(cell, hidden, mode, STEPS, nb, n_dirs=n_dirs, flags=flags, seed=R.case_seed(cell, hidden, nb, mode),
                  **kw)


def _score(case, h_hi, h_lo):
    h_ref, _, slack = R.teacher_forced(case, h_hi, h_lo)
    return float(R.errors(case, h_hi, h_lo, h_ref, slack).max())


CASES = {
    "lstm": dict(cell=R.CELL_LSTM),
    "blstm": dict(cell=R.CELL_LSTM, n_dirs=2),
    "gru": dict(cell=R.CELL_GRU, flags=R.GRU_FLAGS["gru"]),
    "mgrurelu": dict(cell=R.CELL_GRU, flags=R.GRU_FLAGS["mgrurelu"]),
    "wide_gru": dict(cell=R.CELL_GRU, flags=R.GRU_FLAGS["gru"], nb=128),
    "peephole": dict(cell=R.CELL_PEEPHOLE),
}


@pytest.mark.parametrize("mode", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_unmutated_model_passes(name, mode):
    case = _case(mode=mode, **CASES[name])
    h_hi, h_lo, _ = R.simulate(case)
    assert np.isfinite(h_hi).all()
    assert _score(case, h_hi, h_lo) <= 0.5


@pytest.mark.parametrize("mutation,name,mode", [
    ("neighbour_slot", "lstm", "bf16"), ("neighbour_slot", "lstm", "fp16"), ("neighbour_slot", "gru", "bf16"),
    ("neighbour_slot", "lstm", "fp32"),
    ("skip_step", "lstm", "bf16"), ("skip_step", "gru", "fp16"), ("skip_step", "lstm", "fp32"),
    ("bwd_walks_forward", "blstm", "bf16"), ("bwd_walks_forward", "blstm", "fp32"),
    ("state_not_reset", "lstm", "bf16"), ("state_not_reset", "lstm", "fp16"), ("state_not_reset", "peephole", "bf16"),
    ("state_not_reset", "peephole", "fp32"),
    ("u_bias_at_step0", "gru", "bf16"), ("u_bias_at_step0", "mgrurelu", "fp16"), ("u_bias_at_step0", "gru", "fp32"),
    ("u_bias_at_step0", "wide_gru", "bf16"), ("u_bias_at_step0", "wide_gru", "fp16"),
    ("drop_lo", "lstm", "fp32"), ("drop_lo", "gru", "fp32"), ("drop_lo", "peephole", "fp32"),
    ("peep_prev_c", "peephole", "bf16"), ("peep_prev_c", "peephole", "fp16"), ("peep_prev_c", "peephole", "fp32"),
    ("other_type", "lstm", "bf16"), ("other_type", "lstm", "fp16"), ("other_type", "gru", "fp16"),
])
def test_planted_mistake_is_rejected(mutation, name, mode):
    case = _case(mode=mode, **CASES[name])
    h_hi, h_lo, _ = R.simulate(case, mutation)
    assert _score(case, h_hi, h_lo) >= REJECT_MARGIN


@pytest.mark.parametrize("name", ["lstm", "gru"])
def test_c_out_and_gru_state_not_reset_with_carried_state(name):
    """With h0 / c0 the items of a lane must start from THEIR utterances' state, not the previous item's (without h0
    a GRU never reads its initial state: step 0 is h = z * hb)."""
    case = _case(mode="bf16", h0=True, c0=name == "lstm", **CASES[name])
    h_hi, h_lo, c_out = R.simulate(case)
    h_ref, c_ref, slack = R.teacher_forced(case, h_hi, h_lo)
    assert R.errors(case, h_hi, h_lo, h_ref, slack).max() <= 0.5
    if c_ref is not None:
        assert R.c_errors(case, c_out, c_ref).max() <= 0.5
    h_hi, h_lo, _ = R.simulate(case, "state_not_reset")
    assert _score(case, h_hi, h_lo) >= REJECT_MARGIN


@pytest.mark.parametrize("name", sorted(CASES))
def test_recurrent_term_matters(name):
    """||W h|| / ||gx|| >= 0.3 on the rows after step 0: a kernel that dropped the lateral product cannot pass."""
    case = _case(mode="bf16", **CASES[name])
    h_hi, h_lo, _ = R.simulate(case)
    for d in range(case.n_dirs):
        prev = case.prev_row(d)
        rows = prev >= 0
        hp = h_hi[prev[rows], d * case.H:(d + 1) * case.H]
        lat = hp @ case.w_hi[d].T
        used = np.setdiff1d(np.arange(case.lay.G), case.lay.pad_rows())
        ratio = np.linalg.norm(lat[:, used]) / np.linalg.norm(case.gx[d][rows][:, used])
        assert ratio >= 0.3, ratio


def _pack_from_oracle(case, p, x, network):
    """Fill ``case`` (f64 mode) with the oracle's layer-0 parameters in the kernel's packed layout."""
    lay, pre = case.lay, "layer_0/"
    G, H = lay.G, case.H
    rows_x = x[case.row_utt, case.row_step]  # (rows, D) input of every packed row
    w = np.zeros((G, H))
    gx = np.zeros((case.rows, G))
    ub = np.zeros(G)
    if case.cell == R.CELL_GRU:
        names = {"z": "_z", "r": "_r", "c": ""}
        for g, c in lay.cols.items():
            if g == "r" and not lay.reset:
                continue
            w[c] = p[pre + f"U{names[g]}/W"]
            ub[c] = p[pre + f"U{names[g]}/b"]
            gx[:, c] = rows_x @ p[pre + f"W{names[g]}/W"].T.astype(np.float64) + p[pre + f"W{names[g]}/b"]
        if lay.wide_gru:
            gx += ub
    else:
        w[:] = p[pre + "lateral/W"]
        gx[:] = rows_x @ p[pre + "upward/W"].T.astype(np.float64) + p[pre + "upward/b"]
        if case.cell == R.CELL_PEEPHOLE:
            pw = np.zeros((G, H))
            for g in "ifo":
                pw[lay.cols[g]] = p[pre + f"peep_{g}/W"]
            case.pw_hi, case.pw_lo = pw, 0.0
    case.w_hi, case.w_lo, case.gx, case.ub = [w], [0.0], [gx], [ub]


@pytest.mark.parametrize("network,nb", [("lstm", 16), ("peepholelstm", 16), ("gru", 16), ("mgrurelu", 16),
                                        ("mgrurelur", 16), ("gru", 128), ("mgrurelu", 128)])
def test_unrounded_reference_matches_oracle(network, nb):
    """The reference without rounding points against oracle.RecurrentNet (fp32) on one layer: ties the reference's
    packed layouts and cell arithmetic to the existing oracle."""
    H, D = 64, 24
    steps = [12, 7, 1, 9, 4]
    cell = {"lstm": R.CELL_LSTM, "peepholelstm": R.CELL_PEEPHOLE}.get(network, R.CELL_GRU)
    case = R.Case(cell, H, "f64", steps, nb, flags=R.GRU_FLAGS.get(network, 0))
    p = O.init_recurrent(np.random.default_rng(3), network, D, H, 1, 5, bias_scale=0.3)
    x = np.random.default_rng(4).standard_normal((case.n_utt, max(steps), D)).astype(np.float32)
    _pack_from_oracle(case, p, x, network)
    h_hi, _, _ = R.simulate(case)
    h_ref, _, _ = R.teacher_forced(case, h_hi)
    for u in range(case.n_utt):
        net = O.RecurrentNet(p, network, 1)
        for t in range(case.lens[u]):
            net(x[u, t:t + 1])
            want = net.state[0][0][0]
            r = case.row_of[u, t]
            assert np.abs(h_hi[r] - want).max() < 2e-6
            assert np.abs(h_ref[r] - want).max() < 2e-6


def test_rounding_helpers():
    v = np.array([1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, -0.3, 1e-3], np.float32)
    assert np.array_equal(R.bf16(v), torch.from_numpy(v).to(torch.bfloat16).double().numpy())
    assert np.array_equal(R.fp16(v), torch.from_numpy(v).to(torch.float16).double().numpy())
    assert R.ulp16(1.0, "bf16") == 2.0 ** -7 and R.ulp16(1.0, "fp16") == 2.0 ** -10
    assert R.ulp16(0.75, "bf16") == 2.0 ** -8
    hi, lo = R.split(v, "fp32")
    assert np.all(np.abs(hi + lo - v) <= 2.0 ** -16 * np.abs(v))
