"""Frame scoring (nnacousticmodeling_b200.score) without a GPU: target validation happens before any device work,
FrameScore's sums, the rows that are no network output, and the scoring CLI's flags and exit code."""
import importlib
import math

import numpy as np
import pytest

import nnacousticmodeling_b200 as nn
from nnacousticmodeling_b200 import engine, recurrent_engine

# the package exports the functions predict() and score() under the names of their modules
predict_mod = importlib.import_module("nnacousticmodeling_b200.predict")
score_mod = importlib.import_module("nnacousticmodeling_b200.score")


@pytest.fixture
def no_device(monkeypatch):
    """Any attempt to reach the device path fails the test."""
    def boom(*a, **k):
        raise AssertionError("device work started before the targets were validated")
    monkeypatch.setattr(engine, "ff_forward_frames", boom)
    monkeypatch.setattr(recurrent_engine, "forward_utterances", boom)
    monkeypatch.setattr(engine, "get_plan", boom)


def _mlp():
    return nn.get_nn("ff", 2, [64], 39, nn.F.relu, [5])


@pytest.mark.parametrize("targets,match", [
    (np.zeros(9, np.int32), "shape"),                       # one frame short
    (np.zeros(11, np.int64), "shape"),                      # one frame long
    (np.zeros((10, 1), np.int32), "shape"),                 # not 1-D
    (np.zeros(10, np.float32), "integer"),                  # float targets
    (np.zeros(10, np.bool_), "integer"),
    (np.array([0] * 9 + [39], np.int32), r"\[0, 39\)"),     # value == C
    (np.array([0] * 9 + [-2], np.int16), r"\[0, 39\)"),     # value < -1
])
@pytest.mark.parametrize("network", ["ff", "lstm"])
def test_targets_are_checked_before_any_device_work(no_device, targets, match, network):
    x = np.zeros((10, 40), np.float32)
    offsets = np.array([0, 4, 10], np.int32)
    model = _mlp() if network == "ff" else nn.get_nn("lstm", 1, [64], 39, nn.F.relu, [5])
    with pytest.raises(nn.NnamError, match=match):
        nn.score(model, x, offsets, targets, 39, network, 0, 1, 0, None)


def test_valid_targets_reach_the_device_path(no_device):
    x = np.zeros((10, 40), np.float32)
    t = np.array([-1, 0, 38, 5, 5, 5, 0, 1, 2, 3], np.int8)  # any integer dtype
    with pytest.raises(AssertionError, match="device work"):
        nn.score(_mlp(), x, None, t, 39, "ff", 0, 1, 0, None)


def test_gpu_below_zero_is_rejected():
    with pytest.raises(nn.NnamError, match="CPU"):
        nn.score(_mlp(), np.zeros((3, 40), np.float32), None, np.zeros(3, np.int32), 39, "ff", -1, 1, 0, None)


def test_frame_score_sums():
    t = np.array([3, -1, 2, 2, 0, 1], np.int32)
    pred = np.array([3, 0, 1, 2, -1, 1], np.int32)   # frame 4: no network output
    nll = np.array([0.5, 0.0, 2.0, 0.25, 0.0, 1.0], np.float32)
    s = nn.FrameScore(t, nll, pred)
    assert (s.frames, s.scored, s.correct) == (6, 4, 3)
    assert s.loss_sum == pytest.approx(3.75) and isinstance(s.loss_sum, float)
    assert s.loss == pytest.approx(3.75 / 4) and s.accuracy == pytest.approx(0.75)
    d = s.summary()
    assert d == {"frames": 6, "scored": 4, "correct": 3, "loss_sum": s.loss_sum, "loss": s.loss, "accuracy": 0.75}
    pooled = nn.FrameScore.pooled([s, s])
    assert (pooled.frames, pooled.scored, pooled.correct) == (12, 8, 6)
    assert pooled.loss == pytest.approx(s.loss) and pooled.accuracy == pytest.approx(s.accuracy)


def test_loss_sum_is_float64():
    n = 1 << 20
    nll = np.full(n, 1.0 + 2 ** -20, np.float32)  # a float32 running sum would lose the low bits
    s = nn.FrameScore(np.zeros(n, np.int32), nll, np.zeros(n, np.int32))
    assert s.loss_sum == pytest.approx(n * (1.0 + 2 ** -20), rel=1e-12)


@pytest.mark.parametrize("targets", [np.full(4, -1, np.int32), np.zeros(0, np.int32)])
def test_nothing_scored_gives_nan(targets):
    n = len(targets)
    s = nn.FrameScore(targets, np.zeros(n, np.float32), np.zeros(n, np.int32))
    assert s.scored == 0 and math.isnan(s.loss) and math.isnan(s.accuracy)
    assert s.summary()["loss"] is None and s.summary()["accuracy"] is None


def test_empty_set_scores_without_a_device(no_device):
    s = nn.score(_mlp(), np.zeros((0, 40), np.float32), None, np.zeros(0, np.int64), 39, "ff", 0, 1, 0, None)
    assert s.frames == 0 and s.scored == 0 and math.isnan(s.loss)


@pytest.mark.parametrize("td", [0, 1, 5, 200])
def test_rows_without_network_output_are_not_scored(td):
    """Quirk Q4: with timedelay > 0 the last min(td, len_u) frames of every utterance are rows predict() leaves zero;
    the kernels mark them pred = -1, and FrameScore leaves exactly those out."""
    rng = np.random.default_rng(td)
    lens = rng.integers(1, 40, 50)
    lens[:3] = [1, 3, 5]
    off = np.concatenate([[0], np.cumsum(lens)])
    n = int(off[-1])
    pred = rng.integers(0, 39, n).astype(np.int32)
    for u in range(len(lens)):
        pred[max(off[u + 1] - td, off[u]):off[u + 1]] = -1
    t = rng.integers(0, 39, n).astype(np.int32)
    s = nn.FrameScore(t, np.zeros(n, np.float32), pred)
    assert s.scored == n - int(np.minimum(td, lens).sum())


def test_score_cli_shares_the_predict_flags():
    p = predict_mod.fold_arg_parser("x")
    a = p.parse_args([])
    assert (a.fold_data_pattern, a.fold_offset_pattern, a.fold_network_pattern, a.network, a.gpu, a.timedelay) == \
        ("data_{}.npy", "offsets_{}.npy", "fold_{}.npz", "ff", [0], 0)
    with pytest.raises(SystemExit):
        p.parse_args(["--fold-target-pattern", "t_{}.npy"])  # scoring flag only


def test_score_cli_without_fold_models_exits_2(tmp_path, capsys):
    with pytest.raises(SystemExit) as e:
        score_mod.main(["--fold-model-dir", tmp_path, "--fold-data-dir", tmp_path, "--fold-target-pattern",
                        "t_{}.npy", "--json", tmp_path / "s.json", "--network", "lstm", "--units", "64"])
    assert e.value.code == 2
    assert "No fold networks found" in capsys.readouterr().out
    assert not (tmp_path / "s.json").exists()
    assert sorted(p.name for p in tmp_path.iterdir()) == []
