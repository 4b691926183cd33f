"""bench.py --dump-outputs: a fixed sample of the timed path's output, the same on every run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from oracle import nnam_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True,
                          text=True, timeout=900)


def test_dump_rows_are_a_fixed_sample_within_64_mb():
    n = bench.TRAIN_FRAMES
    rows = bench.dump_rows(n)
    assert np.array_equal(rows, bench.dump_rows(n))
    assert len(rows) == bench.DUMP_ROWS and np.all(np.diff(rows) > 0) and 0 <= rows[0] and rows[-1] < n
    assert bench.DUMP_ROWS * bench.N_CLASSES * 4 <= 64 << 20
    assert np.array_equal(bench.dump_rows(100), np.arange(100))


def test_bench_rejects_zero_steps_and_a_dump_of_the_reference_arm(tmp_path):
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        res = _bench(*args)
        assert res.returncode == 2 and "error" in res.stderr, (args, res.stderr[-2000:])
    assert not os.listdir(tmp_path)


@pytest.mark.gpu
def test_dump_outputs_repeat_and_match_the_oracle(tmp_path):
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import nnacousticmodeling_b200 as nn
    from nnacousticmodeling_b200 import synth
    args = ["--workload", "cfg1", "--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--no-cli", "--no-e2e",
            "--extra", ""]
    dumps = []
    for k in range(2):
        res = _bench(*args, "--dump-outputs", str(tmp_path / str(k)))
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 2
        assert os.listdir(tmp_path / str(k)) == ["log_likelihoods.npy"]
        dumps.append(np.load(tmp_path / str(k) / "log_likelihoods.npy"))
    y = dumps[0]
    assert np.array_equal(y, dumps[1])
    assert y.dtype == np.float32 and y.shape == (bench.DUMP_ROWS, bench.N_CLASSES)
    # the dumped rows are the rows dump_rows names: a few of them against the fp32 oracle (fp16 mode tolerance)
    w = bench.WORKLOADS["cfg1"]
    x, _, _ = synth.synth_set(1234, w["utts"], 40, 0, total=w["frames"])
    rows = bench.dump_rows(len(x))
    m = nn.get_nn("ff", w["layers"], [w["units"]], bench.N_CLASSES, nn.F.relu, [5]).init_params(
        440, np.random.default_rng(4321))
    ft = O.load_kaldi_feature_transform(os.path.join(ROOT, "tests", "golden", "final.feature_transform"))
    # sorted: prepare_batch sorts the frame indices it is given, as the reference does
    pick = np.unique(np.concatenate([np.arange(4), np.arange(4, len(rows) - 4, 997), np.arange(len(rows) - 4, len(rows))]))
    feats = O.apply_kaldi_feature_transform(O.prepare_batch(x, rows[pick], 11), ft)
    want = O.log_softmax(O.mlp_forward(m.params, feats, w["layers"]))
    assert np.abs(y[pick] - want).max() < 5e-2
