"""K3 row by row: every recurrence kernel instance the dispatch of ``nnam_rnn_seq`` reaches, against the teacher-forced
float64 step reference of tests/rnn_reference.py.  -m gpu.

Each case builds its descriptor from its own packing (rnn_reference.build_desc) with the streams and groups that
``nnam_rnn_plan`` reports, runs one ``nnam_rnn_seq`` launch and checks every packed row of h (and c_out) against a
one-step bound, plus the NaN pre-fill and the sentinels around h.

Instances reached on a 148-SM B200 (rnn_pick_cfg in csrc/recurrent.cu: the first row of NNAM_RNN_INSTANCES /
NNAM_PEEP_INSTANCES whose slots and precision match, whose KBT is 0 or H / 64, whose shared-memory footprint
(rnn_smem_bytes) is <= 227 KB and whose 4H / m_rows CTAs fit; rnn_mc_groups for the multicast kernel;
rnn_wide_applies / rnn_wide_gru_applies at 128 slots).  Instance = (m_rows, slots, nsplit, KBT, streams, warps).

  kernel                               cells       H      slots  mode        groups  case ids
  X(128,16,1,8,4,4)    (#0)            LSTM, GRU   512    16     bf16/fp16   9       lstm-512-16, gru-512-16
  X(128,32,1,8,1,16)   (#1)            GRU         512    32     bf16/fp16   9       mgrurelu-512-32
                                       LSTM        512    32     16-bit with carried state, or NNAM_RNN_MC=0
  X(128,64,1,8,1,16)   (#2)            LSTM, GRU   512    64     bf16/fp16   9       lstm-512-64, mgrurelur-512-64
  X(64,16,3,8,2,8)     (#3)            LSTM, GRU   512    16     fp32        4       lstm-512-16-fp32, gru-512-16-fp32
  X(64,32,3,8,1,8)     (#4)            LSTM, GRU   512    32     fp32        4       lstm-512-32-fp32, mgrurelu-512-32-fp32
  X(128,16,1,0,4,4)    (#5)            LSTM, GRU   64-448 16     bf16/fp16   74-10   lstm-64-16, gru-64-16, edges
  X(128,32,1,0,2,8)    (#6)            LSTM, GRU   64-448 32     bf16/fp16   74-10   lstm-64-32, mgrurelu-192-32
                                       LSTM        256    32     NNAM_RNN_MC=0 (child process)
  X(128,64,1,0,1,8)    (#7)            LSTM, GRU   64-448 64     bf16/fp16   74-10   lstm-192-64, mgrurelur-64-64
  X(128,32,1,0,1,8)    (#8)            LSTM, GRU   576-640 32    bf16/fp16   8-7     lstm-640-32, gru-640-32
                                       LSTM        256    32     16-bit with carried state (carried-lstm-256-32-*)
  X(64,16,1,0,2,8)     (#9)            LSTM, GRU   576-1088 16   bf16/fp16   4-2     lstm-1024-16, gru-1024-16
  X(64,32,1,0,1,8)     (#10)           LSTM, GRU   704-1152 32   bf16/fp16   3-2     lstm-1024-32, mgrurelu-1024-32
  X(64,16,1,0,1,8)     (#11)           LSTM, GRU   1152-1344 16  bf16/fp16   2-1     lstm-1152-16, gru-1152-16
  X(128,16,3,0,2,8)    (#12)           LSTM, GRU   64-320 16     fp32        74-14   lstm-192-16-fp32, gru-64-16-fp32
  X(128,32,3,0,1,8)    (#13)           LSTM, GRU   64-320 32     fp32        74-14   lstm-192-32-fp32, mgrurelur-256-32-fp32
  X(64,16,3,0,2,8)     (#14)           LSTM, GRU   384-448 16    fp32        6-5     lstm-384-16-fp32, gru-384-16-fp32
  X(64,32,3,0,1,8)     (#15)           LSTM, GRU   384-448 32    fp32        6-5     lstm-384-32-fp32, mgrurelu-448-32-fp32
  X(64,16,3,0,1,8)     (#16)           LSTM, GRU   576-640 16    fp32        4-3     lstm-576-16-fp32, gru-576-16-fp32
  peephole X(64,32,1,8,1,8)   (P0)     PEEPHOLE    512    32     bf16/fp16   4       peep-512-32
  peephole X(64,32,1,0,1,8)   (P1)     PEEPHOLE    64-576 32     bf16/fp16   37-4    peep-128-32
  peephole X(64,16,1,0,1,8)   (P2)     PEEPHOLE    64-640 16     bf16/fp16   37-3    peep-64-16
  peephole X(64,32,3,0,1,8)   (P3)     PEEPHOLE    64-256 32     fp32        37-9    peep-128-32-fp32
  peephole X(64,16,3,0,1,8)   (P4)     PEEPHOLE    64-320 16     fp32        37-7    peep-320-16-fp32
  multicast rnn_seq_mc_kernel<32,4>    LSTM        256    32     bf16/fp16   mc      lstm-256-32, blstm-256-32
  multicast rnn_seq_mc_kernel<32,8>    LSTM        512    32     bf16/fp16   mc      lstm-512-32, mc edges
  wide lstm_seq_wide2_kernel<KBT,2,8>  LSTM        any    128    bf16/fp16           lstm-512-128, blstm-128-128
  wide lstm_seq_wide_kernel<KBT>       LSTM        any    128    NNAM_RNN_WIDE_STREAMS=1 (child process)
  wide lstm_seq_wide2_kernel<KBT,3,4>  LSTM        any    128    NNAM_RNN_WIDE_STREAMS=3 (child process)
  wide GRU gru_seq_wide2_kernel<3,KBT> gru, mgrurelur 128 slots  bf16/fp16           gru-512-128, bgru-192-128
  wide GRU gru_seq_wide2_kernel<2,KBT> mgrurelu    128 slots     bf16/fp16           mgrurelu-256-128

Prefix tables (base[]) are mirrored in shared memory up to BASE_SMEM steps: 2048 (S < 4 instances, multicast, wide
single-stream), 1024 (S = 4, wide two-stream, wide GRU), 768 (wide three-stream); the edge cases run batches of exactly
BASE_SMEM and BASE_SMEM + 1 steps.

The worst error of every case is printed (run with -s to see it) as ``K3 <case> <mode> worst=<e> bound=<b>
of-allowance=<a>``: e in ulps of the 16-bit type in the 16-bit modes, an absolute error (relative above |h| = 1) in the
fp32-accurate mode; a = the worst ratio to the per-element allowance (bound plus the operand-rounding slack of
rnn_reference.errors), which must not exceed 1."""
import os
import subprocess
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

import rnn_reference as R  # noqa: E402

LSTM, GRU, PEEP = R.CELL_LSTM, R.CELL_GRU, R.CELL_PEEPHOLE


@pytest.fixture(scope="module")
def nn():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import nnacousticmodeling_b200 as _nn
    return _nn


def ragged(n_utt, lo, hi, seed):
    return np.random.default_rng(seed).integers(lo, hi + 1, size=n_utt).tolist()


def run_case(name, cell, H, mode, steps, nb, n_dirs=1, flags=0, h0=False, c0=False, max_groups=None, pad_cols=16):
    """One nnam_rnn_seq launch checked row by row; returns the worst error in units of the bound."""
    from nnacousticmodeling_b200 import ops
    from nnacousticmodeling_b200.recurrent_engine import Schedule
    nsplit = R.MODES[mode][0]
    _, plan_groups, _, streams = ops.rnn_plan(cell, H, nb, nsplit)
    groups = plan_groups if max_groups is None else min(max_groups, plan_groups)
    sched = Schedule(steps, nb, n_dirs, groups, "cuda", streams)
    case = R.Case(cell, H, mode, steps, nb, n_dirs=n_dirs, flags=flags, seed=R.case_seed(cell, H, nb, mode), h0=h0,
                  c0=c0, sched=sched)
    desc, bufs = R.build_desc(case, sched, "cuda", streams, pad_cols=pad_cols)
    ops.rnn_seq(desc, 0.0)
    torch.cuda.synchronize()
    n = n_dirs * H
    h_hi = bufs["h_hi"].double().cpu().numpy()
    h_lo = bufs["h_lo"].double().cpu().numpy() if bufs["h_lo"] is not None else None
    for plane in (h_hi,) if h_lo is None else (h_hi, h_lo):
        assert np.all(plane[:case.rows, n:] == 5.0), f"{name}: padding columns of h overwritten"
        assert np.all(plane[case.rows:] == 5.0), f"{name}: rows past the last packed row overwritten"
        assert np.isfinite(plane[:case.rows, :n]).all(), f"{name}: rows of h not written (NaN pre-fill)"
    hh, hl = h_hi[:case.rows], None if h_lo is None else h_lo[:case.rows]
    h_ref, c_ref, slack = R.teacher_forced(case, hh, hl)
    err = R.errors(case, hh, hl, h_ref, slack)
    worst = float(err.max())
    print(f"K3 {name} {mode} worst={float(R.ulp_errors(case, hh, hl, h_ref).max()):.3g} bound={R.BOUNDS[mode]:g} "
          f"of-allowance={worst:.3g} groups={sched.n_groups} streams={streams}")
    if worst > 1.0:
        r, col = np.unravel_index(int(np.argmax(err)), err.shape)
        raise AssertionError(f"{name} {mode}: row {r} (utterance {case.row_utt[r]}, step {case.row_step[r]}) column "
                             f"{col}: kernel {h_hi[r, col]!r} reference {h_ref[r, col]!r} -> {worst:.3g} x allowance")
    if "c_out" in bufs:
        c_out = bufs["c_out"].cpu().numpy()[:case.n_utt]
        ce = float(R.c_errors(case, c_out, c_ref).max())
        print(f"K3 {name} {mode} c_out worst={ce * R.C_BOUNDS[mode]:.3g} bound={R.C_BOUNDS[mode]:g}")
        assert ce <= 1.0, f"{name}: c_out off the teacher-forced c by {ce:.3g} x bound"
    return worst


# ------------------------------------------------------------------------------------------------ instance matrix
F = R.GRU_FLAGS
# (id, cell, flags, H, slots, mode, directions)
MATRIX = [
    ("lstm-64-16", LSTM, 0, 64, 16, "bf16", 1), ("lstm-64-32", LSTM, 0, 64, 32, "fp16", 1),
    ("lstm-192-64", LSTM, 0, 192, 64, "bf16", 1), ("blstm-64-16", LSTM, 0, 64, 16, "fp16", 2),
    ("blstm-64-64", LSTM, 0, 64, 64, "bf16", 2),
    ("lstm-256-32", LSTM, 0, 256, 32, "bf16", 1), ("lstm-256-32", LSTM, 0, 256, 32, "fp16", 1),
    ("blstm-256-32", LSTM, 0, 256, 32, "fp16", 2),
    ("lstm-512-32", LSTM, 0, 512, 32, "bf16", 1), ("lstm-512-32", LSTM, 0, 512, 32, "fp16", 1),
    ("lstm-512-16", LSTM, 0, 512, 16, "bf16", 1), ("lstm-512-64", LSTM, 0, 512, 64, "fp16", 1),
    ("lstm-512-16-fp32", LSTM, 0, 512, 16, "fp32", 1), ("lstm-512-32-fp32", LSTM, 0, 512, 32, "fp32", 1),
    ("lstm-192-16-fp32", LSTM, 0, 192, 16, "fp32", 1), ("lstm-192-32-fp32", LSTM, 0, 192, 32, "fp32", 1),
    ("blstm-192-32-fp32", LSTM, 0, 192, 32, "fp32", 2),
    ("lstm-384-16-fp32", LSTM, 0, 384, 16, "fp32", 1), ("lstm-384-32-fp32", LSTM, 0, 384, 32, "fp32", 1),
    ("lstm-576-16-fp32", LSTM, 0, 576, 16, "fp32", 1), ("lstm-640-32", LSTM, 0, 640, 32, "bf16", 1),
    ("lstm-1024-16", LSTM, 0, 1024, 16, "bf16", 1), ("lstm-1024-32", LSTM, 0, 1024, 32, "fp16", 1),
    ("lstm-1152-16", LSTM, 0, 1152, 16, "fp16", 1),
    ("lstm-512-128", LSTM, 0, 512, 128, "bf16", 1), ("lstm-192-128", LSTM, 0, 192, 128, "fp16", 1),
    ("blstm-128-128", LSTM, 0, 128, 128, "bf16", 2),
    ("gru-64-16", GRU, F["gru"], 64, 16, "bf16", 1), ("mgrurelu-192-32", GRU, F["mgrurelu"], 192, 32, "fp16", 1),
    ("mgrurelur-64-64", GRU, F["mgrurelur"], 64, 64, "bf16", 1), ("bgru-64-32", GRU, F["gru"], 64, 32, "fp16", 2),
    ("gru-512-16", GRU, F["gru"], 512, 16, "fp16", 1), ("mgrurelu-512-32", GRU, F["mgrurelu"], 512, 32, "bf16", 1),
    ("gru-512-32", GRU, F["gru"], 512, 32, "fp16", 1),
    ("mgrurelur-512-64", GRU, F["mgrurelur"], 512, 64, "bf16", 1),
    ("gru-512-16-fp32", GRU, F["gru"], 512, 16, "fp32", 1),
    ("mgrurelu-512-32-fp32", GRU, F["mgrurelu"], 512, 32, "fp32", 1),
    ("gru-64-16-fp32", GRU, F["gru"], 64, 16, "fp32", 1), ("bgru-64-16-fp32", GRU, F["mgrurelur"], 64, 16, "fp32", 2),
    ("mgrurelur-256-32-fp32", GRU, F["mgrurelur"], 256, 32, "fp32", 1),
    ("gru-384-16-fp32", GRU, F["gru"], 384, 16, "fp32", 1),
    ("mgrurelu-448-32-fp32", GRU, F["mgrurelu"], 448, 32, "fp32", 1),
    ("gru-576-16-fp32", GRU, F["gru"], 576, 16, "fp32", 1), ("gru-640-32", GRU, F["gru"], 640, 32, "bf16", 1),
    ("gru-1024-16", GRU, F["gru"], 1024, 16, "bf16", 1),
    ("mgrurelu-1024-32", GRU, F["mgrurelu"], 1024, 32, "fp16", 1),
    ("gru-1152-16", GRU, F["mgrurelur"], 1152, 16, "bf16", 1),
    ("gru-512-128", GRU, F["gru"], 512, 128, "bf16", 1), ("mgrurelur-256-128", GRU, F["mgrurelur"], 256, 128, "fp16", 1),
    ("mgrurelu-256-128", GRU, F["mgrurelu"], 256, 128, "bf16", 1),
    ("mgrurelu-512-128", GRU, F["mgrurelu"], 512, 128, "fp16", 1),
    ("bgru-192-128", GRU, F["gru"], 192, 128, "bf16", 2),
    ("peep-512-32", PEEP, 0, 512, 32, "bf16", 1), ("peep-128-32", PEEP, 0, 128, 32, "fp16", 1),
    ("peep-64-16", PEEP, 0, 64, 16, "bf16", 1), ("peep-64-16", PEEP, 0, 64, 16, "fp16", 1),
    ("peep-128-32-fp32", PEEP, 0, 128, 32, "fp32", 1), ("peep-320-16-fp32", PEEP, 0, 320, 16, "fp32", 1),
]


@pytest.mark.parametrize("name,cell,flags,H,nb,mode,nd", MATRIX, ids=[f"{m[0]}-{m[5]}" for m in MATRIX])
def test_instance_matrix(nn, name, cell, flags, H, nb, mode, nd):
    """Ragged lengths over 2.5 batches (a partial last batch) in every instance the dispatch reaches."""
    n_utt = nb * 5 // 2
    steps = ragged(n_utt, 1, 30 if H <= 512 else 16, seed=H + nb)
    run_case(name, cell, H, mode, steps, nb, n_dirs=nd, flags=flags, pad_cols=0 if nb == 64 else 16)


# ------------------------------------------------------------------------------------------------ schedule edges
EDGE_KERNELS = [  # (id, cell, flags, H, slots, mode): one per exchange family
    ("lstm-64-16", LSTM, 0, 64, 16, "bf16"), ("lstm-64-32-fp32", LSTM, 0, 64, 32, "fp32"),
    ("lstm-256-32-mc", LSTM, 0, 256, 32, "fp16"), ("lstm-256-128", LSTM, 0, 256, 128, "bf16"),
    ("gru-64-32", GRU, F["gru"], 64, 32, "fp16"), ("gru-128-128", GRU, F["gru"], 128, 128, "bf16"),
    ("peep-64-32", PEEP, 0, 64, 32, "bf16"),
]


def _edge_steps(kind, nb):
    if kind == "single-length-1":
        return [1]
    if kind == "equal-lengths":
        return [9] * (2 * nb)  # an exact multiple of the slots
    if kind == "one-long-many-1":
        return [1] * (nb + 5) + [57] + [1] * (nb - 3)  # the active prefix drops to 1 after the first step
    raise ValueError(kind)


@pytest.mark.parametrize("kind", ["single-length-1", "equal-lengths", "one-long-many-1"])
@pytest.mark.parametrize("name,cell,flags,H,nb,mode", EDGE_KERNELS, ids=[e[0] for e in EDGE_KERNELS])
def test_schedule_edges(nn, kind, name, cell, flags, H, nb, mode):
    run_case(f"{name}-{kind}", cell, H, mode, _edge_steps(kind, nb), nb, flags=flags)


@pytest.mark.parametrize("name,cell,flags,H,nb,mode", [
    ("blstm-64-32", LSTM, 0, 64, 32, "bf16"), ("blstm-64-16-fp32", LSTM, 0, 64, 16, "fp32"),
    ("blstm-256-32-mc", LSTM, 0, 256, 32, "bf16"), ("blstm-192-128", LSTM, 0, 192, 128, "fp16"),
    ("bgru-64-64", GRU, F["mgrurelur"], 64, 64, "fp16"), ("bgru-128-128", GRU, F["gru"], 128, 128, "bf16"),
])
def test_one_group_runs_every_item_back_to_back(nn, name, cell, flags, H, nb, mode):
    """n_groups = 1: one lane works through several batches of both directions and reloads the weights in between;
    state must restart at every item."""
    steps = ragged(nb * 3 + 3, 1, 24, seed=5)
    run_case(f"{name}-one-group", cell, H, mode, steps, nb, n_dirs=2, flags=flags, max_groups=1)


@pytest.mark.parametrize("name,cell,flags,H,nb,mode,nd", [
    ("lstm-256-64", LSTM, 0, 256, 64, "bf16", 2), ("lstm-512-32-mc", LSTM, 0, 512, 32, "bf16", 1),
    ("lstm-64-16", LSTM, 0, 64, 16, "fp16", 1), ("gru-512-16-fp32", GRU, F["gru"], 512, 16, "fp32", 1),
    ("lstm-512-128", LSTM, 0, 512, 128, "fp16", 1),
])
def test_every_group_plan_reports(nn, name, cell, flags, H, nb, mode, nd):
    """n_groups at the maximum nnam_rnn_plan reports, with more items than lanes."""
    from nnacousticmodeling_b200 import ops
    _, g, _, s = ops.rnn_plan(cell, H, nb, R.MODES[mode][0])
    steps = ragged(nb * (g * s + 3), 1, 12 if H < 512 else 4, seed=g)
    run_case(f"{name}-max-groups", cell, H, mode, steps, nb, n_dirs=nd, flags=flags)


BASE_EDGES = [  # (id, cell, flags, H, slots, mode, BASE_SMEM of the instance)
    ("lstm-64-16-S4", LSTM, 0, 64, 16, "bf16", 1024), ("lstm-64-32-S2", LSTM, 0, 64, 32, "fp16", 2048),
    ("lstm-64-16-fp32", LSTM, 0, 64, 16, "fp32", 2048), ("lstm-256-32-mc", LSTM, 0, 256, 32, "bf16", 2048),
    ("lstm-128-128-wide2", LSTM, 0, 128, 128, "bf16", 1024), ("gru-64-128-wide", GRU, F["gru"], 64, 128, "fp16", 1024),
    ("gru-64-64", GRU, F["mgrurelu"], 64, 64, "bf16", 2048), ("peep-64-16", PEEP, 0, 64, 16, "bf16", 2048),
]


@pytest.mark.parametrize("extra", [0, 1])
@pytest.mark.parametrize("name,cell,flags,H,nb,mode,base", BASE_EDGES, ids=[e[0] for e in BASE_EDGES])
def test_prefix_table_in_shared_or_global_memory(nn, extra, name, cell, flags, H, nb, mode, base):
    """A batch of exactly BASE_SMEM steps keeps its prefix table in shared memory; one more step reads it from global
    memory.  Shorter utterances ride along so that the active prefix shrinks."""
    steps = [base + extra, base // 2, 40, 3, 1]
    run_case(f"{name}-T{base + extra}", cell, H, mode, steps, nb, n_dirs=2 if cell == LSTM else 1, flags=flags)


# ------------------------------------------------------------------------------------------------ carried state
@pytest.mark.parametrize("mode", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("nb", [16, 32, 64])
@pytest.mark.parametrize("H", [64, 256])
@pytest.mark.parametrize("cell", [LSTM, GRU], ids=["lstm", "gru"])
def test_carried_state(nn, cell, H, nb, mode):
    """h0 / c0 -> c_out (LSTM) and h0 (GRU) with ragged lengths over several batches: c_out is the state at each
    utterance's own last step.  LSTM, H = 256, 32 slots, 16-bit: the multicast kernel nnam_rnn_plan planned for is ruled
    out by the carried state, and the single-stream counter-based instance must take the plan's one stream.  The
    fp32-accurate mode has no 64-slot instance: nnam_rnn_plan must say so on the host."""
    from nnacousticmodeling_b200 import NnamError, ops
    if mode == "fp32" and nb == 64:
        with pytest.raises(NnamError):
            ops.rnn_plan(cell, H, nb, R.MODES[mode][0])
        return
    steps = ragged(nb * 2 + 5, 1, 20, seed=nb)
    run_case(f"carried-{'lstm' if cell == LSTM else 'gru'}-{H}-{nb}", cell, H, mode, steps, nb,
             flags=0 if cell == LSTM else F["gru"], h0=True, c0=cell == LSTM)


def test_carried_state_descriptor_accepted_for_every_plan(nn):
    """For every (cell, H, slots, mode) nnam_rnn_plan accepts, a carried-state descriptor built with the plan's
    streams is accepted and computes the right thing (one short utterance per configuration)."""
    from nnacousticmodeling_b200 import NnamError, ops
    n = 0
    for cell in (LSTM, GRU):
        for H in range(64, 1345, 64):
            for nb in (16, 32, 64):
                for mode in ("bf16", "fp16", "fp32"):
                    try:
                        ops.rnn_plan(cell, H, nb, R.MODES[mode][0])
                    except NnamError:
                        continue
                    run_case(f"plan-{cell}-{H}-{nb}", cell, H, mode, [3, 2], nb, flags=F["gru"] if cell == GRU else 0,
                             h0=True, c0=cell == LSTM)
                    n += 1
    assert n >= 100


# ------------------------------------------------------------------------------------------------ process-wide switches
CHILD_CASES = {
    "NNAM_RNN_MC=0": [("lstm-512-32-single", LSTM, 512, 32, "bf16", 1, [40, 33, 7, 1] * 9),
                      ("lstm-512-32-single", LSTM, 512, 32, "fp16", 2, [25, 9, 3] * 12),
                      ("lstm-256-32-2streams", LSTM, 256, 32, "bf16", 1, [30, 12, 5, 1] * 20),
                      ("lstm-512-32-single-T2049", LSTM, 512, 32, "bf16", 1, [2049, 100, 3, 1])],
    "NNAM_RNN_WIDE_STREAMS=1": [("lstm-512-128-wide1", LSTM, 512, 128, "bf16", 1, [30, 12, 5, 1] * 70),
                                ("blstm-192-128-wide1", LSTM, 192, 128, "fp16", 2, [19, 8, 2] * 90),
                                ("lstm-128-128-wide1-T2048", LSTM, 128, 128, "bf16", 1, [2048, 50, 1]),
                                ("lstm-128-128-wide1-T2049", LSTM, 128, 128, "bf16", 1, [2049, 50, 1])],
    "NNAM_RNN_WIDE_STREAMS=3": [("lstm-512-128-wide3", LSTM, 512, 128, "bf16", 1, [30, 12, 5, 1] * 100),
                                ("blstm-128-128-wide3", LSTM, 128, 128, "fp16", 2, [19, 8, 2] * 150),
                                ("lstm-128-128-wide3-T768", LSTM, 128, 128, "bf16", 1, [768, 50, 1]),
                                ("lstm-128-128-wide3-T769", LSTM, 128, 128, "fp16", 1, [769, 50, 1])],
}


def _child(switch):
    for name, cell, H, nb, mode, nd, steps in CHILD_CASES[switch]:
        run_case(name, cell, H, mode, steps, nb, n_dirs=nd)
    print("CHILD OK")


@pytest.mark.parametrize("switch", sorted(CHILD_CASES))
def test_process_wide_switches(nn, switch):
    """NNAM_RNN_MC and NNAM_RNN_WIDE_STREAMS are read once per process: their kernels run in a child process, which is
    waited for (and killed on timeout) before the test returns."""
    key, val = switch.split("=")
    env = dict(os.environ, **{key: val})
    res = subprocess.run([sys.executable, os.path.abspath(__file__), switch], cwd=ROOT, env=env, capture_output=True,
                         text=True, timeout=900)
    print(res.stdout)
    assert res.returncode == 0 and "CHILD OK" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]


# ------------------------------------------------------------------------------------------------ end to end
@pytest.mark.parametrize("network,units,prec", [("lstm", 256, "bf16"), ("lstm", 256, "fp16"), ("lstm", 512, "fp16"),
                                                ("gru", 256, "bf16")])
def test_stateful_call_16bit(nn, network, units, prec):
    """Stateful model(x) on a 16-bit net against oracle.RecurrentNet: the user-facing surface of carried state."""
    from oracle import nnam_oracle as O
    p = O.init_recurrent(np.random.default_rng(units), network, 40, units, 2, 39, bias_scale=0.2)
    m = nn.get_nn(network, 2, [units], 39, nn.F.relu, [5])
    m.load_params(p)
    m.precision = prec
    ref = O.RecurrentNet(p, network, 2)
    xs = np.random.default_rng(units + 1).standard_normal((5, 6, 40)).astype(np.float32)
    m.reset_state()
    for t in range(5):
        assert np.abs(m(xs[t]) - ref(xs[t])).max() < 5e-2


# ------------------------------------------------------------------------------------------------ rejected on the host
def test_unsupported_sizes_are_rejected_on_the_host(nn):
    from nnacousticmodeling_b200 import NnamError, ops
    from oracle import nnam_oracle as O
    for nb in (16, 32, 64, 128):
        with pytest.raises(NnamError):
            ops.rnn_plan(LSTM, 1024, nb, 3)
    for cell in (LSTM, GRU, PEEP):
        with pytest.raises(NnamError):
            ops.rnn_plan(cell, 96, 32, 1)
    off = np.array([0, 5, 8], np.int32)
    x = np.random.default_rng(0).standard_normal((8, 40)).astype(np.float32)
    for units, prec in ((1024, "fp32"), (96, "bf16")):
        p = O.init_recurrent(np.random.default_rng(1), "lstm", 40, units, 1, 39)
        m = nn.get_nn("lstm", 1, [units], 39, nn.F.relu, [5])
        m.load_params(p)
        m.precision = prec
        with pytest.raises(NnamError):
            nn.predict(m, x, off, 39, "lstm", 0, 1, 0, None, progress=False)


if __name__ == "__main__":  # child process of test_process_wide_switches
    _child(sys.argv[1])
