"""Float64 step reference of the K3 recurrence kernels (``nnam_rnn_seq``) with the kernels' rounding points.

Test infrastructure, not part of the product.  It works on the packed time-major layout of include/nnam_b200.h:
row (t, u) of batch b is ``row0_b + base_b[t] + u``, utterances in length-sorted order, and direction 1 walks every
utterance backwards.  ``recurrent_engine.Schedule`` (tested on the CPU in test_schedule_cpu.py) supplies the packed
rows and the lane assignment; everything else -- weight packing, gx, descriptor -- is built here from the header's
layout description.

Cells (header contract)
  LSTM       gate rows interleaved per unit [a, i, f, o] (Chainer order); c = tanh(a) s(i) + s(f) c; h = s(o) tanh(c).
  GRU family rows per unit [U_z, U_r | 0, U, 0]; the U terms and their biases are absent at step 0 unless h0 is given
             (MGRU.py); flags bit 0 = reset gate, bits 1-2 = candidate activation.
  wide GRU   (128 slots) gate-blocked rows: per 32 units the 32 rows of z, [r,] candidate.  gx already holds W_b + U_b;
             the kernel subtracts u_bias at step 0.
  PEEPHOLE   LSTM rows plus the block in w_hi[1], rows per unit [0, P_i, P_f, P_o]: i, f see P c_{t-1}, o sees P_o c_t.
  s(x) = tanh(x/2)/2 + 1/2 (Chainer's sigmoid, as oracle.sigmoid).

Rounding points (read from the kernel source; everything else is fp32 in the kernels and float64 here)
  gx            read as stored: 16-bit in single-pass modes, fp32 in the fp32-accurate mode (nsplit 3)
                (recurrent.cu:372-388 load_gx / gx_val; recurrent_mc.cu:295; recurrent_wide.cu:545-546;
                recurrent_wide_gru.cu:251-254)
  weights       16-bit hi plane, + bf16 lo plane in fp32 mode (TMA loads, recurrent.cu:289-298)
  h (output and MMA operand)   rounded to the 16-bit type, + bf16 lo = bf16(h - hi) in fp32 mode
                (recurrent.cu:390-396 stage_put; recurrent_mc.cu:254; recurrent_wide.cu:248-250, 554;
                recurrent_wide_gru.cu:320)
  GRU r*h       crosses the exchange as a 16-bit tile (+ lo): recurrent.cu:546, recurrent_wide_gru.cu:288
  peephole c'   crosses the exchange as a 16-bit tile (+ lo) for P_o c' (recurrent.cu:478) and, one step later,
                for P_i c, P_f c (the c tile keeps c_{t-1}, recurrent.cu:449)
  LSTM c        fp32 registers for the whole utterance (recurrent.cu:348-362, 516)
  GRU h state   fp32 registers (recurrent.cu:357-359, 574; recurrent_wide_gru.cu:318); only the MMA operand is 16-bit
  h0 / c0       h0 read as 16-bit hi (+ lo), c0 as fp32 (recurrent.cu:335-362)

Teacher forcing.  Every row of step t is recomputed from the kernel's OWN output h at step t-1 (t+1 for direction 1):
that output is exactly the 16-bit MMA operand the kernel used.  Only the fp32 state (LSTM c, GRU h, peephole c) is
carried by the reference, along the kernel's trajectory.  Each row therefore carries a one-step error, and a slip
(wrong slot, row or direction, stale exchange slot, state not reset between the items of a lane, bias missing or
extra at step 0, dropped lo plane) shows at the row where it happens.

Error model of one step of h (what the bounds in BOUNDS cover):
  * one output rounding: <= 0.5 ulp of the 16-bit type (fp32 mode: hi + lo keep 16 significant bits, <= 2^-17 |h|);
  * tanh.approx.f32 in the 16-bit modes: relative error <= 2^-11 per call, five calls feed h (a, i, f, o, tanh c) --
    about 0.1 bf16 ulp or 1-2 fp16 ulp; the fp32 mode uses tanhf;
  * fp32 accumulation of the MMA over K = H terms, and the carried state's drift from the same per-step errors
    (damped by the forget gate / 1 - z): well below the above for the H of the tests.
  Near h = 0 these errors are absolute rather than relative, so the ulp is taken at max(|h_ref|, H_FLOOR).
  One more term is not a one-step rounding of h: the GRU reset gate's r*h and the peephole's c tiles are rounded by the
  kernel from ITS r and state, which the test cannot observe.  Where the reference's value and the kernel's straddle a
  rounding boundary the two roundings differ by one step of the 16-bit type (of the bf16 lo plane in fp32 mode), and the
  following product carries that as an absolute error into the candidate (the i / f / o pre-activations).  The
  allowance adds, per element, three standard deviations of such independent flips over the whole operand, propagated
  through the gate's slope (``slack``, see _flip_spread and errors()).
"""
from __future__ import annotations

import numpy as np

CELL_LSTM, CELL_GRU, CELL_PEEPHOLE = 0, 1, 2
ACT_RELU, ACT_SIGMOID, ACT_TANH = 1, 2, 3
GRU_FLAGS = {"gru": 1 | (ACT_TANH << 1), "mgrurelu": ACT_RELU << 1, "mgrurelur": 1 | (ACT_RELU << 1)}

# mode -> (nsplit, elem, 16-bit type of the hi plane)
MODES = {"bf16": (1, 0, "bf16"), "fp16": (1, 1, "fp16"), "fp32": (3, 0, "bf16"),
         "f64": (3, 0, None)}  # f64: no rounding anywhere (ties the reference to oracle.RecurrentNet)
# bound on |h_kernel - h_ref| per row: ulps of the 16-bit type at max(|h_ref|, H_FLOOR), or, in fp32 mode, absolute
# for |h_ref| <= 1 and relative above (the ReLU GRU's h is unbounded)
BOUNDS = {"bf16": 2.0, "fp16": 4.0, "fp32": 3e-5}
H_FLOOR = 2.0 ** -4
# bound on |c_out - c_ref| / max(|c_ref|, 1)
C_BOUNDS = {"bf16": 2e-3, "fp16": 2e-3, "fp32": 2e-5}


# ------------------------------------------------------------------------------------------------ 16-bit arithmetic
def bf16(x):
    """fp32 -> bf16 round-to-nearest-even (what __float2bfloat16_rn does), as float64 values."""
    b = np.ascontiguousarray(np.asarray(x, np.float32)).view(np.uint32).astype(np.uint64)
    b = ((b + 0x7FFF + ((b >> 16) & 1)) >> 16) << 16
    return b.astype(np.uint32).view(np.float32).astype(np.float64)


def fp16(x):
    return np.asarray(x, np.float32).astype(np.float16).astype(np.float64)


def round16(x, kind):
    return bf16(x) if kind == "bf16" else fp16(x)


def other_type_bits(x, kind):
    """``x`` encoded as the OTHER 16-bit type and read back as ``kind``: a kernel passing the wrong element flag."""
    if kind == "fp16":
        b = (np.ascontiguousarray(bf16(x).astype(np.float32)).view(np.uint32) >> 16).astype(np.uint16)
        return b.view(np.float16).astype(np.float64)
    b = np.ascontiguousarray(np.asarray(x, np.float32).astype(np.float16)).view(np.uint16).astype(np.uint32) << 16
    return b.view(np.float32).astype(np.float64)


def split(x, mode):
    """The kernels' h staging: (hi, lo) with hi = the 16-bit value and lo = bf16(x - hi) in fp32 mode (else 0)."""
    if mode == "f64":
        return np.asarray(x, np.float64), 0.0
    x = np.asarray(x, np.float32)
    hi = round16(x, MODES[mode][2])
    lo = bf16(x - hi) if mode == "fp32" else np.zeros_like(hi)
    return hi, lo


def ulp16(x, kind):
    _, e = np.frexp(np.abs(np.asarray(x, np.float64)))
    if kind == "bf16":
        return np.ldexp(1.0, np.maximum(e - 8, -133))
    return np.ldexp(1.0, np.maximum(e - 11, -24))


def sigmoid(x):
    return np.tanh(0.5 * x) * 0.5 + 0.5


_ACT = {0: lambda v: v, ACT_RELU: lambda v: np.maximum(v, 0.0), ACT_SIGMOID: sigmoid, ACT_TANH: np.tanh}


# ------------------------------------------------------------------------------------------------ layouts
class Layout:
    """Gate-row layout of one cell: ``cols[g]`` = packed row (= gx column) of gate g for every unit."""

    def __init__(self, cell, hidden, flags=0, wide_gru=False):
        self.cell, self.H, self.flags, self.wide_gru = cell, hidden, flags, wide_gru
        self.reset = cell == CELL_GRU and bool(flags & 1)
        self.act = (flags >> 1) & 3
        j = np.arange(hidden)
        if cell == CELL_GRU and wide_gru:
            names = ["z", "r", "c"] if self.reset else ["z", "c"]
            ng = len(names)
            self.G = ng * hidden
            self.cols = {g: (j // 32) * (32 * ng) + k * 32 + j % 32 for k, g in enumerate(names)}
        elif cell == CELL_GRU:
            self.G = 4 * hidden
            self.cols = {"z": 4 * j, "r": 4 * j + 1, "c": 4 * j + 2}
        else:
            self.G = 4 * hidden
            self.cols = {g: 4 * j + k for k, g in enumerate("aifo")}

    def pad_rows(self):
        """Packed rows the kernel never uses (zero in the weights; their gx columns hold noise)."""
        used = np.zeros(self.G, bool)
        for g, c in self.cols.items():
            if not (g == "r" and not self.reset):
                used[c] = True
        return np.nonzero(~used)[0]


# ------------------------------------------------------------------------------------------------ test data
def case_seed(cell, hidden, nb, mode):
    """Seed of the test data of one (cell, H, slots, mode): shared by the GPU cases and the CPU margin checks."""
    return 1000 * cell + hidden + 7 * nb + {"bf16": 0, "fp16": 1, "fp32": 2, "f64": 3}[mode]


class Case:
    """One K3 launch: cell, shapes, schedule and the operands exactly as the kernel reads them (float64 values that
    the 16-bit / fp32 buffers represent exactly).  Per-utterance arrays (h0, c0, c_out) are in sorted order."""

    def __init__(self, cell, hidden, mode, steps, nb, n_dirs=1, flags=0, seed=0, h0=False, c0=False, sched=None,
                 w_scale=None, gx_scale=1.0):
        self.cell, self.H, self.mode, self.nb, self.n_dirs, self.flags = cell, hidden, mode, nb, n_dirs, flags
        self.nsplit, self.elem, self.kind = MODES[mode]
        self.steps = np.asarray(steps, np.int64)
        self.lay = Layout(cell, hidden, flags, wide_gru=(cell == CELL_GRU and nb == 128))
        if sched is None:
            from nnacousticmodeling_b200.recurrent_engine import Schedule
            sched = Schedule(self.steps, nb, n_dirs, 1, "cpu", 1)
        self.sched = sched
        self.lens = self.steps[sched.order]  # sorted order
        self.n_utt = len(self.lens)
        self.rows = sched.n_rows
        self.row_utt = np.asarray(sched.row_sorted_utt, np.int64)
        self.row_step = np.asarray(sched.row_step, np.int64)
        self.row_of = np.full((self.n_utt, int(self.lens.max())), -1, np.int64)
        self.row_of[self.row_utt, self.row_step] = np.arange(self.rows)
        starts = sched.d_group_start.cpu().numpy()
        ib, idr = sched.d_item_batch.cpu().numpy(), sched.d_item_dir.cpu().numpy()
        self.lanes = [list(zip(ib[a:b].tolist(), idr[a:b].tolist())) for a, b in zip(starts[:-1], starts[1:])]

        rng = np.random.default_rng(seed)
        H, G, lay = hidden, self.lay.G, self.lay
        # lateral weights scaled so that the recurrent term is a sizeable part of every pre-activation
        # (tests/test_rnn_reference_cpu.py holds ||W h|| / ||gx|| >= 0.3)
        if w_scale is None:
            w_scale = 1.5 if cell != CELL_GRU else 1.2
        self.w_hi, self.w_lo, self.ub, self.gx = [], [], [], []
        for d in range(n_dirs):
            w = (w_scale / np.sqrt(H)) * rng.standard_normal((G, H))
            w[lay.pad_rows()] = 0.0
            hi, lo = split(w, mode)
            self.w_hi.append(hi)
            self.w_lo.append(lo)
            ub = np.zeros(G)
            if cell == CELL_GRU:
                ub = np.asarray(0.3 * rng.standard_normal(G), np.float32).astype(np.float64)
                ub[lay.pad_rows()] = 0.0
            self.ub.append(ub)
            gx = gx_scale * rng.standard_normal((self.rows, G))
            if cell in (CELL_LSTM, CELL_PEEPHOLE):
                gx[:, lay.cols["f"]] += 1.0  # Chainer's forget-gate bias
            if lay.wide_gru:
                gx = gx + ub  # the projection bias holds W_b + U_b
            if mode == "f64":
                self.gx.append(gx)
            elif self.nsplit == 3:
                self.gx.append(np.asarray(gx, np.float32).astype(np.float64))
            else:
                self.gx.append(round16(gx, self.kind))
        self.pw_hi = self.pw_lo = None
        if cell == CELL_PEEPHOLE:
            pw = (0.8 / np.sqrt(H)) * rng.standard_normal((G, H))
            pw[lay.cols["a"]] = 0.0
            self.pw_hi, self.pw_lo = split(pw, mode)
        self.h0_hi = self.h0_lo = self.c0 = None
        if h0:
            self.h0_hi, self.h0_lo = split(0.6 * np.tanh(rng.standard_normal((self.n_utt, n_dirs * H))), mode)
        if c0:
            self.c0 = np.asarray(rng.standard_normal((self.n_utt, n_dirs * H)), np.float32).astype(np.float64)

    # direction d's step index of every row, and the row holding its previous h (-1: none)
    def step_index(self, d):
        t, u = self.row_step, self.row_utt
        return t if d == 0 else self.lens[u] - 1 - t

    def prev_row(self, d):
        t, u = self.row_step, self.row_utt
        tp = t - 1 if d == 0 else t + 1
        ok = (tp >= 0) & (tp < self.lens[u])
        return np.where(ok, self.row_of[u, np.clip(tp, 0, self.row_of.shape[1] - 1)], -1)


# ------------------------------------------------------------------------------------------------ one step
def _flip_spread(q, w, mode):
    """Spread of q . w^T when every element of the rounded operand q may sit one rounding step away from where the
    kernel rounded it: three standard deviations of independent one-ulp flips of random sign."""
    if mode == "f64":
        return 0.0
    u = ulp16(q, MODES[mode][2]) * (2.0 ** -8 if mode == "fp32" else 1.0)  # fp32 mode: the step of the lo plane
    return 3.0 * np.sqrt((u * u) @ (w * w).T)


_ACT_SLOPE = {0: lambda v: np.ones_like(v), ACT_RELU: lambda v: np.ones_like(v),
              ACT_SIGMOID: lambda v: sigmoid(v) * (1.0 - sigmoid(v)), ACT_TANH: lambda v: 1.0 - np.tanh(v) ** 2}


def _step(case, d, gx, lat, state, have_h, u_bias_at_step0=False, peep_prev_c=False):
    """Gate arithmetic of one step for n rows.  gx: (n, G) projection; lat: (n, G) = h_prev . W^T or None (no h);
    state: (n, H) fp32 state (LSTM / peephole c, GRU h).  Returns (h, new state, slack): slack is what the rounding of
    an operand the test cannot observe (GRU r*h, peephole c tiles) may add to |h - h_ref| (see errors())."""
    lay, mode = case.lay, case.mode
    cols = lay.cols
    pre = gx.copy()
    if have_h:
        pre += lat
        if case.cell == CELL_GRU and not lay.wide_gru:
            pre += case.ub[d]
    elif case.cell == CELL_GRU and lay.wide_gru and not u_bias_at_step0:
        pre -= case.ub[d]
    elif case.cell == CELL_GRU and not lay.wide_gru and u_bias_at_step0:
        pre += case.ub[d]
    if case.cell == CELL_GRU:
        z = sigmoid(pre[:, cols["z"]])
        slack = 0.0
        if lay.reset and have_h:
            r = sigmoid(pre[:, cols["r"]])
            rh = sum(split(r * state, mode))
            w_c = (case.w_hi[d] + case.w_lo[d])[cols["c"]]
            cand = gx[:, cols["c"]] + rh @ w_c.T + (0.0 if lay.wide_gru else case.ub[d][cols["c"]])
            slack = z * _ACT_SLOPE[lay.act](cand) * _flip_spread(rh, w_c, mode)
        else:
            cand = pre[:, cols["c"]]
        hb = _ACT[lay.act](cand)
        h = z * hb + (1.0 - z) * state if have_h else z * hb
        return h, h, slack
    a = np.tanh(pre[:, cols["a"]])
    pi, pf, po = pre[:, cols["i"]], pre[:, cols["f"]], pre[:, cols["o"]]
    s_i = s_f = 0.0
    if case.cell == CELL_PEEPHOLE:
        pw = case.pw_hi + case.pw_lo
        if have_h:
            cq = sum(split(state, mode))
            pi = pi + cq @ pw[cols["i"]].T
            pf = pf + cq @ pw[cols["f"]].T
            s_i, s_f = _flip_spread(cq, pw[cols["i"]], mode), _flip_spread(cq, pw[cols["f"]], mode)
    i, f = sigmoid(pi), sigmoid(pf)
    c = a * i + f * state
    if case.cell != CELL_PEEPHOLE:
        return sigmoid(po) * np.tanh(c), c, 0.0
    cq = sum(split(state if peep_prev_c else c, mode))
    po = po + cq @ pw[cols["o"]].T
    o, tc = sigmoid(po), np.tanh(c)
    slack = (np.abs(tc) * o * (1.0 - o) * _flip_spread(cq, pw[cols["o"]], mode)
             + o * (1.0 - tc * tc) * (np.abs(a) * i * (1.0 - i) * s_i + np.abs(state) * f * (1.0 - f) * s_f))
    return o * tc, c, slack


def _initial_state(case, d, utts):
    H = case.H
    st = np.zeros((len(utts), H))
    if case.cell == CELL_GRU and case.h0_hi is not None:
        st = (case.h0_hi + case.h0_lo)[utts, d * H:(d + 1) * H]
    elif case.cell == CELL_LSTM and case.c0 is not None:
        st = case.c0[utts, d * H:(d + 1) * H].copy()
    return st


# ------------------------------------------------------------------------------------------------ teacher forcing
def teacher_forced(case, h_hi, h_lo=None):
    """Reference h of every packed row from the kernel's own previous h.  h_hi / h_lo: (rows, >= n_dirs*H) values the
    kernel wrote.  Returns (h_ref (rows, n_dirs*H), c_last (n_utt, n_dirs*H) or None, slack (rows, n_dirs*H)): slack
    is the error the kernel's own rounding of r*h / the peephole c tiles may add (see errors())."""
    H, rows = case.H, case.rows
    h_k = np.asarray(h_hi, np.float64)[:, :case.n_dirs * H]
    if h_lo is not None:
        h_k = h_k + np.asarray(h_lo, np.float64)[:, :case.n_dirs * H]
    h_ref = np.full((rows, case.n_dirs * H), np.nan)
    slack = np.zeros((rows, case.n_dirs * H))
    c_last = np.full((case.n_utt, case.n_dirs * H), np.nan) if case.cell == CELL_LSTM else None
    for d in range(case.n_dirs):
        prev = case.prev_row(d)
        s_idx = case.step_index(d)
        hp = np.where(prev[:, None] >= 0, h_k[np.maximum(prev, 0), d * H:(d + 1) * H], 0.0)
        first = prev < 0
        if case.h0_hi is not None:  # the first row of every utterance sees h0
            h0 = (case.h0_hi + case.h0_lo)[:, d * H:(d + 1) * H]
            hp[first] = h0[case.row_utt[first]]
        lat = hp @ (case.w_hi[d] + case.w_lo[d]).T  # one float64 product over all rows
        gx = case.gx[d]
        state = _initial_state(case, d, np.arange(case.n_utt))
        order = np.lexsort((case.row_utt, s_idx))
        bounds = np.searchsorted(s_idx[order], np.arange(int(case.lens.max()) + 1))
        for s in range(int(case.lens.max())):
            rs = order[bounds[s]:bounds[s + 1]]
            us = case.row_utt[rs]
            have_h = s > 0 or case.h0_hi is not None
            h, st, sl = _step(case, d, gx[rs], lat[rs], state[us], have_h)
            state[us] = st
            h_ref[rs, d * H:(d + 1) * H] = h
            slack[rs, d * H:(d + 1) * H] = sl
            if c_last is not None:
                done = case.lens[us] - 1 == s
                c_last[us[done], d * H:(d + 1) * H] = st[done]
    return h_ref, c_last, slack


def errors(case, h_hi, h_lo, h_ref, slack=0.0):
    """Per-element error in units of its allowance (<= 1 passes).  Allowance: BOUNDS[mode] ulps of the 16-bit type at
    max(|h_ref|, H_FLOOR), or max(|h_ref|, 1) * BOUNDS['fp32'] in fp32 mode, plus ``slack`` (teacher_forced)."""
    n = case.n_dirs * case.H
    got = np.asarray(h_hi, np.float64)[:, :n]
    if case.mode == "fp32":
        got = got + np.asarray(h_lo, np.float64)[:, :n]
        allow = np.maximum(np.abs(h_ref), 1.0) * BOUNDS["fp32"]
    else:
        allow = ulp16(np.maximum(np.abs(h_ref), H_FLOOR), case.kind) * BOUNDS[case.mode]
    e = np.abs(got - h_ref) / (allow + slack)
    return np.where(np.isfinite(e), e, np.inf)


def ulp_errors(case, h_hi, h_lo, h_ref):
    """|h - h_ref| in the unit BOUNDS states it: ulps of the 16-bit type at max(|h_ref|, H_FLOOR), or, in fp32 mode,
    the error over max(|h_ref|, 1)."""
    return errors(case, h_hi, h_lo, h_ref) * BOUNDS[case.mode]


def c_errors(case, c_out, c_ref):
    return np.abs(np.asarray(c_out, np.float64) - c_ref) / np.maximum(np.abs(c_ref), 1.0) / C_BOUNDS[case.mode]


# ------------------------------------------------------------------------------------------------ free-running model
MUTATIONS = ("neighbour_slot", "skip_step", "bwd_walks_forward", "state_not_reset", "u_bias_at_step0", "drop_lo",
             "peep_prev_c", "other_type")


def simulate(case, mutation=None):
    """A model of the kernel: the lanes' items run in order, each a batch walked step by step over its active prefix,
    with the kernel's rounding points.  ``mutation`` plants one of MUTATIONS.  Returns (h_hi, h_lo, c_out)."""
    H, mode = case.H, case.mode
    h_hi = np.full((case.rows, case.n_dirs * H), np.nan)
    h_lo = np.zeros_like(h_hi)
    c_out = np.full((case.n_utt, case.n_dirs * H), np.nan)
    nb = case.nb
    shortest = case.n_utt - 1
    first_item = True
    for lane in case.lanes:
        carried = None
        for b, d in lane:
            utts = np.arange(b * nb, min((b + 1) * nb, case.n_utt))
            lens = case.lens[utts]
            state = _initial_state(case, d, utts)
            if mutation == "state_not_reset" and carried is not None and carried[0] == d:
                state = carried[1][:len(utts)].copy()
            hq = None  # previous step's MMA operand (hi + lo), per slot
            if case.h0_hi is not None:
                hq = (case.h0_hi + case.h0_lo)[utts, d * H:(d + 1) * H]
            for s in range(int(lens.max())):
                n_s = int((lens > s).sum())
                us = utts[:n_s]
                bwd = d == 1 and mutation != "bwd_walks_forward"
                t = lens[:n_s] - 1 - s if bwd else np.full(n_s, s)
                rows = case.row_of[us, t]
                have_h = hq is not None
                op = hq[:n_s] if have_h else None
                if have_h and mutation == "neighbour_slot" and first_item and n_s >= 2 and s == lens[1] // 2:
                    op = op.copy()
                    op[0] = hq[1]
                if have_h and mutation == "drop_lo" and s > 0:
                    op = round16(op, case.kind)
                lat = op @ (case.w_hi[d] + case.w_lo[d]).T if have_h else None
                h, st, _ = _step(case, d, case.gx[d][rows], lat, state[:n_s], have_h,
                              u_bias_at_step0=mutation == "u_bias_at_step0",
                              peep_prev_c=mutation == "peep_prev_c")
                hi, lo = split(h, mode)
                if mutation == "skip_step" and s == 1 and shortest in us and case.lens[shortest] >= 3:
                    k = int(np.nonzero(us == shortest)[0][0])
                    prev_row = case.row_of[shortest, t[k] + (1 if bwd else -1)]
                    hi[k], lo[k], st[k] = h_hi[prev_row, d * H:(d + 1) * H], h_lo[prev_row, d * H:(d + 1) * H], state[k]
                state[:n_s] = st
                new_q = hi + lo
                hq = new_q if hq is None else np.concatenate([new_q, hq[n_s:]])
                h_hi[rows, d * H:(d + 1) * H] = other_type_bits(hi, case.kind) if mutation == "other_type" else hi
                h_lo[rows, d * H:(d + 1) * H] = lo
                done = lens[:n_s] - 1 == s
                c_out[us[done], d * H:(d + 1) * H] = st[done]
            carried = (d, state)
            first_item = False
    return h_hi, h_lo, c_out


# ------------------------------------------------------------------------------------------------ descriptor
def build_desc(case, sched, device, streams, n_groups_check=None, pad_cols=0, pad_rows=3):
    """_native.RnnDesc for ``case`` from this module's own packing (include/nnam_b200.h), with device buffers:
    every buffer 32-byte aligned, gx_ld / h_ld larger than needed by ``pad_cols`` (rounded to 16 elements), h filled
    with NaN, and sentinels in the padding columns and in ``pad_rows`` rows past the last one.  Returns (desc, bufs)."""
    import torch
    from nnacousticmodeling_b200._native import RnnDesc

    H, nd, G, rows = case.H, case.n_dirs, case.lay.G, case.rows
    t16 = torch.float16 if case.kind == "fp16" else torch.bfloat16
    keep = []

    def dev(a, dtype):
        t = torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64).to(dtype).to(device)
        assert t.data_ptr() % 32 == 0
        keep.append(t)
        return t

    def rup(v, m):
        return (v + m - 1) // m * m

    gx_ld = rup(nd * G + pad_cols, 16)
    h_ld = rup(nd * H + pad_cols, 16)
    gx_t = torch.float32 if case.nsplit == 3 else t16
    gx = torch.full((rows + pad_rows, gx_ld), 3.0, dtype=gx_t, device=device)
    for d in range(nd):
        gx[:rows, d * G:(d + 1) * G] = torch.as_tensor(case.gx[d]).to(gx_t).to(device)
    keep.append(gx)
    h_hi = torch.full((rows + pad_rows, h_ld), float("nan"), dtype=t16, device=device)
    h_hi[:, nd * H:] = 5.0
    h_hi[rows:] = 5.0
    h_lo = None
    if case.nsplit == 3:
        h_lo = torch.full((rows + pad_rows, h_ld), float("nan"), dtype=torch.bfloat16, device=device)
        h_lo[:, nd * H:] = 5.0
        h_lo[rows:] = 5.0
    w_hi = [dev(w, t16) for w in case.w_hi]
    w_lo = [dev(w, torch.bfloat16) for w in case.w_lo] if case.nsplit == 3 else [None] * nd
    x_rows = sched.n_lanes * 4 * case.nb
    xchg_hi = torch.full((x_rows, H), float("nan"), dtype=t16, device=device)
    xchg_lo = torch.full((x_rows, H), float("nan"), dtype=torch.bfloat16, device=device) if case.nsplit == 3 else None

    desc = RnnDesc()
    desc.cell, desc.hidden, desc.n_dirs, desc.batch = case.cell, H, nd, case.nb
    desc.streams, desc.nsplit, desc.flags, desc.elem = streams, case.nsplit, case.flags, case.elem
    for d in range(nd):
        desc.gx[d] = gx.data_ptr() + gx.element_size() * d * G
        desc.w_hi[d] = w_hi[d].data_ptr()
        desc.w_lo[d] = w_lo[d].data_ptr() if w_lo[d] is not None else None
        desc.u_bias[d] = dev(case.ub[d], torch.float32).data_ptr() if case.cell == CELL_GRU else None
    if case.cell == CELL_PEEPHOLE:
        desc.w_hi[1] = dev(case.pw_hi, t16).data_ptr()
        desc.w_lo[1] = dev(case.pw_lo, torch.bfloat16).data_ptr() if case.nsplit == 3 else None
    desc.gx_ld, desc.w_ld = gx_ld, H
    desc.h_hi, desc.h_lo, desc.h_ld = h_hi.data_ptr(), (h_lo.data_ptr() if h_lo is not None else None), h_ld
    desc.xchg_hi = xchg_hi.data_ptr()
    desc.xchg_lo = xchg_lo.data_ptr() if xchg_lo is not None else None
    desc.n_items, desc.item_batch, desc.item_dir = sched.n_items, sched.d_item_batch.data_ptr(), sched.d_item_dir.data_ptr()
    desc.n_groups, desc.group_item_start = sched.n_groups, sched.d_group_start.data_ptr()
    desc.batch_row0, desc.batch_steps = sched.d_row0.data_ptr(), sched.d_steps.data_ptr()
    desc.batch_nutt, desc.batch_base_off = sched.d_nutt.data_ptr(), sched.d_boff.data_ptr()
    desc.base, desc.utt_len = sched.d_base.data_ptr(), sched.d_utt_len.data_ptr()
    n_pad = sched.n_batches * case.nb  # the kernels index per-utterance state by batch * nb + slot
    bufs = dict(gx=gx, h_hi=h_hi, h_lo=h_lo, xchg=(xchg_hi, xchg_lo), keep=keep, sched=sched)
    if case.h0_hi is not None:
        pad = np.zeros((n_pad - case.n_utt, nd * H))
        desc.h0_hi = dev(np.concatenate([case.h0_hi, pad]), t16).data_ptr()
        desc.h0_lo = dev(np.concatenate([case.h0_lo, pad]), torch.bfloat16).data_ptr() if case.nsplit == 3 else None
    if case.c0 is not None:
        desc.c0 = dev(np.concatenate([case.c0, np.zeros((n_pad - case.n_utt, nd * H))]), torch.float32).data_ptr()
    if case.cell == CELL_LSTM and (case.h0_hi is not None or case.c0 is not None):
        c_out = torch.full((n_pad, nd * H), float("nan"), dtype=torch.float32, device=device)
        desc.c_out = c_out.data_ptr()
        bufs["c_out"] = c_out
    desc.counters = sched.d_counters.data_ptr()
    return desc, bufs
