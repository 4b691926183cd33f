"""Host side of the recurrent path (K3): weight packing, the packed time-major schedule, and
``forward_utterances`` = feature gather -> per layer (input-projection GEMM over all frames, persistent
recurrence kernel) -> output GEMM -> head with scatter back to frame order.

Packed layout.  Utterances of a shard are sorted by step count (descending) and cut into batches of NB.
Batch b occupies rows [row0_b, row0_b + sum(steps)) in time-major order: row(t, u) = row0_b + base_b[t] + u,
where base_b[t] = number of (utterance, step) pairs of the batch with step < t.  No padding rows exist, so
unlike the reference (predict_folds.py:34-64 computes ALL utterances at every t up to Lmax) no work is spent
on finished utterances.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import engine, ops
from ._native import NnamError, RnnDesc
from .engine import HeadSpec, LinearDev, _as_host_tensor, _dev_vec, _device, fused_head_ok, get_plan
from .ops import OUT_BF16, OUT_BF16_SPLIT, OUT_F32, round_up

CELL_LSTM, CELL_GRU, CELL_PEEPHOLE = 0, 1, 2
PROFILE_CYCLES = None  # set to a list to collect per-CTA phase cycle counters of every K3 launch
DEFAULT_BATCH = None  # None: pick the slots per batch (16 / 32 / 64 / 128) from a cost model of the schedule: the step cost
# (nnam_rnn_plan, measured in profiles/r01_k3_phase_cycles.md) grows sub-linearly in the batch width, but fewer and
# larger work items balance worse over the CTA groups and lengthen the critical path of the longest utterance


# ------------------------------------------------------------------------------------------
# plan: packed weights per layer
# ------------------------------------------------------------------------------------------
class RecLayer:
    pass


_ACT_CODE = {"identity": 0, "relu": 1, "sigmoid": 2, "tanh": 3}


def _interleave4(blocks, h, cols):
    """Stack up to three (h, cols) blocks as rows 4j+k (k = 0,1,2), row 4j+3 and missing blocks are zero."""
    out = np.zeros((4 * h, cols), dtype=np.float32)
    for k, blk in enumerate(blocks):
        if blk is not None:
            out[k::4] = blk
    return out


def build_plan(plan, model):
    p, dev, split = model.params, plan.device, plan.split
    net = model.network
    plan.n_dirs = 2 if model.bidirectional else 1
    plan.hidden = h = model.n_units
    plan.rec_layers = []
    plan.gru_flags = 0
    kind = plan.act_kind  # bf16 / fp16 hi plane, or the bf16 hi/lo pair of the fp32-accurate mode
    dirs = ("fwd/", "bwd/") if model.bidirectional else ("",)

    def to_dev_bf16(w):
        return ops.convert_f32(torch.from_numpy(np.ascontiguousarray(w, dtype=np.float32)).to(dev), kind)

    if model.bidirectional and net == "peepholelstm":
        raise NnamError("bidirectional peephole LSTM is not defined (SURVEY A9 covers LSTM and GRU)")
    if net in ("lstm", "zoneoutlstm", "zoneoutdropoutlstm", "blstm"):
        plan.cell = CELL_LSTM
        for l in range(model.layers):
            L = RecLayer()
            up_w = np.concatenate([p[f"layer_{l}/{d}upward/W"] for d in dirs], axis=0)
            up_b = np.concatenate([p[f"layer_{l}/{d}upward/b"] for d in dirs], axis=0)
            L.upward = LinearDev(up_w, up_b, dev, split, plan.elem)  # gx for both directions in one GEMM
            L.lat = [to_dev_bf16(p[f"layer_{l}/{d}lateral/W"]) for d in dirs]
            L.u_bias = [None for _ in dirs]
            plan.rec_layers.append(L)
    elif net in ("gru", "mgrurelu", "mgrurelur", "mgru", "bgru"):
        # MGRU.py: W_* act on x (folded into the gx GEMM), U_* on h (resident in K3); rows interleaved per unit
        # as [z, r, candidate, pad] so that the LSTM kernel's slice/quad structure carries over.
        plan.cell = CELL_GRU
        reset = model.use_reset_gate
        plan.gru_flags = (1 if reset else 0) | (_ACT_CODE[model.activation.name] << 1)
        for l in range(model.layers):
            L = RecLayer()
            ups, upb, L.lat, L.u_bias = [], [], [], []
            for d in dirs:
                pre = f"layer_{l}/{d}"
                d_in = p[pre + "W_z/W"].shape[1]
                ups.append(_interleave4([p[pre + "W_z/W"], p[pre + "W_r/W"] if reset else None, p[pre + "W/W"]], h, d_in))
                upb.append(_interleave4([p[pre + "W_z/b"][:, None], p[pre + "W_r/b"][:, None] if reset else None,
                                         p[pre + "W/b"][:, None]], h, 1)[:, 0])
                L.lat.append(to_dev_bf16(_interleave4([p[pre + "U_z/W"], p[pre + "U_r/W"] if reset else None,
                                                       p[pre + "U/W"]], h, h)))
                ub = _interleave4([p[pre + "U_z/b"][:, None], p[pre + "U_r/b"][:, None] if reset else None,
                                   p[pre + "U/b"][:, None]], h, 1)[:, 0]
                L.u_bias.append(torch.from_numpy(np.ascontiguousarray(ub)).to(dev))
            L.upward = LinearDev(np.concatenate(ups, axis=0), np.concatenate(upb, axis=0), dev, split, plan.elem)
            plan.rec_layers.append(L)
    elif net == "peepholelstm":
        # chainer_networks.py:103-121.  The time-step engine (peephole_engine) always exists: it serves the stateful
        # model(x) surface and shapes the persistent kernel cannot hold.  Where the lateral slice, the peephole block
        # [0, P_i, P_f, P_o] per unit and two operand tiles fit in shared memory, whole sets run in K3.
        from . import peephole_engine
        plan.cell = CELL_PEEPHOLE
        peephole_engine.build_plan(plan, model)
        plan.peep_persistent = False
        try:
            for cand in (32, 16):
                try:
                    ops.rnn_plan(CELL_PEEPHOLE, h, cand, 3 if split else 1)
                    plan.peep_persistent = True
                    break
                except NnamError:
                    continue
        except Exception:  # noqa: BLE001
            plan.peep_persistent = False
        if plan.peep_persistent:
            for l in range(model.layers):
                pre = f"layer_{l}/"
                L = RecLayer()
                L.upward = LinearDev(p[pre + "upward/W"], p[pre + "upward/b"], dev, split, plan.elem)
                pblock = _interleave4([None, p[pre + "peep_i/W"], p[pre + "peep_f/W"]], h, h)
                pblock[3::4] = p[pre + "peep_o/W"]
                L.lat = [to_dev_bf16(p[pre + "lateral/W"]), to_dev_bf16(pblock)]
                L.u_bias = [None]
                plan.rec_layers.append(L)
        return
    else:
        raise NnamError(f"network '{net}' is not implemented on the B200 path")
    plan.out = LinearDev(p["out/W"], p["out/b"], dev, split, plan.elem)


def _block32(blocks, h):
    """Gate-blocked row order of the 128-slot GRU kernel: for every 32 units the rows of gate 0, then gate 1, ..."""
    cols = blocks[0].shape[1:]
    a = np.stack([np.asarray(b, dtype=np.float32).reshape((h // 32, 32) + cols) for b in blocks], axis=1)
    return np.ascontiguousarray(a.reshape((len(blocks) * h,) + cols))


def gru_wide_layers(plan, model):
    """Second packing of a GRU-family net for the 128-slot kernel (csrc/recurrent_wide_gru.cu): rows / gx columns
    [z(32) | r(32) | cand(32)] per 32 units (no reset gate: [z | cand]), and the U biases folded into the projection
    bias (the kernel takes them out again at step 0, where MGRU.py:70-83 has no U terms).  Built on first use."""
    layers = plan.__dict__.get("_gru_wide_layers")
    if layers is not None:
        return layers
    p, dev, h = model.params, plan.device, plan.hidden
    reset = bool(plan.gru_flags & 1)
    dirs = ("fwd/", "bwd/") if model.bidirectional else ("",)
    names = ["z", "r", ""] if reset else ["z", ""]

    def key(pre, mat, g):
        return f"{pre}{mat}_{g}" if g else f"{pre}{mat}"

    layers = []
    for l in range(model.layers):
        L = RecLayer()
        ups, upb, L.lat, L.u_bias = [], [], [], []
        for d in dirs:
            pre = f"layer_{l}/{d}"
            ub = _block32([p[key(pre, "U", g) + "/b"][:, None] for g in names], h)[:, 0]
            ups.append(_block32([p[key(pre, "W", g) + "/W"] for g in names], h))
            upb.append(_block32([p[key(pre, "W", g) + "/b"][:, None] for g in names], h)[:, 0] + ub)
            L.lat.append(ops.convert_f32(torch.from_numpy(_block32([p[key(pre, "U", g) + "/W"] for g in names], h)).to(dev),
                                         plan.prec.out16))
            L.u_bias.append(torch.from_numpy(np.ascontiguousarray(ub)).to(dev))
        L.upward = LinearDev(np.concatenate(ups, axis=0), np.concatenate(upb, axis=0), dev, False, plan.elem)
        L.gate_cols = len(names) * h
        layers.append(L)
    plan._gru_wide_layers = layers
    return layers


# ------------------------------------------------------------------------------------------
# schedule
# ------------------------------------------------------------------------------------------
def assign_lanes(bsteps, n_dirs, max_groups, streams, solo_ratio=1.0):
    """Spread the (batch, direction) work items over lanes = (CTA group, stream).  Returns (items per lane, groups
    used, critical path in steps).

    One stream per group (the usual case): a group just works through its items (direction 0 first), so its time
    is the sum of their step counts -- longest-processing-time-first, then moves / swaps out of the fullest group
    until nothing improves (on the test-shaped set that takes the critical path from 880 to 798 steps; the bound is
    the longest utterance, 785).  Several streams per group: per direction LPT over the lanes; the critical path
    accounts for a group switching direction only when all of its streams are done with the current one.  Two streams
    per group (the 128-slot kernel): see :func:`_assign_pairs`."""
    if streams in (2, 3):
        return _assign_pairs(bsteps, n_dirs, max_groups, solo_ratio, streams)
    n_batches = len(bsteps)
    bsteps = [int(t) for t in bsteps]
    n_groups = max(1, min(max_groups, (n_batches * (n_dirs if streams == 1 else 1) + streams - 1) // streams))
    if streams == 1:
        n_groups = max(1, min(max_groups, n_batches * n_dirs))
        items = sorted(((bsteps[b], b, d) for b in range(n_batches) for d in range(n_dirs)), key=lambda t: -t[0])
        bins = [[] for _ in range(n_groups)]
        load = [0] * n_groups
        for it in items:
            g = min(range(n_groups), key=load.__getitem__)
            bins[g].append(it)
            load[g] += it[0]
        improved = n_groups > 1
        while improved:
            improved = False
            gmax = max(range(n_groups), key=load.__getitem__)
            for i, it in enumerate(bins[gmax]):
                for g in range(n_groups):
                    if g == gmax:
                        continue
                    if load[g] + it[0] < load[gmax]:  # move
                        bins[g].append(bins[gmax].pop(i))
                        load[g] += it[0]
                        load[gmax] -= it[0]
                        improved = True
                        break
                    for j, other in enumerate(bins[g]):  # swap with a shorter item
                        if other[0] < it[0] and max(load[gmax] - it[0] + other[0], load[g] - other[0] + it[0]) < load[gmax]:
                            bins[gmax][i], bins[g][j] = other, it
                            delta = it[0] - other[0]
                            load[gmax] -= delta
                            load[g] += delta
                            improved = True
                            break
                    if improved:
                        break
                if improved:
                    break
        per_lane = [sorted(((b, d) for _, b, d in bn), key=lambda t: (t[1], -bsteps[t[0]])) for bn in bins]
        return per_lane, n_groups, (max(load) if n_batches else 0)
    n_groups = max(1, min(max_groups, (n_batches + streams - 1) // streams))
    n_lanes = n_groups * streams
    per_lane = [[] for _ in range(n_lanes)]
    load = np.zeros((n_lanes, n_dirs), np.int64)
    by_len = np.argsort(-np.asarray(bsteps), kind="stable")
    for d in range(n_dirs):
        for b in by_len:
            ln = int(np.argmin(load[:, d]))
            load[ln, d] += int(bsteps[b])
            per_lane[ln].append((int(b), d))  # direction-sorted by construction
    per_group = load.reshape(n_groups, streams, n_dirs).max(axis=1).sum(axis=1)
    return per_lane, n_groups, (int(per_group.max()) if n_batches else 0)


def _assign_pairs(bsteps, n_dirs, max_groups, solo_ratio, streams=2):
    """Lane assignment for groups of two (or three) streams.  A step of a stream costs ``c_busy`` cycles while its sibling is
    busy and ``c_solo = solo_ratio * c_busy`` once the sibling has run out of work, so (in units of busy steps) a
    group needs  solo_ratio * longest lane + (1 - solo_ratio) * mean of the other lanes  per direction, and all streams
    switch direction together.  Greedy longest-first onto the lane that leaves its group cheapest, then moves / swaps out of
    the most expensive group while that lowers the maximum.  Returns (items per lane, groups, critical path in busy
    steps)."""
    n_batches = len(bsteps)
    bsteps = [int(t) for t in bsteps]
    n_groups = max(1, min(max_groups, n_batches))
    r = float(solo_ratio)
    S = int(streams)
    load = np.zeros((n_groups, S, n_dirs), np.float64)
    lanes = [[[] for _ in range(S)] for _ in range(n_groups)]

    def gcost(g):
        a = load[g]
        top = a.max(axis=0)
        return float((r * top + (1.0 - r) * (a.sum(axis=0) - top) / (S - 1)).sum())

    def gcost_with(g, s_, d, delta):
        load[g, s_, d] += delta
        c = gcost(g)
        load[g, s_, d] -= delta
        return c

    items = sorted(((bsteps[b], b, d) for b in range(n_batches) for d in range(n_dirs)), key=lambda t: -t[0])
    for t, b, d in items:
        best = None
        for g in range(n_groups):
            for s_ in range(S):
                c = gcost_with(g, s_, d, t)
                if best is None or c < best[0] - 1e-9:
                    best = (c, g, s_)
            if not load[g].any():
                break  # all further groups are empty too: same cost
        _, g, s_ = best
        load[g, s_, d] += t
        lanes[g][s_].append((t, b, d))
    cost = [gcost(g) for g in range(n_groups)]
    for _ in range(400):
        gw = int(np.argmax(cost))
        done = True
        for sw in range(S):
            for i, (t, b, d) in enumerate(lanes[gw][sw]):
                for g in range(n_groups):
                    if g == gw:
                        continue
                    for s_ in range(S):
                        # move
                        load[gw, sw, d] -= t
                        load[g, s_, d] += t
                        if max(gcost(gw), gcost(g)) < cost[gw] - 1e-9:
                            lanes[g][s_].append(lanes[gw][sw].pop(i))
                            cost[gw], cost[g] = gcost(gw), gcost(g)
                            done = False
                            break
                        load[gw, sw, d] += t
                        load[g, s_, d] -= t
                        # swap with a shorter item of the same direction
                        for j, (t2, b2, d2) in enumerate(lanes[g][s_]):
                            if d2 != d or t2 >= t:
                                continue
                            load[gw, sw, d] += t2 - t
                            load[g, s_, d] += t - t2
                            if max(gcost(gw), gcost(g)) < cost[gw] - 1e-9:
                                lanes[gw][sw][i], lanes[g][s_][j] = (t2, b2, d2), (t, b, d)
                                cost[gw], cost[g] = gcost(gw), gcost(g)
                                done = False
                                break
                            load[gw, sw, d] -= t2 - t
                            load[g, s_, d] -= t - t2
                        if not done:
                            break
                    if not done:
                        break
                if not done:
                    break
            if not done:
                break
        if done:
            break
    used = max((g + 1 for g in range(n_groups) if any(lanes[g])), default=1)
    per_lane = [sorted(((b, d) for _, b, d in lanes[g][s_]), key=lambda t: (t[1], -bsteps[t[0]]))
                for g in range(used) for s_ in range(S)]
    return per_lane, used, (int(np.ceil(max(cost))) if n_batches else 0)


class Schedule:
    """Packed time-major schedule of a set of utterances (host arrays + device copies).

    Utterances are sorted by length and cut into batches of ``nb`` slots.  Work items are (batch, direction) pairs;
    they are spread over LANES = (CTA group, stream): a group runs ``streams`` batches concurrently against one
    resident weight slice, so all streams of a group work on the same direction at a time (direction 0 first)."""

    def __init__(self, steps, nb, n_dirs, max_groups, device, streams=1, solo_ratio=1.0, row_offset=0):
        steps = np.asarray(steps, dtype=np.int64)
        n_utt = len(steps)
        self.nb, self.n_utt, self.streams = nb, n_utt, streams
        self.order = np.argsort(-steps, kind="stable")  # sorted position -> original utterance
        s_sorted = steps[self.order]
        n_batches = (n_utt + nb - 1) // nb
        row0 = np.zeros(n_batches, np.int32)
        bsteps = np.zeros(n_batches, np.int32)
        bnutt = np.zeros(n_batches, np.int32)
        boff = np.zeros(n_batches, np.int32)
        bases = []
        # per packed row: sorted-utterance index and step
        row_utt, row_step = [], []
        r = int(row_offset)  # first packed row of this schedule (a MixedSchedule packs its parts one after the other)
        off = 0
        for b in range(n_batches):
            ls = s_sorted[b * nb:(b + 1) * nb]
            t_max = int(ls[0])
            active = (ls[None, :] > np.arange(t_max)[:, None])  # (T, nutt)
            n_t = active.sum(axis=1)
            base = np.concatenate([[0], np.cumsum(n_t)]).astype(np.int32)
            row0[b], bsteps[b], bnutt[b], boff[b] = r, t_max, len(ls), off
            bases.append(base)
            tt, uu = np.nonzero(active)  # time-major order, u ascending within t  == packed order
            row_utt.append(uu + b * nb)
            row_step.append(tt)
            r += int(base[-1])
            off += len(base)
        self.n_rows = r - int(row_offset)
        self.n_batches = n_batches
        self.h_base = bases  # host copies of the per-batch prefix-sum tables
        self.row_sorted_utt = np.concatenate(row_utt) if row_utt else np.zeros(0, np.int64)
        self.row_step = np.concatenate(row_step) if row_step else np.zeros(0, np.int64)
        utt_len = np.zeros(n_batches * nb, np.int32)
        utt_len[:n_utt] = s_sorted
        per_lane, self.n_groups, self.max_group_steps = assign_lanes(bsteps, n_dirs, max_groups, streams, solo_ratio)
        n_lanes = self.n_groups * streams
        flat = [it for ln in per_lane for it in ln]
        starts = np.concatenate([[0], np.cumsum([len(ln) for ln in per_lane])]).astype(np.int32)
        self.n_items, self.n_lanes = len(flat), n_lanes
        self.total_steps = int(bsteps.sum()) * n_dirs

        def dv(a):
            return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(device)

        self.d_item_batch = dv([b for b, _ in flat])
        self.d_item_dir = dv([d for _, d in flat])
        self.d_group_start = dv(starts)
        self.d_row0, self.d_steps, self.d_nutt, self.d_boff = dv(row0), dv(bsteps), dv(bnutt), dv(boff)
        self.d_base = dv(np.concatenate(bases) if bases else np.zeros(1, np.int32))
        self.d_utt_len = dv(utt_len)
        self.d_counters = torch.zeros(max(n_lanes, 1), dtype=torch.int32, device=device)


class MixedSchedule:
    """Two schedules over one packed row space, run as two concurrent cooperative launches on disjoint SM sets: the
    longest utterances in the low-latency 32-slot kernel (they are the critical path of a layer: 785 steps x 4.3 k
    cycles against 10 k in the 128-slot kernel; the groups holding shorter batches work through up to three of them one
    after the other), everything else in the 128-slot two-stream kernel on the remaining groups.  Exposes the attributes forward_utterances() reads from a Schedule."""

    def __init__(self, steps, k_long, groups_long, nb_long, streams_long, nb_bulk, groups_bulk, streams_bulk,
                 ratio_bulk, n_dirs, device):
        steps = np.asarray(steps, dtype=np.int64)
        by_len = np.argsort(-steps, kind="stable")
        idx_a, idx_b = by_len[:k_long], by_len[k_long:]
        sa = Schedule(steps[idx_a], nb_long, n_dirs, groups_long, device, streams_long)
        sb = Schedule(steps[idx_b], nb_bulk, n_dirs, groups_bulk, device, streams_bulk, ratio_bulk, row_offset=sa.n_rows)
        self.parts = [(sa, nb_long), (sb, nb_bulk)]
        self.nb = ("mixed", int(k_long), int(groups_long), int(nb_long))
        self.n_utt = len(steps)
        self.n_rows = sa.n_rows + sb.n_rows
        self.order = np.concatenate([idx_a[sa.order], idx_b[sb.order]])
        self.row_sorted_utt = np.concatenate([sa.row_sorted_utt, sb.row_sorted_utt + len(idx_a)])
        self.row_step = np.concatenate([sa.row_step, sb.row_step])
        self.streams = None
        self._cuda_streams = None

    def cuda_streams(self):
        if self._cuda_streams is None:
            # The long part's stream has the higher priority: both launches of a layer become runnable on the same
            # event, and the long part's CTAs must be placed FIRST -- its multicast kernel (csrc/recurrent_mc.cu) runs as
            # clusters of 16 CTAs, which need a whole GPC's worth of free SMs each; placed after the bulk kernel has
            # spread over every GPC they would wait for it to finish, and the two parts would run one after the other.
            self._cuda_streams = [torch.cuda.Stream(priority=-1 if i == 0 else 0) for i in range(len(self.parts))]
        return self._cuda_streams


def _mixed_candidate(plan, steps, s_sorted, nsplit, best_cost):
    """Cost of the best long / bulk split (None if the plain schedules win or the kernels do not apply):
    (cost, utterances in the long part, its groups, its slots per batch, its streams, bulk groups, bulk streams,
    bulk solo ratio)."""
    if os.environ.get("NNAM_RNN_MIXED", "1") == "0" or plan.cell not in (CELL_LSTM, CELL_GRU) or nsplit != 1:
        return None
    try:
        _, max_b, cyc_b, streams_b = ops.rnn_plan(plan.cell, plan.hidden, 128, nsplit)
    except NnamError:
        return None
    if streams_b not in (2, 3) or len(steps) < 32 * 4:
        return None
    ratio = _solo_ratio(plan, 128, nsplit, cyc_b, streams_b)
    best = None
    forced = os.environ.get("NNAM_RNN_MIXED_GROUPS")  # tuning aid
    for nb_a in (32, 64):
        try:
            _, max_a, cyc_a, streams_a = ops.rnn_plan(plan.cell, plan.hidden, nb_a, nsplit)
        except NnamError:
            continue
        if streams_a != 1:
            continue
        # both kernels use 16-CTA groups on disjoint SMs: g_a groups (clusters, for the multicast kernel, of which at
        # most max_a are resident) leave max_b - g_a groups for the bulk part
        forced_b = os.environ.get("NNAM_RNN_MIXED_BATCHES")  # tuning aid
        for g_a in ((int(forced),) if forced else (1, 2, 3, 4, 5, 6)):
            if max_b - g_a < 1 or g_a > max_a:
                break
            # At least one batch per group (a bidirectional net needs a group per direction of a batch to keep the two
            # passes over its longest utterance side by side); up to three, worked through one after the other: the
            # groups that hold the 2nd, 3rd ... longest batch have time left while the first walks the longest
            # utterance, and every batch they take shortens the bulk part's own longest lane.
            b_min = max(1, g_a // plan.n_dirs)
            for n_bat in ((int(forced_b),) if forced_b else range(b_min, 3 * b_min + 1)):
                k = nb_a * n_bat
                if len(steps) - k < 128:
                    break
                _, _, crit_a = assign_lanes(s_sorted[:k:nb_a], plan.n_dirs, g_a, streams_a)
                _, _, crit_b = assign_lanes(s_sorted[k::128], plan.n_dirs, max_b - g_a, streams_b, ratio)
                cost = max(crit_a * cyc_a, crit_b * cyc_b)
                if best is None or cost < best[0]:
                    best = (cost, k, g_a, nb_a, streams_a, max_b - g_a, streams_b, ratio)
                if crit_a * cyc_a > crit_b * cyc_b and not forced_b:
                    break  # the long part is already the longer one: more batches only make it longer
    if best is None or (best[0] > 0.95 * best_cost and os.environ.get("NNAM_RNN_MIXED") != "force"):
        return None
    return best


def _solo_ratio(plan, nb, nsplit, busy_cycles, streams):
    if streams not in (2, 3) or nb != 128:
        return 1.0
    return min(1.0, ops.rnn_solo_step_cycles(plan.cell, plan.hidden, nb, nsplit) / float(busy_cycles))


def pick_schedule(plan, steps, device, nb=None, allow_mixed=True):
    """Build the packed schedule; with nb=None choose the slots-per-stream (16 x 4 streams, 32 x 2, 64 x 1) that
    minimises the critical path (longest group) under the measured per-step cost.  The schedule depends only on the
    utterance lengths, so it is cached on the plan (a repeated call on the same data set re-uses it)."""
    steps = np.asarray(steps, dtype=np.int64)
    key = (steps.tobytes(), nb, plan.n_dirs, bool(allow_mixed))
    cache = plan.__dict__.setdefault("_sched_cache", {})
    hit = cache.get(key)
    if hit is not None:
        return hit
    nsplit = 3 if plan.split else 1
    cands = [nb] if nb else [16, 32, 64, 128]
    s_sorted = -np.sort(-steps, kind="stable")
    best = None
    for cand in cands:
        try:
            _, max_groups, cycles, streams = ops.rnn_plan(plan.cell, plan.hidden, cand, nsplit)
        except NnamError:
            if len(cands) == 1:
                raise
            continue
        ratio = _solo_ratio(plan, cand, nsplit, cycles, streams)
        # a batch runs as long as its longest utterance
        _, _, crit = assign_lanes(s_sorted[::cand], plan.n_dirs, max_groups, streams, ratio)
        cost = crit * cycles
        if best is None or cost < best[0]:
            best = (cost, cand, max_groups, streams, ratio)
    if best is None:
        raise NnamError("no recurrent kernel configuration fits this layer size / precision")
    mixed = _mixed_candidate(plan, steps, s_sorted, nsplit, best[0]) if (nb is None and allow_mixed) else None
    if mixed is not None:
        _, k, g_a, nb_a, streams_a, g_b, streams_b, ratio_b = mixed
        ms = MixedSchedule(steps, k, g_a, nb_a, streams_a, 128, g_b, streams_b, ratio_b, plan.n_dirs, device)
        res = (ms, ms.nb)
    else:
        _, cand, max_groups, streams, ratio = best
        res = (Schedule(steps, cand, plan.n_dirs, max_groups, device, streams, ratio), cand)
    if len(cache) >= 8:
        cache.pop(next(iter(cache)))
    cache[key] = res
    return res


class _StartFlags:
    """Pinned host words a launch's CTAs set when they start (NnamRnnDesc.started); the host polls them."""

    def __init__(self):
        self.buf = torch.zeros(256, dtype=torch.int32, pin_memory=True)
        self.view = self.buf.numpy()
        self.tag = 0

    def arm(self, desc):
        self.tag = (self.tag % 0x3fffffff) + 1
        desc.started = self.buf.data_ptr()
        desc.started_tag = self.tag

    def wait(self, n_ctas, timeout_s=0.25):
        import time
        t0 = time.perf_counter()
        v = self.view[:n_ctas]
        while not (v == self.tag).all():
            if time.perf_counter() - t0 > timeout_s:  # never block a pass on the hint: the launches are still correct
                return False
        return True


def _fill_desc(plan, sched, layer, gx, h_hi, h_lo, nb, h0=None, c0=None, c_out=None, xchg=None):
    H, nd = plan.hidden, plan.n_dirs
    d = RnnDesc()
    d.cell, d.hidden, d.n_dirs, d.batch, d.nsplit = plan.cell, H, nd, nb, 3 if plan.split else 1
    d.streams = sched.streams
    d.flags = plan.gru_flags
    d.elem = plan.elem
    for k in range(nd):
        d.gx[k] = gx.data_ptr() + gx.element_size() * k * getattr(layer, "gate_cols", 4 * H)
        d.w_hi[k] = layer.lat[k][0].data_ptr()
        d.w_lo[k] = layer.lat[k][1].data_ptr() if plan.split else None
        d.u_bias[k] = layer.u_bias[k].data_ptr() if layer.u_bias[k] is not None else None
    if plan.cell == CELL_PEEPHOLE:  # the peephole block travels in the direction-1 weight slot
        d.w_hi[1] = layer.lat[1][0].data_ptr()
        d.w_lo[1] = layer.lat[1][1].data_ptr() if plan.split else None
    xh, xl = xchg
    d.xchg_hi = xh.data_ptr()
    d.xchg_lo = xl.data_ptr() if xl is not None else None
    d.gx_ld = gx.stride(0)
    d.w_ld = layer.lat[0][0].stride(0)
    d.h_hi, d.h_lo, d.h_ld = h_hi.data_ptr(), (h_lo.data_ptr() if h_lo is not None else None), h_hi.stride(0)
    d.n_items, d.item_batch, d.item_dir = sched.n_items, sched.d_item_batch.data_ptr(), sched.d_item_dir.data_ptr()
    d.n_groups, d.group_item_start = sched.n_groups, sched.d_group_start.data_ptr()
    d.batch_row0, d.batch_steps = sched.d_row0.data_ptr(), sched.d_steps.data_ptr()
    d.batch_nutt, d.batch_base_off = sched.d_nutt.data_ptr(), sched.d_boff.data_ptr()
    d.base, d.utt_len = sched.d_base.data_ptr(), sched.d_utt_len.data_ptr()
    if h0 is not None:
        d.h0_hi = h0[0].data_ptr()
        d.h0_lo = h0[1].data_ptr() if h0[1] is not None else None
    d.c0 = c0.data_ptr() if c0 is not None else None
    d.c_out = c_out.data_ptr() if c_out is not None else None
    d.counters = sched.d_counters.data_ptr()
    if PROFILE_CYCLES is not None:
        buf = torch.zeros(148 * 8, dtype=torch.int64, device=plan.device)
        PROFILE_CYCLES.append(buf)
        d.debug_cycles = buf.data_ptr()
    return d


def _run_layers_mixed(model, plan, sched, a_hi, a_lo, rows, tag, ws):
    """run_layers for a MixedSchedule (bf16 mode, no carried state): per layer the input projection over all rows, then
    the two recurrence launches side by side on their own CUDA streams.  LSTM: both kernels read the same projection.
    GRU family: the 128-slot kernel takes gate-blocked columns, so each part gets its own projection GEMM over its own
    row range."""
    H, nd = plan.hidden, plan.n_dirs
    main = torch.cuda.current_stream()
    side = sched.cuda_streams()
    n_mats = 4 if plan.cell == CELL_LSTM else (3 if plan.gru_flags & 1 else 2)
    row_lo = 0
    ranges = []
    for part, _ in sched.parts:
        ranges.append((row_lo, row_lo + part.n_rows))
        row_lo += part.n_rows
    for l in range(len(plan.rec_layers)):
        h_hi = ws.get(f"{tag}.h{l % 2}.hi", rows, nd * H, plan.tdt)
        part_layers, part_gx = [], []
        for pi, (part, nb) in enumerate(sched.parts):
            layer = (gru_wide_layers(plan, model) if (plan.cell == CELL_GRU and nb == 128) else plan.rec_layers)[l]
            part_layers.append(layer)
            if pi > 0 and layer is part_layers[0]:
                part_gx.append(part_gx[0])  # same weights, same layout: one GEMM over all rows (below)
                continue
            gate_cols = getattr(layer, "gate_cols", 4 * H)
            shared = all(((gru_wide_layers(plan, model) if (plan.cell == CELL_GRU and nb2 == 128)
                           else plan.rec_layers)[l]) is layer for _, nb2 in sched.parts)
            gx = ws.get(f"{tag}.gx16" if shared else f"{tag}.gx16.p{pi}", rows, nd * gate_cols, plan.tdt)
            r0, r1 = (0, rows) if shared else ranges[pi]
            if r1 > r0:
                layer.upward(a_hi[r0:r1], None, r1 - r0, "identity", plan.prec.out16, out=(gx[r0:r1], None))
            part_gx.append(gx)
        ready = torch.cuda.Event()
        ready.record(main)
        for pi, ((part, nb), st) in enumerate(zip(sched.parts, side)):
            x_rows = part.n_lanes * 4 * nb
            name = f"{tag}.xchg{pi}.hi"
            fresh = ws.buf.get(name) is None or ws.buf[name].numel() < x_rows * H
            xchg = (ws.get(name, x_rows, H, plan.tdt), None)
            if fresh:
                xchg[0].zero_()
                ready.record(main)
            desc = _fill_desc(plan, part, part_layers[pi], part_gx[pi], h_hi, None, nb, xchg=xchg)
            first = pi == 0 and len(sched.parts) > 1
            if first:
                # The long part must be RESIDENT before the bulk part is submitted: its kernel runs as clusters of 16
                # CTAs (csrc/recurrent_mc.cu), which only fit while whole GPCs are free; submitted side by side the
                # bulk grid spread over every GPC first and the clusters waited for it to drain (measured: 3.9 ms
                # instead of 1.9 ms for the long part of cfg3).  Its CTAs announce themselves in pinned host memory.
                flags = plan.__dict__.get("_start_flags")
                if flags is None:
                    flags = plan._start_flags = _StartFlags()
                flags.arm(desc)
            with torch.cuda.stream(st):
                st.wait_event(ready)
                ops.rnn_seq(desc, 2.0 * part.n_rows * nd * n_mats * H * H)
                done = torch.cuda.Event()
                done.record(st)
            if first:
                flags.wait(part.n_groups * (4 * H // 128) if nb != 128 else 0)
            main.wait_event(done)
        a_hi, a_lo = h_hi, None
    return a_hi, a_lo, []


def run_layers(model, plan, sched, a_hi, a_lo, rows, nb, state_in=None, want_state=False, tag="rnn", ws=None):
    """All recurrent layers on packed rows; returns (h_hi, h_lo) of the last layer and the new state.
    ``ws``: workspace to use (ensembles share the first member's buffers; launches are stream-ordered)."""
    ws = ws or plan.ws
    H, nd = plan.hidden, plan.n_dirs
    if isinstance(sched, MixedSchedule):
        return _run_layers_mixed(model, plan, sched, a_hi, a_lo, rows, tag, ws)
    state_out = []
    rec_layers = plan.rec_layers
    if nb == 128 and plan.cell == CELL_GRU:  # the 128-slot GRU kernel takes gate-blocked rows
        rec_layers = gru_wide_layers(plan, model)
    for l, layer in enumerate(rec_layers):
        # input projection of every frame: fp32 in the fp32-accurate mode, bf16 in bf16 mode
        gate_cols = getattr(layer, "gate_cols", 4 * H)
        if plan.split:
            gx = ws.get(f"{tag}.gx", rows, nd * 4 * H, torch.float32)
            layer.upward(a_hi, a_lo, rows, "identity", OUT_F32, out=(gx, None))
        else:
            gx = ws.get(f"{tag}.gx16", rows, nd * gate_cols, plan.tdt)
            layer.upward(a_hi, a_lo, rows, "identity", plan.prec.out16, out=(gx, None))
        slot = l if want_state else l % 2  # a carried state needs every layer's h kept
        h_hi = ws.get(f"{tag}.h{slot}.hi", rows, nd * H, plan.tdt)
        h_lo = ws.get(f"{tag}.h{slot}.lo", rows, nd * H, torch.bfloat16) if plan.split else None
        h0 = c0 = c_out = None
        if state_in is not None:
            h0, c0 = state_in[l]
        if want_state and plan.cell == CELL_LSTM:
            c_out = torch.zeros((sched.n_batches * nb, nd * H), dtype=torch.float32, device=plan.device)
        # exchange buffer: per lane 4 slots (h parity 0/1, r*h parity 0/1) of nb rows x H; zeroed once when it is created
        x_rows = sched.n_lanes * 4 * nb
        fresh = ws.buf.get(f"{tag}.xchg.hi") is None or ws.buf[f"{tag}.xchg.hi"].numel() < x_rows * H
        xchg = (ws.get(f"{tag}.xchg.hi", x_rows, H, plan.tdt),
                ws.get(f"{tag}.xchg.lo", x_rows, H, torch.bfloat16) if plan.split else None)
        if fresh:
            xchg[0].zero_()
            if xchg[1] is not None:
                xchg[1].zero_()
        desc = _fill_desc(plan, sched, layer, gx, h_hi, h_lo, nb, h0, c0, c_out, xchg)
        # algorithmic lateral flops: LSTM 4 gates, GRU 3 (2 without reset gate) H x H products per frame
        n_mats = {CELL_LSTM: 4, CELL_PEEPHOLE: 7}.get(plan.cell, 3 if plan.gru_flags & 1 else 2)
        ops.rnn_seq(desc, 2.0 * rows * nd * n_mats * H * H)
        if want_state:
            state_out.append(((h_hi, h_lo), c_out))
        a_hi, a_lo = h_hi, h_lo
    return a_hi, a_lo, state_out


def _phase_split(lens):
    """Utterance subsets (indices into the shard, ascending) that are computed one after the other so that the
    device->host copy of a finished subset overlaps the computation of the next one.  Results only exist after the last
    layer, and a layer's time is set by its longest utterance, so the first subset takes the SHORTEST utterances (about
    30 % of the frames: quick to compute, and long enough on the wire to cover the second subset's computation).  Small
    shards and NNAM_RNN_PHASES=1 keep one subset."""
    n = len(lens)
    total = int(lens.sum())
    n_ph = int(os.environ.get("NNAM_RNN_PHASES", "2"))
    if n_ph <= 1 or n < 256 or total < 150000:
        return [np.arange(n)]
    by_len = np.argsort(lens, kind="stable")
    csum = np.cumsum(lens[by_len])
    cuts = [0.3] if n_ph == 2 else [0.15, 0.45]  # cumulative frame fractions at which a new subset starts
    bounds = [0]
    for c in cuts:
        k = int(np.searchsorted(csum, c * total))
        k = max(bounds[-1] + 128, min(k, n - 128))
        if k >= n - 127 or k <= bounds[-1]:
            break
        bounds.append(k)
    bounds.append(n)
    return [np.sort(by_len[a:b]) for a, b in zip(bounds[:-1], bounds[1:])]


def _forward_phase(models, plans, head, x_dev, iv_dev, add, mul, starts, lens, dest, timedelay, fix_timedelay_tail,
                   nb, device, stepwise, out_starts=None):
    """One subset of utterances (start frame relative to the shard and length of each) through the whole net:
    packed gather -> layers -> output GEMM -> head, which scatters the rows into the head destination ``dest`` (see
    engine.run_head) over all frames of the shard.  ``out_starts``: first OUTPUT row of every utterance when that
    differs from its first input frame (the compact format packs the rows of a subset one after the other)."""
    if out_starts is None:
        out_starts = starts
    plan = plans[0]
    ws = plan.ws
    split = plan.split
    if stepwise:  # time-step launches over ONE batch holding every utterance of the subset
        nb = len(lens)
        sched = Schedule(lens + timedelay, nb, 1, 1, device, 1)
    else:
        # members of one architecture (the usual fold ensemble) share the schedule, mixed or not; a heterogeneous
        # ensemble re-packs per architecture with a fixed batch width, which a mixed schedule does not have
        homog = all((p_.cell, p_.hidden, p_.n_dirs) == (plan.cell, plan.hidden, plan.n_dirs) for p_ in plans)
        sched, nb = pick_schedule(plan, lens + timedelay, device, nb, allow_mixed=homog)
    scheds = {(plan.cell, plan.hidden, plan.n_dirs): sched}
    rows = sched.n_rows
    # packed row -> source frame (edge-padded by `timedelay`) and -> destination frame (or -1); like the schedule
    # these maps depend only on where the utterances lie, and are cached with it
    maps = plan.__dict__.setdefault("_map_cache", {})
    mkey = (starts.tobytes(), lens.tobytes(), timedelay, bool(fix_timedelay_tail), nb,
            None if out_starts is starts else out_starts.tobytes())
    if mkey not in maps:
        utt = sched.order[sched.row_sorted_utt]  # utterance index inside the subset
        step = sched.row_step
        l_row = lens[utt]
        start = starts[utt]
        src = start + np.minimum(step, l_row - 1)
        dst = out_starts[utt] + step - timedelay
        keep = step >= timedelay
        dst = np.where(keep, dst, -1)
        if not fix_timedelay_tail:
            # predict_folds.py:50,60-61: rows are written only while utt_len > t (quirk Q4), so the last `timedelay`
            # frames of every utterance stay 0; the head zero-fills exactly those rows (entry -2 - row) and every
            # output row is written once -- no separate memset of the (N, C) matrix
            dst = np.where(keep & (step >= l_row), -2 - dst, dst)
        if len(maps) >= 8:
            maps.pop(next(iter(maps)))
        maps[mkey] = (torch.from_numpy(src.astype(np.int32)).to(device),
                      torch.from_numpy(dst.astype(np.int32)).to(device))
    d_src, d_dst = maps[mkey]

    d_in = models[0].in_size
    ld_in = round_up(d_in, 8)
    a_hi = ws.get("rnn.a.hi", rows, ld_in, plan.tdt)
    a_lo = ws.get("rnn.a.lo", rows, ld_in, torch.bfloat16) if split else None
    ops.gather_transform(x_dev, d_src, add, mul, iv_dev, out_kind=plan.act_kind, ldo=ld_in, out=(a_hi, a_lo))
    n_out = models[0].n_out
    logits = []
    fused = fused_head_ok(models, head, plans[0].out.k)
    for k, (m, pl) in enumerate(zip(models, plans)):
        key = (pl.cell, pl.hidden, pl.n_dirs)
        pl_stepwise = pl.cell == CELL_PEEPHOLE and not pl.peep_persistent
        if pl_stepwise != stepwise:
            raise NnamError("forward_utterances: time-step and persistent nets cannot share one ensemble pass")
        if pl_stepwise:
            from . import peephole_engine
            h_hi, h_lo = peephole_engine.run_layers(m, pl, sched, a_hi, a_lo, rows, ws=ws)
        else:
            if key not in scheds:  # same utterances and batch width => same packed row order, other grouping
                scheds[key], _ = pick_schedule(pl, lens + timedelay, device, nb)
            h_hi, h_lo, _ = run_layers(m, pl, scheds[key], a_hi, a_lo, rows, nb, ws=ws)
        if fused:
            break  # one member: its output layer runs fused with the head below
        lg = ws.get(f"rnn.logits{k}", rows, round_up(n_out, 16), torch.float32)
        pl.out(h_hi, h_lo, rows, "identity", OUT_F32, out=(lg, None))
        logits.append(lg)
    for u in np.nonzero(lens < timedelay)[0]:  # utterances shorter than the delay have rows no packed row maps to
        engine.zero_rows(dest, int(out_starts[u]), int(out_starts[u] + lens[u]))
    engine.run_head(head.device_args(device), dest, rows, out_row_map=d_dst, logits=logits, n_out=n_out,
                    fused=plans[0].out if fused else None, h=(h_hi, h_lo))


class _PackedDrainer:
    """Ships the packed compact rows of finished utterance subsets to the host on its own thread, so that the thread
    which launches kernels never blocks on the staging ring (launching one subset takes several ms of host time, and the
    previous subset's rows should be on the wire meanwhile).  The packed rows cross PCIe in pieces of a few thousand rows
    through a small ring of pinned buffers; engine._ChunkWriter's helper thread widens each piece into its frame
    positions of ``out`` while the piece is still in the last-level cache (as in the feed-forward path)."""

    def __init__(self, plan, out, out16, n_out, side, device, threads):
        import queue
        import threading
        stage = engine.staging_ring(plan, True, max(256, int(os.environ.get("NNAM_PIECE_ROWS", "4096"))), n_out)
        out_np = out.numpy() if isinstance(out, torch.Tensor) else out
        self.writer = engine._ChunkWriter(stage, True, out_np, None, n_out, threads)
        self.out16, self.side, self.device = out16, side, device
        self.err = None
        self.q = queue.Queue()
        self.thread = threading.Thread(target=self._run, name="nnam-drain", daemon=True)
        self.thread.start()

    def add(self, done, p0, dst_rows):
        self.q.put((done, p0, dst_rows))

    def _run(self):
        try:
            with torch.cuda.device(self.device):
                while True:
                    item = self.q.get()
                    if item is None:
                        return
                    if self.err is None:
                        self._drain(*item)
        except BaseException as e:  # noqa: BLE001 -- re-raised in close()
            self.err = e
            while self.q.get() is not None:
                pass

    def _drain(self, done, p0, dst_rows):
        self.side.wait_event(done)
        self.writer.ship(self.side, (self.out16[0][p0:], self.out16[1][p0:]), len(dst_rows), dst_rows)

    def close(self):
        self.q.put(None)
        self.thread.join()
        self.writer.close()
        if self.err is not None:
            raise self.err

    def abort(self):
        self.err = self.err or NnamError("aborted")
        self.q.put(None)
        self.thread.join()
        try:
            self.writer.close()
        except Exception:  # noqa: BLE001 -- the original error is the one to report
            pass


def forward_utterances(model, x, offsets, out, u0, u1, ft=None, ivectors=None, timedelay=0, device=0, head=None,
                       fix_timedelay_tail=False, nb=DEFAULT_BATCH, transfer=None, host_threads=None, score=None):
    """Recurrent hot path on ONE device for utterances [u0, u1) (predict_folds.py:28-68 semantics).

    model: one recurrent spec or a list of them (ensemble: the logits are combined in the head, evaluate.py:35-51).
    x / ivectors: (N, dim) / (N, I) float32, host arrays or CUDA tensors; out: (N, C) float32 host array or CUDA
    tensor, rows [offsets[u0], offsets[u1]) are written.  Output frame f of an utterance is the network output at
    step f + timedelay; like the reference, the last ``timedelay`` frames stay 0 unless fix_timedelay_tail.
    With a host ``out`` a large shard is computed in two subsets of utterances (:func:`_phase_split`) and the copy of
    the first one to the host runs under the computation of the second.  ``transfer`` / ``host_threads``: as in
    engine.ff_forward_frames -- in the 16-bit modes the rows cross PCIe in the compact format (fp16 offsets from the row
    maximum) into a pinned staging area and host threads widen them into ``out`` while the GPU computes the next subset.
    ``score``: (targets, nll, pred) host arrays of shape (N,) to score the rows against their targets instead of writing
    them (``out`` is None then), as in engine.ff_forward_frames.  The targets go up once per shard in frame order (the
    kernels index them by output row, so the packed order needs no gather); the utterance subsets, schedules and kernel
    choices are those of a host ``out``, and 8 B per frame come back at the end of the shard.
    """
    models = list(model) if isinstance(model, (list, tuple)) else [model]
    device = _device(device)
    head = head or HeadSpec()
    offsets = np.asarray(offsets, dtype=np.int64)
    if u1 <= u0:
        return out
    f_lo, f_hi = int(offsets[u0]), int(offsets[u1])
    lens = (offsets[u0 + 1:u1 + 1] - offsets[u0:u1]).astype(np.int64)
    starts = (offsets[u0:u1] - f_lo).astype(np.int64)
    if np.any(lens <= 0):
        raise NnamError("forward_utterances: empty utterance in offsets")
    with torch.cuda.device(device):
        plans = [get_plan(m, device) for m in models]
        engine.check_ensemble(models, plans, "forward_utterances: ")
        plan = plans[0]
        ws = plan.ws
        stepwise = plan.cell == CELL_PEEPHOLE and not plan.peep_persistent

        if isinstance(x, torch.Tensor) and x.is_cuda:
            x_dev = x[f_lo:f_hi]
        else:
            x_dev = ws.get("rnn.x", f_hi - f_lo, x.shape[1], torch.float32)
            x_dev.copy_(_as_host_tensor(x)[f_lo:f_hi], non_blocking=True)
        iv_dev = None
        if ivectors is not None:
            if isinstance(ivectors, torch.Tensor) and ivectors.is_cuda:
                iv_dev = ivectors[f_lo:f_hi]
            else:
                iv_dev = ws.get("rnn.iv", f_hi - f_lo, ivectors.shape[1], torch.float32)
                iv_dev.copy_(_as_host_tensor(ivectors)[f_lo:f_hi], non_blocking=True)
        add = mul = None
        if ft is not None:
            add, mul = _dev_vec(ft["addShift"], device), _dev_vec(ft["rescale"], device)
            if add.numel() != x.shape[1]:
                raise NnamError("forward_utterances: recurrent nets take the shift-0 transform block (adapt_transform)")
        d_in = models[0].in_size
        if d_in != x.shape[1] + (0 if ivectors is None else ivectors.shape[1]):
            raise NnamError(f"forward_utterances: model expects {d_in} inputs, data provides "
                            f"{x.shape[1] + (0 if ivectors is None else ivectors.shape[1])}")
        n_out = models[0].n_out
        on_dev = isinstance(out, torch.Tensor) and out.is_cuda
        n_rows = f_hi - f_lo
        if score is not None and out is not None:
            raise NnamError("forward_utterances: a scoring pass writes no rows (out must be None)")
        compact = (not on_dev and score is None) and engine.use_compact_transfer(plan, transfer, recurrent=True,
                                                                                 host_threads=host_threads)
        if score is not None:
            sc_dev = engine.score_buffers(ws, "rnn", score[0], f_lo, f_hi)
            dest = {"score": sc_dev}
        elif compact:
            out16 = (ws.get("rnn.out16", n_rows, round_up(n_out, 8), torch.float16),
                     ws.get("rnn.ref", n_rows, 1, torch.float32).view(-1))
            dest = {"out16": out16}
        else:
            out_dev = out[f_lo:f_hi] if on_dev else ws.get("rnn.out", n_rows, n_out, torch.float32)
            dest = {"out": out_dev}
        phases = [np.arange(len(lens))] if (on_dev or stepwise) else _phase_split(lens)
        main = torch.cuda.current_stream()
        side = None
        drainer = None  # compact: helper thread that ships finished subsets while this thread launches the next one
        packed = 0
        try:
            for idx in phases:
                whole = len(idx) == len(lens)
                p_starts, p_lens = (starts, lens) if whole else (starts[idx], lens[idx])
                # compact format: the rows of this subset are packed one utterance after the other, so that they cross PCIe
                # as ONE contiguous block (a subset's utterances lie all over the shard); the host scatters them back
                o_starts = None
                if compact:
                    o_starts = packed + np.concatenate([[0], np.cumsum(p_lens[:-1])]).astype(np.int64)
                _forward_phase(models, plans, head, x_dev, iv_dev, add, mul, p_starts, p_lens, dest, timedelay,
                               fix_timedelay_tail, nb, device, stepwise, out_starts=o_starts)
                if on_dev or score is not None:
                    continue
                out_host = None if compact else _as_host_tensor(out)
                if len(phases) == 1 and not compact:
                    out_host[f_lo:f_hi].copy_(out_dev, non_blocking=True)
                    continue
                if side is None:
                    side = plan.__dict__.get("_d2h_stream")
                    if side is None:
                        side = plan._d2h_stream = torch.cuda.Stream()
                done = torch.cuda.Event()
                done.record(main)
                if compact:
                    n_p = int(p_lens.sum())
                    dst_rows = f_lo + np.repeat(p_starts - np.concatenate([[0], np.cumsum(p_lens[:-1])]), p_lens) + np.arange(n_p)
                    if drainer is None:
                        drainer = _PackedDrainer(plan, out, out16, n_out, side, device,
                                                 host_threads or engine.default_host_threads())
                    drainer.add(done, packed, dst_rows.astype(np.int64))
                    packed += n_p
                    continue
                # rows of this subset, as maximal runs of neighbouring utterances, on the copy stream
                brk = np.nonzero(np.diff(idx) != 1)[0] + 1
                with torch.cuda.stream(side):
                    side.wait_event(done)
                    for run in np.split(idx, brk):
                        r0, r1 = int(starts[run[0]]), int(starts[run[-1]] + lens[run[-1]])
                        out_host[f_lo + r0:f_lo + r1].copy_(out_dev[r0:r1], non_blocking=True)
            if drainer is not None:
                drainer.close()
                drainer = None
        finally:
            if drainer is not None:  # an error above: let the helper thread go
                drainer.abort()
        if score is not None:
            engine.download_scores(sc_dev, score, f_lo, f_hi)
        main.synchronize()
        if side is not None:
            side.synchronize()
    return out


def step(model, plan, xd):
    """Stateful ``model(x)`` for recurrent specs: one time step for a batch of B rows
    (chainer_networks.py:58-62); ``reset_state()`` clears the carried (h, c)."""
    if plan.cell == CELL_PEEPHOLE:
        from . import peephole_engine
        return peephole_engine.step(model, plan, xd)
    B = xd.shape[0]
    nb = 32
    split = plan.split
    if model.bidirectional:
        raise NnamError("bidirectional models have no per-step form; use predict()/forward_utterances()")
    _, max_groups, _, streams = ops.rnn_plan(plan.cell, plan.hidden, nb, 3 if split else 1)
    st = model._state
    if st is not None and st["B"] != B:
        raise NnamError("model(x): batch size changed between steps; call reset_state() first")
    sched = st["sched"] if st is not None else Schedule(np.ones(B, np.int64), nb, 1, max_groups, plan.device, streams)
    a_hi, a_lo = ops.convert_f32(xd.contiguous(), plan.act_kind)
    h_hi, h_lo, new = run_layers(model, plan, sched, a_hi, a_lo, B, nb, state_in=None if st is None else st["s"],
                                 want_state=True, tag="step")
    # carry state: all lengths are 1 and the sort is stable, so packed rows == sorted order == input order.
    # The h buffers are workspace memory that the next call overwrites while reading -> keep private copies.
    new_state = [((hh.clone(), None if hl is None else hl.clone()), c) for (hh, hl), c in new]
    model._state = {"B": B, "sched": sched, "s": new_state}
    logits = plan.ws.get("step.logits", B, round_up(model.n_out, 16), torch.float32)
    plan.out(h_hi, h_lo, B, "identity", OUT_F32, out=(logits, None))
    return logits[:B, :model.n_out].clone()
