#!/usr/bin/env python3
"""Headline benchmark: acoustic-model frames/sec of the network-output hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg1|cfg3|cfg4|...]
                  [--precision fp16|bf16|fp32]

A "step" is one pass of the hot path (splice/transform -> network -> log-softmax head) over one synthetic data set.
Default workload = BASELINE.json configs[1]: 6x2048 ReLU MLP on 440 spliced fMLLR + 100-dim i-vectors -> 1909 pdfs,
TIMIT-train-shaped set (3696 utterances, 1,124,823 frames), 16-bit tcgen05 GEMMs.  Default precision "fp16": the
single-pass 16-bit mode that meets north_star's parity gate (<= 5e-2 max-abs AND >= 99.5 % raw frame-argmax agreement
with the fp32 forward; single-pass bf16 does not -- DESIGN.md section 3); same kind::f16 tensor-pipe rate as bf16.

  value      frames/s with the inputs already resident in HBM and the outputs left in HBM (CUDA events)
  e2e        frames/s through the public predict() with pinned HOST buffers: H2D of features / i-vectors and D2H of the
             (N, 1909) fp32 log-likelihoods inside the timed region; beside it the box's measured D2H ceiling
  N > 1      "value"/"e2e": weak scaling, every rank its own full-size set (the driver's contract);
             "strong": ONE set split by offset ranges across the ranks (the product's sharded path, SURVEY 8e), with a
             bit-identity check of every shard's sampled rows against rank 0's single-GPU pass
  parity     (N = 1) max-abs / raw argmax agreement of the device output against the CPU baseline leg's output
  --impl reference   the reference's CPU forward (NumPy restatement = what Chainer's CPU backend executes; Chainer
             itself is not installable offline), ALL host cores, on a bounded sample of the workload
  --dump-outputs DIR writes DIR/log_likelihoods.npy: float32 rows of the device-resident leg's (N, 1909) output after
             its last timed step -- all of them, or a fixed seeded sample of DUMP_ROWS when N is larger -- so that two
             builds run with the same arguments (same seeded inputs and weights) can be compared output for output

The product arm builds its workload, weights and transform through the package only (nnacousticmodeling_b200.synth,
Network.init_params, loadKaldiFeatureTransform); oracle/ is imported by the cpu_baseline / reference legs alone.
"""
from __future__ import annotations

import os
import sys

if "reference" in sys.argv or "--cpu-threads-all" in sys.argv:
    # torch.distributed.run exports OMP_NUM_THREADS=1 when nproc > 1; the reference arm is ONE process (rank 0) that
    # must use every host core, and OpenBLAS reads these when NumPy is imported
    for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_k] = str(os.cpu_count() or 1)

import argparse  # noqa: E402
import importlib  # noqa: E402
import json  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_CLASSES = 1909
TRAIN_UTTS, TRAIN_FRAMES = 3696, 1124823
TEST_UTTS = 1344
GOLDEN = os.path.join(ROOT, "tests", "golden")
DUMP_ROWS = 8192  # x 1909 float32 = 62.5 MB, within the 64 MB that --dump-outputs may write

WORKLOADS = {
    # name: network, i-vector dim, units, layers, set, algorithmic flop/frame (SURVEY 8d)
    "cfg1": dict(network="ff", ivec=0, units=1024, layers=6, utts=TEST_UTTS, frames=None, flop=15296512,
                 desc="cfg1: 6x1024 ReLU MLP, 440 spliced fMLLR -> 1909, test-shaped 1344 utts"),
    "cfg2": dict(network="ff", ivec=100, units=2048, layers=6, utts=TRAIN_UTTS, frames=TRAIN_FRAMES, flop=51974144,
                 desc="cfg2: 6x2048 ReLU MLP, 440 spliced fMLLR + 100 i-vector -> 1909, train-shaped 3696 utts / 1,124,823 frames"),
    "cfg3": dict(network="lstm", ivec=0, units=512, layers=4, utts=TEST_UTTS, frames=None, flop=16798720,
                 desc="cfg3: 4x512 LSTM, 40 fMLLR -> 1909, timedelay 5, test-shaped 1344 utts"),
    "cfg3t": dict(network="lstm", ivec=0, units=512, layers=4, utts=TRAIN_UTTS, frames=TRAIN_FRAMES, flop=16798720,
                  desc="cfg3t: 4x512 LSTM, 40 fMLLR -> 1909, timedelay 5, train-shaped 3696 utts / 1,124,823 frames"),
    "cfg4": dict(network="blstm", ivec=100, units=512, layers=4, utts=TEST_UTTS, frames=None, flop=46999552,
                 desc="cfg4: 4x(2x512) bidirectional LSTM, 40 fMLLR + 100 i-vector -> 1909, test-shaped 1344 utts"),
    "cfg4g": dict(network="bgru", ivec=100, units=512, layers=4, utts=TEST_UTTS, frames=None,
                  flop=2 * (2 * (140 * 1536 + 512 * 1536) + 3 * 2 * (1024 * 1536 + 512 * 1536) + 1024 * 1909),
                  desc="cfg4g: 4x(2x512) bidirectional GRU, 40 fMLLR + 100 i-vector -> 1909, test-shaped 1344 utts"),
    # cfg5: ensembles of 10 fold models, logit mean fused into the head (evaluate.py:35-51)
    "cfg5": dict(network="ff", ivec=0, units=1024, layers=6, utts=TEST_UTTS, frames=None, flop=10 * 15296512, folds=10,
                 desc="cfg5: ensemble of 10 fold 6x1024 MLPs (logit mean), 440 spliced fMLLR -> 1909, test-shaped 1344 utts"),
    "cfg5b": dict(network="blstm", ivec=100, units=512, layers=4, utts=TEST_UTTS, frames=None, flop=10 * 46999552,
                  folds=10,
                  desc="cfg5b: ensemble of 10 fold 4x(2x512) BLSTMs (logit mean), 40 fMLLR + 100 i-vector -> 1909, test-shaped 1344 utts"),
}


def host_info():
    """CPU model / core count / L3 size of the box: the end-to-end leg is bound by the host (PCIe ingest, then the memory
    system of the widening threads), and the pod's boxes differ."""
    info = {"cores": os.cpu_count()}
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                info["cpu"] = ln.split(":", 1)[1].strip()
                break
        info["l3"] = open("/sys/devices/system/cpu/cpu0/cache/index3/size").read().strip()
    except OSError:
        pass
    return info


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


# ------------------------------------------------------------------------------------------ workload (product side)
def make_workload(name, rank=0):
    """(spec, x, offsets, ivectors) of a synthetic set; rank r of a weak-scaling run gets its own seed."""
    from nnacousticmodeling_b200 import synth
    w = WORKLOADS[name]
    x, offsets, iv = synth.synth_set(1234 + 17 * rank, w["utts"], 40, w["ivec"], total=w["frames"])
    return w, x, offsets, iv


def make_models(w, precision, device):
    """Random-init members (Chainer default initialisers) of the workload's net: one model, or the folds of an ensemble."""
    import nnacousticmodeling_b200 as nn
    net = w["network"]
    d_in = (440 if net == "ff" else 40) + w["ivec"]
    members = []
    for k in range(w.get("folds", 1)):
        m = nn.get_nn(net, w["layers"], [w["units"]], N_CLASSES, nn.F.relu, [5])
        m.init_params(d_in, np.random.default_rng(4321 + k))
        m.precision = precision
        m.to_gpu(device)
        members.append(m)
    return members


def make_params(w, seed=4321):
    """Oracle-side random-init parameters (tests/tools/gpu_parity_table.py, the reference arm; NOT the product arm)."""
    from oracle import nnam_oracle as O
    rng = np.random.default_rng(seed)
    if w["network"] == "ff":
        return O.init_mlp(rng, 440 + w["ivec"], w["units"], w["layers"], N_CLASSES)
    bid = w["network"] in ("blstm", "bgru")
    cell = "gru" if w["network"] == "bgru" else "lstm"
    return O.init_recurrent(rng, cell, 40 + w["ivec"], w["units"], w["layers"], N_CLASSES, bidirectional=bid)


# --------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock, power and throttle reasons through NVML in a background thread DURING the timed
    region (same data as the nvidia-smi clocks line of the profiling recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.thread, self.err = index, [], False, None, None

    def _handle(self, nv):
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            return nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:  # noqa: BLE001
            return nv.nvmlDeviceGetHandleByIndex(self.index)

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = self._handle(nv)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            while not self.stop_flag:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:  # noqa: BLE001
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((sm, mx, pw, rs))
                time.sleep(0.02)
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def start(self):
        import threading
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=5)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples: " + str(self.err)]}
        bits = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        reasons = set()
        for r in self.rows:
            for b, n in bits.items():
                if r[3] & b:
                    reasons.add(n)
        sm = [r[0] for r in self.rows]
        return {"sm_mhz": float(np.median(sm)), "sm_min_mhz": float(min(sm)), "sm_max_mhz": float(self.rows[0][1]),
                "reasons": sorted(reasons), "power_w_max": float(max(r[2] for r in self.rows)), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU baseline (oracle port)
def cpu_reference_rate(wname, sample_frames, params_list, x, offsets, iv, steps=1, warmup=0, with_python_prepare=False):
    """Frames/s of the reference-equivalent NumPy CPU forward (oracle port) on a bounded sample, with the reference's
    own control flow (predict_folds.py:27-95).  Returns (rate, seconds, sample description, frames, (rows, output)).

    FF: the first ``n`` frames through predict()'s 1024-frame loop.  ``with_python_prepare`` times the reference's
    per-frame Python splice loop (kw_nn_utils.py:26-36, restated) instead of the oracle's vectorised one -- BASELINE.md
    section 3 asks for both figures.  RNN: a LENGTH-STRATIFIED sample of utterances through the time-major loop, as
    wide as the budget allows (the reference batches every utterance of the set per step)."""
    from oracle import nnam_oracle as O
    w = WORKLOADS[wname]
    folds = len(params_list)
    p = params_list[0]
    ft = O.load_kaldi_feature_transform(os.path.join(GOLDEN, "final.feature_transform"))
    if folds > 1:
        sample_frames = max(sample_frames // folds, 2048)
    if w["network"] == "ff":
        n = int(min(sample_frames, len(x)))
        xs, ivs = x[:n], (iv[:n] if iv is not None else None)

        def prepare(o, e):
            if not with_python_prepare:
                return O.prepare_batch(xs, np.arange(o, e), 11)
            out = np.zeros((e - o, 440), dtype=np.float32)  # kw_nn_utils.py:26-36: one Python iteration per frame
            for k, i in enumerate(range(o, e)):
                lo, hi = i - 5, i + 6
                if lo < 0 or hi > n:
                    out[k] = xs[np.clip(np.arange(lo, hi), 0, n - 1)].flatten()
                else:
                    out[k] = xs[lo:hi].flatten()
            return out

        def run():
            ys = []
            for o in range(0, n, 1024):  # predict_folds.predict FF loop (batch 1024), train/evaluate feature order
                e = min(o + 1024, n)
                f = O.apply_kaldi_feature_transform(prepare(o, e), ft)
                if ivs is not None:
                    f = np.concatenate((f, ivs[o:e]), axis=1)
                if folds > 1:  # evaluate.py:35-51: mean of the fold logits, then log-softmax
                    ys.append(O.log_softmax(O.nn_with_rpl(None, [(lambda v, q=q: O.mlp_forward(q, v, w["layers"]))
                                                                 for q in params_list], None, f)))
                else:
                    ys.append(O.log_softmax(O.mlp_forward(p, f, w["layers"])))
            return np.concatenate(ys)
        # the last 5 sampled frames see a clamp the full set does not have: keep them out of the parity comparison
        rows = np.arange(max(n - 5, 0)) if n < len(x) else np.arange(n)
        sample = (f"first {n} frames, predict() FF loop batch 1024, "
                  + ("per-frame Python prepareBatch" if with_python_prepare else "vectorised prepare_batch"))
    else:
        bid = w["network"] in ("blstm", "bgru")
        cell = "gru" if w["network"] == "bgru" else "lstm"
        lens = np.diff(offsets)
        n_utt = int(min(max(sample_frames // 300, 16), len(lens)))
        if bid:  # no batched reference loop exists for the bidirectional nets: per-utterance, so a smaller sample
            n_utt = max(n_utt // 16, 8) if folds == 1 else max(n_utt // (16 * folds), 2)
        # every (U / n_utt)-th utterance of the length-sorted set: same length distribution (padding waste) as the set
        order = np.argsort(lens, kind="stable")
        pick = np.sort(order[np.linspace(0, len(lens) - 1, n_utt).round().astype(int)])
        sub = np.concatenate([[0], np.cumsum(lens[pick])])
        n = int(sub[-1])
        rows = np.concatenate([np.arange(offsets[u], offsets[u + 1]) for u in pick])
        ftm = O.select_transform_for_network(ft, "lstm")
        xs = x[rows] if iv is None else np.concatenate((O.apply_kaldi_feature_transform(x[rows], ftm), iv[rows]), axis=1)
        td = 5 if w["network"] == "lstm" else 0

        def run():
            if bid:
                return np.concatenate([O.log_softmax(sum(O.birnn_forward_utterance(q, cell, w["layers"], xs[sub[i]:sub[i + 1]])
                                                         for q in params_list) / np.float32(folds)) for i in range(n_utt)])
            net = O.RecurrentNet(p, w["network"], w["layers"])
            return O.predict(net, xs, sub, w["network"], 1, td, ftm if iv is None else None)
        sample = (f"{n_utt} utterances stratified by length ({n} frames), "
                  + ("per-utterance bidirectional forward" if bid else f"time-major loop, {n_utt} rows per step"))
    for _ in range(warmup):
        run()
    t0 = time.perf_counter()
    for _ in range(steps):
        y = run()
    dt = (time.perf_counter() - t0) / steps
    return n / dt, dt, sample, n, (rows, y[:len(rows)])


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    try:
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=os.cpu_count())  # in case the BLAS was initialised with fewer threads
    except Exception:  # noqa: BLE001
        pass
    w, x, offsets, iv = make_workload(args.workload, 0)
    params = [make_params(w, 4321 + k) for k in range(w.get("folds", 1))]
    rate, dt, sample, n, _ = cpu_reference_rate(args.workload, args.cpu_sample, params, x, offsets, iv,
                                                steps=max(args.steps, 1), warmup=min(args.warmup, 1))
    cores = os.cpu_count()
    line = {
        "impl": "reference", "metric": "acoustic-model frames/sec", "value": rate, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["desc"], "sample": sample},
        "cpu_baseline": {"value": rate, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample,
                         "blas_threads": os.environ.get("OMP_NUM_THREADS"),
                         "note": "NumPy/OpenBLAS restatement of the Chainer CPU forward (Chainer 3.5 not installable "
                                 "offline), pinned to outputs of the reference's own code (tests/golden/nets)"},
        "e2e": {"value": rate, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------ product arm
class Bench:
    """One workload on one rank: models, host / device buffers and the timed legs."""

    def __init__(self, wname, precision, local, data_rank):
        import torch
        import nnacousticmodeling_b200 as nn
        self.torch, self.nn, self.wname = torch, nn, wname
        self.local = local
        self.dev = torch.device("cuda", local)
        self.w, self.x, self.offsets, self.iv = make_workload(wname, data_rank)
        self.n = len(self.x)
        self.net = self.w["network"]
        self.recurrent = nn.is_nn_recurrent(self.net)
        self.members = make_models(self.w, precision, local)
        folds = len(self.members)
        self.model = self.members[0] if folds == 1 else self.members
        self.head = None if folds == 1 else nn.HeadSpec(weights=[1.0 / folds] * folds)
        self.ft = nn.adapt_transform(nn.loadKaldiFeatureTransform(os.path.join(GOLDEN, "final.feature_transform")),
                                     self.net, 5, self.recurrent)
        self.timedelay = 5 if self.net == "lstm" else 0
        self.xp = nn.empty_pinned(self.x.shape)
        self.xp[:] = self.x
        self.ivp = None
        if self.iv is not None:
            self.ivp = nn.empty_pinned(self.iv.shape)
            self.ivp[:] = self.iv
        self.out_host = nn.empty_pinned((self.n, N_CLASSES))
        self.x_dev = torch.from_numpy(self.xp).to(self.dev)
        self.iv_dev = None if self.ivp is None else torch.from_numpy(self.ivp).to(self.dev)
        self.out_dev = torch.empty((self.n, N_CLASSES), dtype=torch.float32, device=self.dev)

    # -- one pass over the set (or over one rank's shard of it), inputs and outputs resident in HBM
    def step_device(self, shard=None):
        from nnacousticmodeling_b200 import engine, recurrent_engine
        if self.recurrent:
            u0, u1 = (0, len(self.offsets) - 1) if shard is None else shard[:2]
            recurrent_engine.forward_utterances(self.model, self.x_dev, self.offsets, self.out_dev, u0, u1, ft=self.ft,
                                                ivectors=self.iv_dev, timedelay=self.timedelay, device=self.local,
                                                head=self.head)
        else:
            f0, f1 = (0, self.n) if shard is None else shard[2:]
            engine.ff_forward_frames(self.model, self.x_dev, self.ft, 5, self.out_dev, f0, f1, ivectors=self.iv_dev,
                                     device=self.local, head=self.head)

    # -- the public call with pinned host buffers (H2D + D2H inside)
    def step_e2e(self, shard=None):
        from nnacousticmodeling_b200 import engine, recurrent_engine
        if shard is None:
            self.nn.predict(self.model, self.xp, self.offsets if self.recurrent else None, N_CLASSES, self.net,
                            self.local, 11, self.timedelay, self.ft, progress=False, ivectors=self.ivp,
                            out=self.out_host, head=self.head)
        elif self.recurrent:  # what predict(gpu=[...]) runs per device (predict.py): this rank's utterance range
            recurrent_engine.forward_utterances(self.model, self.xp, self.offsets, self.out_host, shard[0], shard[1],
                                                ft=self.ft, ivectors=self.ivp, timedelay=self.timedelay,
                                                device=self.local, head=self.head)
        else:
            engine.ff_forward_frames(self.model, self.xp, self.ft, 5, self.out_host, shard[2], shard[3],
                                     ivectors=self.ivp, device=self.local, head=self.head)


def dump_rows(n):
    """Output rows written by --dump-outputs: every row, or the same seeded sample of DUMP_ROWS rows on every run."""
    if n <= DUMP_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))


def timed_device(torch, fn, steps, barrier):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(steps):
        fn()
    ev1.record()
    barrier()
    return ev0.elapsed_time(ev1) / steps


def timed_host(torch, fn, steps, barrier):
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    barrier()
    return dt


def d2h_ceiling(torch, dev, barrier, max_over_ranks, world, gib=1, blocks=4, reps=3):
    """Measured device->pinned-host copy rate with every rank copying at once (cudaMemcpyAsync of 1 GiB blocks): the
    ceiling of the e2e leg, whose timed region moves 7,636 B/frame over PCIe into one host's DRAM."""
    n = gib << 30
    src = torch.empty(n, dtype=torch.uint8, device=dev)
    dst = [torch.empty(n, dtype=torch.uint8, pin_memory=True) for _ in range(blocks)]
    for d in dst:
        d.copy_(src, non_blocking=True)  # touch the pages
    torch.cuda.synchronize()
    best = 0.0
    for _ in range(reps):
        barrier()
        t0 = time.perf_counter()
        for d in dst:
            d.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        best = max(best, world * blocks * n / dt / 1e9)
    del src, dst
    return best


def kernel_table(prof, steps):
    kern = {}
    for name, s, e, work in prof:
        k = kern.setdefault(name, {"launches": 0, "ms": 0.0, "work": 0.0})
        k["launches"] += 1
        k["ms"] += s.elapsed_time(e)
        k["work"] += work
    for name, k in kern.items():
        k["ms_per_step"] = k["ms"] / steps
        if name in ("gemm", "rnn"):
            k["tflops"] = k["work"] / (k["ms"] * 1e-3) / 1e12
        else:
            k["gbs"] = k["work"] / (k["ms"] * 1e-3) / 1e9
        del k["work"], k["ms"]
    return kern


def roofline_block(kern, peaks, wname, steps):
    dom = max(kern, key=lambda a: kern[a]["ms_per_step"])
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(f"{wname}:{dom}")
    if dom in ("gemm", "rnn"):
        roof = {"bound": "tensor", "kernel": ("gemm_bias_act_2sm_kernel + gemm_bias_act_kernel (+ gemm_logsoftmax_kernel where the output layer runs fused with the head: K <= 1024)"
                           if dom == "gemm" else "rnn_seq_kernel"),
                "achieved": kern[dom]["tflops"], "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                "frac": kern[dom]["tflops"] / peaks["tf_sustained"], "traffic": traffic,
                "peak_source": f"{peaks['src']} 16-bit dense sustained (kernel timed inside a long step); burst peak "
                               f"{peaks['tf_burst']} -> frac {kern[dom]['tflops'] / peaks['tf_burst']:.3f}",
                "launches_per_step": kern[dom]["launches"] // steps}
        if dom == "rnn":
            roof["note"] = ("K3 is sequential in t and bound by the per-step exchange latency, not by the tensor pipe "
                            "(SURVEY 8d: no roofline claim); achieved = algorithmic lateral FLOP / kernel time")
    else:
        roof = {"bound": "hbm", "kernel": dom, "achieved": kern[dom]["gbs"], "peak": peaks["hbm"], "unit": "GB/s",
                "frac": kern[dom]["gbs"] / peaks["hbm"], "traffic": traffic, "peak_source": peaks["src"]}
    return roof


def cli_wall_clock(b, precision):
    """Wall clock of the drop-in CLI (predict.main, fold mode) on the same workload: np.load of the inputs, model load,
    the pass, and the streamed .npy output -- what a master_script.py run of this step pays."""
    import shutil
    import tempfile
    nn = b.nn
    need = b.n * N_CLASSES * 4 + b.x.nbytes + (0 if b.iv is None else b.iv.nbytes) + (1 << 30)
    base = None
    for cand in ("/dev/shm", tempfile.gettempdir()):
        try:
            if shutil.disk_usage(cand).free > need:
                base = cand
                break
        except OSError:
            continue
    if base is None or isinstance(b.model, list):
        return {"skipped": "no scratch space for the output file" if base is None else "single-model workloads only"}
    root = tempfile.mkdtemp(prefix="nnam_cli_", dir=base)
    try:
        os.makedirs(os.path.join(root, "data"))
        shutil.copy(os.path.join(GOLDEN, "final.feature_transform"), os.path.join(root, "data"))
        np.save(os.path.join(root, "data_0.npy"), b.x)
        np.save(os.path.join(root, "offsets_0.npy"), b.offsets)
        cmd = ["--tri", "--ft", "final.feature_transform", "--data-dir", os.path.join(root, "data"), "--fold-data-dir", root,
               "--fold-output-dir", os.path.join(root, "out"), "--fold-model-dir", root, "-n", b.net, "-l", b.w["layers"],
               "-u", b.w["units"], "-d", 0, "--no-progress", "--precision", precision, "--gpu", b.local]
        if not b.recurrent:
            cmd += ["--splice", 5]
        if b.timedelay:
            cmd += ["--timedelay", b.timedelay]
        if b.iv is not None:
            np.save(os.path.join(root, "ivectors_0.npy"), b.iv)
            cmd += ["--ivector-dir", root]
        nn.save_npz(os.path.join(root, "fold_0.npz"), nn.Classifier(b.model))
        cli = importlib.import_module("nnacousticmodeling_b200.predict")
        t0 = time.perf_counter()
        cli.main(cmd)
        dt = time.perf_counter() - t0
        size = os.path.getsize(os.path.join(root, "out", "data_0.npy"))
        return {"seconds": dt, "frames_per_s": b.n / dt, "output_bytes": size, "scratch": base}
    finally:
        shutil.rmtree(root, ignore_errors=True)


def run_ours(args):
    import torch
    from nnacousticmodeling_b200 import dist_util, ops

    world, rank, local = dist_util.env_world()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist_util.init("nccl", dev)
    numa_cpus = dist_util.bind_to_gpu_numa(local) if world > 1 else None  # before the pinned buffers are allocated
    peaks = load_peaks()
    steps, warmup = args.steps, max(args.warmup, 3)

    def barrier():
        torch.cuda.synchronize()
        dist_util.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        return dist_util.max_over_ranks(v, dev)

    b = Bench(args.workload, args.precision, local, data_rank=rank)
    w, n = b.w, b.n

    # ---- device-resident leg ("value"): inputs in HBM, outputs left in HBM, CUDA events, weak scaling over ranks
    for _ in range(warmup):
        b.step_device()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = sum(ops.LAUNCHES.values())
    ops.PROFILE = []
    dev_ms = max_over_ranks(timed_device(torch, b.step_device, steps, barrier))
    clocks = sampler.stop()
    prof, ops.PROFILE = ops.PROFILE, None
    launches = sum(ops.LAUNCHES.values()) - launches0
    value = world * n / (dev_ms * 1e-3)
    # taken now: the legs below write other results into out_dev
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = b.out_dev[torch.from_numpy(dump_rows(n)).to(dev)].cpu().numpy()
    kern = kernel_table(prof, steps)
    roof = roofline_block(kern, peaks, args.workload, steps)

    # ---- end-to-end leg: public predict() with pinned host buffers, H2D + D2H inside the timed region
    h2d = b.x.nbytes + (0 if b.iv is None else b.iv.nbytes)
    d2h = n * N_CLASSES * 4
    if args.no_e2e:  # profiling runs only (ncu): the printed line is then not a bench value
        e2e = {"value": None, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h}
    else:
        for _ in range(4):  # also lets the transfer mix settle (engine._TransferStats probes during these passes)
            barrier()       # ranks share the host: measure the candidates with every rank running
            b.step_e2e()
        e2e_s = max_over_ranks(timed_host(torch, b.step_e2e, steps, barrier))
        from nnacousticmodeling_b200 import engine
        plan0 = engine.get_plan(b.members[0], local)
        compact = engine.use_compact_transfer(plan0, recurrent=b.recurrent, mixable=True)
        stats = plan0.__dict__.get("_xfer_stats")
        if compact and stats is not None and stats.last_d2h_bytes:  # counted from the copies of the last pass
            d2h = int(stats.last_d2h_bytes)
        elif compact:  # fp16 offsets (rows padded to 8 columns) + one float32 maximum per row
            d2h = n * ((N_CLASSES + 7) // 8 * 8 * 2 + 4)
        host_vs_dev = float((torch.from_numpy(b.out_host[:65536]).to(dev) - b.out_dev[:65536]).abs().max())
        ceiling = d2h_ceiling(torch, dev, barrier, max_over_ranks, world)
        achieved = world * d2h / e2e_s / 1e9
        e2e = {"value": world * n / e2e_s, "unit": "frames/s", "ms_per_step": e2e_s * 1e3, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "host_output_bytes_per_step": n * N_CLASSES * 4,
               "transfer": ((f"mixed: {stats.current:.2f} of the chunks compact (fp16 offsets from the row maximum "
                             f"+ the maximum, widened to the float32 (N, 1909) layout by host threads), the rest float32 "
                             f"rows; measured PCIe {stats.pcie / 1e9:.1f} GB/s, widening {stats.widen / 1e9:.1f} GB/s")
                            if (compact and stats is not None) else
                            ("compact: fp16 offsets from the row maximum + the maximum, widened to the float32 (N, 1909) "
                             "layout by host threads" if compact else "float32 rows")),
               "host_threads": engine.default_host_threads() if compact else 0,
               "probed_compact_fractions": ({f"{k:.3f}": round(v) for k, v in stats.tried.items()}
                                            if (compact and stats is not None and stats.tried) else None),
               "max_abs_host_vs_device_leg": host_vs_dev,
               "d2h": {"achieved_gbs": achieved, "ceiling_gbs": ceiling, "frac": achieved / ceiling,
                       "how": f"{world} rank(s) x cudaMemcpyAsync device -> pinned host, 4 x 1 GiB, best of 3; "
                              "achieved = output bytes / whole e2e step (compute and H2D included)"}}

    line = {
        "metric": "acoustic-model frames/sec", "value": value, "unit": "frames/s", "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": dev_ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "bf16x3(fp32-accurate)"}.get(args.precision, args.precision),
        "data": "synthetic",
        "config": {"workload": w["desc"], "frames_per_gpu": n, "precision": args.precision,
                   "l2": "inputs+activations larger than L2 (no flush needed)",
                   "parallelism": f"dp{world} utterance/frame shards, no collective",
                   "cpu_binding": None if numa_cpus is None else f"{len(numa_cpus)} CPUs local to the GPU"},
        "clocks": clocks, "host": host_info(), "e2e": e2e, "gpu_launches": launches, "roofline": roof, "kernels": kern,
        "flop_per_frame": w["flop"], "model_tflops": value * w["flop"] / 1e12,
    }

    # ---- strong scaling (N > 1): ONE set (rank 0's) split by offset ranges, the product's sharded path
    if world > 1 and not args.no_strong:
        if rank != 0:  # every rank works on rank 0's set now: drop this rank's own (8.6 GB of pinned host memory)
            b = None
            import gc
            gc.collect()
            torch.cuda.empty_cache()
        line["strong"] = strong_leg(args, torch, dist_util, b, rank, local, world, steps, barrier, max_over_ranks)

    # ---- N = 1 extras: CPU baseline + parity, CLI wall clock, the other BASELINE configs as extra records
    if world == 1 and rank == 0:
        if not args.no_cpu_baseline:
            params = [m.params for m in b.members]
            rate, dt, sample, _, (rows, y_cpu) = cpu_reference_rate(args.workload, args.cpu_sample, params, b.x, b.offsets, b.iv)
            line["cpu_baseline"] = {"value": rate, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": sample, "seconds": dt}
            # the product's output = what the e2e leg left in the HOST array (after the compact transfer, if any)
            got = b.out_host[rows] if not args.no_e2e else b.out_dev[torch.from_numpy(rows).to(dev)].cpu().numpy()
            keep = np.abs(y_cpu).sum(axis=1) > 0  # quirk Q4 rows are 0 on both sides
            line["parity"] = {"vs": "cpu_baseline leg (fp32 NumPy forward, same weights and inputs)",
                              "of": "host output of the e2e leg" if not args.no_e2e else "device output",
                              "frames": int(keep.sum()), "max_abs": float(np.abs(got - y_cpu).max()),
                              "argmax_agreement_raw": float(np.mean(got[keep].argmax(axis=1) == y_cpu[keep].argmax(axis=1))),
                              "gate": "north_star: <= 5e-2 and >= 0.995 (16-bit modes), <= 1e-3 (fp32 mode)"}
            if args.cpu_python_prepare and not b.recurrent:
                r2, dt2, s2, _, _ = cpu_reference_rate(args.workload, min(args.cpu_sample, 32768), params, b.x, b.offsets,
                                                       b.iv, with_python_prepare=True)
                line["cpu_baseline"]["with_reference_python_splice"] = {"value": r2, "sample": s2, "seconds": dt2}
        if not args.no_cli:
            try:
                line["cli"] = cli_wall_clock(b, args.precision)
            except Exception as e:  # noqa: BLE001
                line["cli"] = {"error": repr(e)}
        extras = [e for e in args.extra.split(",") if e in WORKLOADS and e != args.workload]
        del b
        torch.cuda.empty_cache()
        line["extra"] = []
        for wname in extras:
            try:  # an extra record must never cost the headline line
                line["extra"].append(extra_record(args, torch, wname, local, steps, warmup, barrier, peaks))
            except Exception as e:  # noqa: BLE001
                line["extra"].append({"workload": wname, "error": repr(e)})
    elif rank == 0:
        line["cpu_baseline"] = None
    if rank == 0:
        if dumped is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "log_likelihoods.npy"), dumped)
        emit(line)
    dist_util.finalize()
    return 0


def extra_record(args, torch, wname, local, steps, warmup, barrier, peaks):
    """A shorter record of another BASELINE config (device-resident + e2e), so that the driver sees more than cfg2."""
    from nnacousticmodeling_b200 import ops
    e = Bench(wname, args.precision, local, data_rank=0)
    for _ in range(warmup):
        e.step_device()
    ops.PROFILE = []
    ms = timed_device(torch, e.step_device, steps, barrier)
    prof, ops.PROFILE = ops.PROFILE, None
    kern = kernel_table(prof, steps)
    e.step_e2e()
    s = timed_host(torch, e.step_e2e, steps, barrier)
    rec = {"workload": e.w["desc"], "precision": args.precision, "value": e.n / (ms * 1e-3), "ms_per_step": ms,
           "e2e": e.n / s, "frames": e.n, "kernels": kern, "roofline": roofline_block(kern, peaks, wname, steps),
           "model_tflops": e.n / (ms * 1e-3) * e.w["flop"] / 1e12}
    del e
    torch.cuda.empty_cache()
    return rec


def strong_leg(args, torch, dist_util, b_weak, rank, local, world, steps, barrier, max_over_ranks):
    """ONE data set for the whole job: rank r computes its dist_util.rank_shard (frames with a +-5 halo for the MLP,
    an utterance range for the recurrent nets) into its rows of a host array -- predict(gpu=[0..N-1]) with one process
    per GPU.  Afterwards rank 0 runs the whole set alone and every rank's sampled rows must equal it bit for bit."""
    import torch.distributed as dist
    dev = torch.device("cuda", local)
    # rank 0's weak-scaling set is seed 1234 + 17 * 0: it reuses it; the others build the same set
    b = b_weak if b_weak is not None else Bench(args.workload, args.precision, local, data_rank=0)
    barrier()
    n = b.n
    shard = dist_util.rank_shard(b.offsets, n, b.recurrent, world, rank)
    f0, f1 = shard[2], shard[3]
    for _ in range(2):
        b.step_device(shard)
    ms = max_over_ranks(timed_device(torch, lambda: b.step_device(shard), steps, barrier))
    b.step_e2e(shard)
    s = max_over_ranks(timed_host(torch, lambda: b.step_e2e(shard), steps, barrier))
    # bit identity: first / middle / last 512 rows of every shard against the single-GPU pass of rank 0
    b.step_device(shard)
    take = [r for a in (f0, (f0 + f1) // 2 - 256, f1 - 512) for r in range(max(a, f0), min(max(a, f0) + 512, f1))]
    idx = torch.tensor(sorted(set(take)), device=dev)
    mine = torch.zeros((1536, N_CLASSES), dtype=torch.float32, device=dev)
    mine[:len(idx)] = b.out_dev[idx]
    ids = torch.full((1536,), -1, dtype=torch.int64, device=dev)
    ids[:len(idx)] = idx
    all_rows = [torch.empty_like(mine) for _ in range(world)]
    all_ids = [torch.empty_like(ids) for _ in range(world)]
    dist.all_gather(all_rows, mine)  # verification only, outside every timed region
    dist.all_gather(all_ids, ids)
    identical = None
    if rank == 0:
        b.step_device(None)  # the whole set on one GPU
        torch.cuda.synchronize()
        identical = all(bool(torch.equal(b.out_dev[i[i >= 0]], r[:int((i >= 0).sum())])) for r, i in zip(all_rows, all_ids))
    barrier()
    return {"scaling": "strong", "frames_total": n, "value": n / (ms * 1e-3), "ms_per_step": ms,
            "e2e": n / s, "e2e_ms_per_step": s * 1e3, "shards": "dist_util.rank_shard: "
            + ("utterance ranges balanced on frames" if b.recurrent else "equal frame ranges + 5-frame halo"),
            "bit_identical_to_single_gpu": identical, "rows_checked_per_rank": int(len(idx))}


_RESULT_OUT = None


def _claim_stdout():
    """Rank 0 prints ONE JSON line on stdout.  Libraries also write there (NCCL prints its version banner from C code
    at communicator creation, whatever NCCL_DEBUG_FILE says), so the real stdout is kept aside for the result line and
    file descriptor 1 points at stderr for everything else."""
    global _RESULT_OUT
    if _RESULT_OUT is None:
        sys.stdout.flush()
        _RESULT_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _RESULT_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="fp16",
                    help="fp16 | bf16 | fp32 (bf16x3) | bf16+a[:layers][+w[:layers]] -- see engine.Precision")
    ap.add_argument("--cpu-sample", type=int, default=None,
                    help="frames of the workload timed on the CPU (default: ~10-30 s of host work)")
    ap.add_argument("--no-cpu-python-prepare", dest="cpu_python_prepare", action="store_false",
                    help="skip the second CPU figure: the baseline with the reference's per-frame Python splice loop "
                         "(kw_nn_utils.py:26-36; BASELINE.md section 3 asks for both)")
    ap.add_argument("--cpu-threads-all", action="store_true", help="force every host core for BLAS (reference arm default)")
    ap.add_argument("--extra", default="cfg3,cfg4", help="other workloads reported as short extra records at N = 1")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cli", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the end-to-end leg (profiling runs under ncu only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the device-resident leg's output of its last timed step to DIR/log_likelihoods.npy "
                         f"(float32; a fixed seeded sample of {DUMP_ROWS} rows when the set is larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the output of the device path: --impl ours only")
    if args.cpu_sample is None:
        # the cpu_baseline leg runs once (~10-30 s); the reference arm repeats its sample steps + warmup times
        args.cpu_sample = 65536 if args.impl == "reference" else 262144
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
