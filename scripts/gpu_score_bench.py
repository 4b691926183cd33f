"""score() against predict() on the same host inputs: frames/s of each, alternated in one process.

    python scripts/gpu_score_bench.py --workload cfg2 [--runs 5] [--warmup 3] [--out profiles/r03_score_cfg2.json]

predict() writes the (N, 1909) float32 rows into a pinned host array (7,636 B per frame over PCIe, the end-to-end limit
of that path); score() returns 8 B per frame.  Both start from the same host features, targets are seeded random
labels.  The workloads and models are bench.py's (synth sets, Network.init_params), in fp16 mode.  Each run is timed
with a host clock around a call that ends in a device synchronise; the two calls alternate, so both see the same
machine state.  The GPU's name and power limit are read with nvidia-smi in the same process.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    res = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return res.stdout.strip().splitlines()[0] if res.returncode == 0 and res.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3"])
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--precision", default="fp16")
    ap.add_argument("--out", default=None, help="write the record as JSON here")
    args = ap.parse_args()

    import torch
    import bench
    import nnacousticmodeling_b200 as nn
    from nnacousticmodeling_b200 import engine

    if not torch.cuda.is_available():
        raise SystemExit("gpu_score_bench: needs a CUDA device")
    w, x, offsets, iv = bench.make_workload(args.workload)
    model = bench.make_models(w, args.precision, 0)[0]
    net = w["network"]
    winlen, td = (11, 0) if net == "ff" else (1, 5)
    off = offsets if nn.is_nn_recurrent(net) else None
    n = len(x)
    targets = np.random.default_rng(7).integers(0, bench.N_CLASSES, n).astype(np.int32)
    out = engine.empty_pinned((n, bench.N_CLASSES))

    def run_predict():
        nn.predict(model, x, off, bench.N_CLASSES, net, 0, winlen, td, None, progress=False, ivectors=iv, out=out)

    def run_score():
        return nn.score(model, x, off, targets, bench.N_CLASSES, net, 0, winlen, td, None, ivectors=iv)

    times = {"predict": [], "score": []}
    for i in range(args.warmup + args.runs):
        for name, fn in (("predict", run_predict), ("score", run_score)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                times[name].append(dt)
    s = run_score()
    rec = {
        "workload": args.workload, "desc": w["desc"], "precision": args.precision, "frames": n,
        "gpu": gpu_info(), "runs": args.runs, "warmup": args.warmup,
        "score_loss": s.loss, "score_accuracy": s.accuracy,
    }
    for name, ts in times.items():
        rec[name] = {"median_frames_per_s": n / statistics.median(ts), "best_frames_per_s": n / min(ts),
                     "seconds": ts}
    rec["median_speedup"] = rec["score"]["median_frames_per_s"] / rec["predict"]["median_frames_per_s"]
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
