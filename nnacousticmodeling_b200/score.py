"""Frame scoring against targets: the cross-entropy and frame accuracy of ``predict()``'s output, computed on the device.

In the reference, loss and accuracy exist only inside training (L.Classifier with F.softmax_cross_entropy and
F.accuracy, train.py); generate_folds.py writes the frame targets ``targets_{k}.npy`` next to ``data_{k}.npy``, so
fold model k scored on fold k's data is the cross-validated figure.  ``score()`` computes it without shipping the
(N, C) rows to the host: the output kernels reduce each row to its nll and argmax on the device, 8 B per frame.
"""
from __future__ import annotations

import json
import math
import sys
from pathlib import Path

import numpy as np

from . import engine
from ._native import NnamError
from .networks import is_nn_recurrent, load_npz
from .predict import _devices, fold_arg_parser, fold_setup


class FrameScore:
    """Per-frame scores and their sums.

    ``nll`` (N,) float32: -y_f[t_f] on scored frames, 0 elsewhere.  ``pred`` (N,) int32: argmax_c y_f[c] (lowest index on
    ties), -1 on rows that are no network output (the last ``timedelay`` frames of an utterance that ``predict()`` leaves
    zero, quirk Q4).  A frame is scored when its target is >= 0 and its row is a network output.  ``loss_sum`` is the
    float64 sum of nll over the scored frames; ``loss`` and ``accuracy`` are NaN when no frame is scored."""

    def __init__(self, targets, nll, pred):
        self.nll, self.pred = nll, pred
        scored = (np.asarray(targets) >= 0) & (pred >= 0)
        self.frames = int(len(nll))
        self.scored = int(scored.sum())
        self.correct = int((pred[scored] == np.asarray(targets)[scored]).sum())
        self.loss_sum = float(nll[scored].astype(np.float64).sum())

    @classmethod
    def pooled(cls, scores):
        """One FrameScore over the frames of several (the sums add up; nll / pred are concatenated)."""
        out = cls.__new__(cls)
        out.nll = np.concatenate([s.nll for s in scores]) if scores else np.zeros(0, np.float32)
        out.pred = np.concatenate([s.pred for s in scores]) if scores else np.zeros(0, np.int32)
        out.frames = sum(s.frames for s in scores)
        out.scored = sum(s.scored for s in scores)
        out.correct = sum(s.correct for s in scores)
        out.loss_sum = float(sum(s.loss_sum for s in scores))
        return out

    @property
    def loss(self):
        return self.loss_sum / self.scored if self.scored else math.nan

    @property
    def accuracy(self):
        return self.correct / self.scored if self.scored else math.nan

    def summary(self):
        """frames, scored, correct, loss_sum, loss, accuracy (NaN as None, so that the dict is valid JSON)."""
        def num(v):
            return None if isinstance(v, float) and math.isnan(v) else v
        return {"frames": self.frames, "scored": self.scored, "correct": self.correct, "loss_sum": self.loss_sum,
                "loss": num(self.loss), "accuracy": num(self.accuracy)}

    def __repr__(self):
        return (f"FrameScore(frames={self.frames}, scored={self.scored}, loss={self.loss:.6f}, "
                f"accuracy={self.accuracy:.6f})")


def check_targets(targets, n_frames, num_classes):
    """The targets as a contiguous int32 (N,) array; NnamError unless they are integers of shape (N,) in [-1, C)."""
    t = np.asarray(targets)
    if t.dtype == np.bool_ or not np.issubdtype(t.dtype, np.integer):
        raise NnamError(f"score: targets must be an integer array (got dtype {t.dtype})")
    if t.shape != (n_frames,):
        raise NnamError(f"score: targets must have shape ({n_frames},) (got {t.shape})")
    if n_frames and (int(t.min()) < -1 or int(t.max()) >= num_classes):
        raise NnamError(f"score: targets must lie in [0, {num_classes}) or be -1 (ignore), got values in "
                        f"[{int(t.min())}, {int(t.max())}]")
    return np.ascontiguousarray(t, dtype=np.int32)


def score(model, x, offsets, targets, num_classes, network, gpu, winlen, timedelay, ft, ivectors=None,
          fix_timedelay_tail=False, head=None, presliced=False):
    """Score ``predict()``'s output against frame targets without shipping it to the host.

    Arguments as :func:`predict.predict`, plus ``targets`` (N,) integers in [0, num_classes) or -1 (Chainer's
    ignore_label).  Returns a :class:`FrameScore`.  With the same model, precision and devices, nll[f] ==
    -predict(..., transfer="f32")[f, t_f] bit for bit and pred[f] == its argmax on every scored frame: the rows are
    computed by the same kernels with the same chunking, and reduced in the kernels' epilogues.  ``gpu`` may be a list:
    frame / utterance ranges are sharded across the devices as predict() shards them."""
    devs = _devices(gpu)
    x = np.ascontiguousarray(x, dtype=np.float32)
    n = x.shape[0]
    t = check_targets(targets, n, num_classes)
    recurrent = is_nn_recurrent(network)
    if recurrent and offsets is None:
        raise NnamError("score: recurrent networks need utterance offsets")
    nll = np.zeros(n, dtype=np.float32)
    pred = np.full(n, -1, dtype=np.int32)
    if n == 0:
        return FrameScore(t, nll, pred)
    dest = (t, nll, pred)
    if recurrent:
        from . import recurrent_engine
        offsets = np.asarray(offsets)
        shards = engine.partition_utterances(offsets, len(devs))
        engine.run_sharded(
            lambda sh, d: recurrent_engine.forward_utterances(model, x, offsets, None, sh[0], sh[1], ft=ft,
                                                              ivectors=ivectors, timedelay=timedelay, device=d,
                                                              fix_timedelay_tail=fix_timedelay_tail, head=head,
                                                              score=dest),
            shards, devs)
    else:
        splice = int(winlen) // 2
        shards = engine.partition_frames(n, len(devs))
        engine.run_sharded(
            lambda sh, d: engine.ff_forward_frames(model, x, ft, splice, None, sh[0], sh[1], ivectors=ivectors,
                                                   device=d, head=head, presliced=presliced, score=dest),
            shards, devs)
    return FrameScore(t, nll, pred)


def _line(name, s):
    return (f"{name}: frames {s.frames} scored {s.scored} loss {s.loss:.6f} accuracy {s.accuracy:.6f}")


def main(arg_list=None):
    """Score every fold model fold_{k}.npz on its held-out fold data_{k}.npy against targets_{k}.npy (the files
    generate_folds.py writes).  Same flags and defaults as the predict_folds CLI in fold mode, plus
    --fold-target-pattern and --json.  Prints one line per fold and a pooled line; writes no .npy output."""
    parser = fold_arg_parser("B200 frame scoring of fold models against their held-out frame targets")
    parser.add_argument("--fold-target-pattern", default="targets_{}.npy")
    parser.add_argument("--json", help="also write the figures to this JSON file")
    args = parser.parse_args(list(map(str, arg_list)) if arg_list is not None else None)

    model, model_cls, num_classes, recurrent, winlen, ft, gpu = fold_setup(args)
    results = []
    fold = 0
    while True:
        f = Path(args.fold_model_dir, args.fold_network_pattern.format(fold))
        if not f.is_file():
            break
        load_npz(str(f), model_cls)
        x = np.load(str(Path(args.fold_data_dir, args.fold_data_pattern.format(fold))))
        offsets = np.load(str(Path(args.fold_data_dir, args.fold_offset_pattern.format(fold)))) if recurrent else None
        iv = (np.load(str(Path(args.fold_data_dir, args.fold_ivector_pattern.format(fold))))
              if args.ivector_dir else None)
        targets = np.load(str(Path(args.fold_data_dir, args.fold_target_pattern.format(fold))))
        s = score(model, x, offsets, targets, num_classes, args.network, gpu, winlen, args.timedelay, ft, ivectors=iv)
        print(_line(f"fold {fold}", s))
        results.append(s)
        fold += 1
    if not results:
        print("Error: No fold networks found")
        sys.exit(2)
    pooled = FrameScore.pooled(results)
    print(_line("pooled", pooled))
    if args.json:
        doc = {"folds": [dict(fold=k, **s.summary()) for k, s in enumerate(results)], "pooled": pooled.summary()}
        Path(args.json).parent.mkdir(exist_ok=True, parents=True)
        with open(args.json, "w") as fh:
            json.dump(doc, fh, indent=1)


if __name__ == "__main__":
    main()
