"""``predict()`` and the ``predict_folds`` CLI of the reference (scripts/common/predict_folds.py),
re-hosted on the B200 kernels.  Same signature and file conventions; ``gpu`` may also be a list of
device indices (utterance/frame ranges are sharded across them with no collective)."""
from __future__ import annotations

import argparse
import sys
from pathlib import Path

import numpy as np

from . import engine, functions as F
from ._native import NnamError
from .features import adapt_transform, loadKaldiFeatureTransform
from .networks import Classifier, get_nn, is_nn_recurrent, load_npz


def _devices(gpu):
    devs = list(gpu) if isinstance(gpu, (list, tuple)) else [gpu]
    if any(int(d) < 0 for d in devs):
        raise NnamError("gpu < 0 (CPU) is not supported by nnacousticmodeling_b200")
    return [int(d) for d in devs]


def predict(model, x, offsets, num_classes, network, gpu, winlen, timedelay, ft, progress=True, ivectors=None,
            out=None, fix_timedelay_tail=False, head=None, presliced=False, sink=None, transfer=None):
    """predict_folds.py:27-95.  Returns (N, num_classes) float32 log-softmax outputs.

    Extensions: ``ivectors`` (N, I) are appended AFTER splice + transform (train.py:255-258 /
    evaluate.py:169-171 order; see SURVEY quirk Q2); ``out`` may be a caller-owned (pinned) array;
    ``fix_timedelay_tail`` fills the last ``timedelay`` frames that the reference leaves 0 (quirk Q4);
    ``model`` may be a list of same-shaped nets whose outputs are combined on the device by ``head``
    (an ``engine.HeadSpec``: logit mean of evaluate.py:35-51, log-prob mean of predict_folds.py:199-219, RPL4,
    prior); ``presliced`` says ``x`` is already spliced/transformed (the evaluate.py data flow); ``sink`` (an
    ``engine.RowSink``) receives the output rows chunk by chunk instead of an array being returned (the CLI streams
    them into the .npy file while the next chunk is computed); ``transfer`` = "f32" | "f16" | None picks how rows cross
    PCIe (engine.use_compact_transfer: the 16-bit precision modes send fp16 offsets from each row's maximum -- half
    the bytes, <= 2^-12 relative to an entry's distance from the maximum -- and host threads widen them back to the
    float32 layout; the fp32-accurate mode sends float32).

    The returned array is page-locked when the function allocates it: the device->host copies of the (N, C) matrix
    -- 7.6 KB per frame, the end-to-end bottleneck -- then run asynchronously at PCIe speed under the computation.
    """
    devs = _devices(gpu)
    x = np.ascontiguousarray(x, dtype=np.float32)
    n = x.shape[0]
    if sink is not None and len(devs) == 1 and not is_nn_recurrent(network) and n > 0:
        engine.ff_forward_frames(model, x, ft, int(winlen) // 2, None, 0, n, ivectors=ivectors, device=devs[0],
                                 head=head, presliced=presliced, sink=sink, transfer=transfer)
        return None
    if out is None:
        out = engine.empty_pinned((n, num_classes)) if n > 0 else np.zeros((0, num_classes), dtype=np.float32)
    elif out.shape != (n, num_classes) or out.dtype != np.float32:
        raise NnamError("predict: out must be float32 of shape (N, num_classes)")
    if n == 0:
        if sink is not None:
            return None
        return out
    threads = max(1, engine.default_host_threads() // len(devs))  # per device: host threads widening compact rows
    if is_nn_recurrent(network):
        from . import recurrent_engine
        if offsets is None:
            raise NnamError("predict: recurrent networks need utterance offsets")
        offsets = np.asarray(offsets)
        shards = engine.partition_utterances(offsets, len(devs))
        engine.run_sharded(
            lambda sh, d: recurrent_engine.forward_utterances(model, x, offsets, out, sh[0], sh[1], ft=ft,
                                                              ivectors=ivectors, timedelay=timedelay, device=d,
                                                              fix_timedelay_tail=fix_timedelay_tail, head=head,
                                                              transfer=transfer, host_threads=threads),
            shards, devs)
    else:
        splice = int(winlen) // 2
        shards = engine.partition_frames(n, len(devs))
        engine.run_sharded(
            lambda sh, d: engine.ff_forward_frames(model, x, ft, splice, out, sh[0], sh[1], ivectors=ivectors,
                                                   device=d, head=head, presliced=presliced, transfer=transfer,
                                                   host_threads=threads),
            shards, devs)
    if sink is not None:  # recurrent nets finish utterance subsets out of row order, several devices interleave:
        sink.write(0, n, out)  # the rows go to the sink in one piece at the end
        return None
    return out


class NpyFileSink(engine.RowSink):
    """Streams rows, in order, into a ``.npy`` file that ``np.load`` reads back as the (N, C) float32 C-contiguous
    array ``np.save`` would have written (predict_folds.py:240)."""

    def __init__(self, path, n_rows, n_cols):
        self.f = open(path, "wb")
        np.lib.format.write_array_header_1_0(
            self.f, {"descr": np.lib.format.dtype_to_descr(np.dtype(np.float32)), "fortran_order": False,
                     "shape": (int(n_rows), int(n_cols))})
        self.next_row, self.n_rows = 0, int(n_rows)

    def write(self, r0, r1, rows):
        if r0 != self.next_row:
            raise NnamError(f"NpyFileSink: rows [{r0}, {r1}) arrived out of order (expected row {self.next_row})")
        self.f.write(memoryview(np.ascontiguousarray(rows, dtype=np.float32)).cast("B"))
        self.next_row = r1

    def close(self):
        self.f.close()
        if self.next_row != self.n_rows:
            raise NnamError(f"NpyFileSink: {self.next_row} of {self.n_rows} rows were written")


def _activation(name):
    if name not in ("sigmoid", "tanh", "relu"):
        print("Wrong activation function specified")
        sys.exit(1)
    return F.resolve(name)


def fold_arg_parser(description):
    """The predict_folds flags (predict_folds.py:97-130) with their names and defaults, shared by this module's CLI and
    the scoring CLI (score.main)."""
    parser = argparse.ArgumentParser(description=description)
    parser.add_argument("--network", "-n", default="ff")
    parser.add_argument("--gpu", "-g", type=int, nargs="+", default=[0], help="GPU id(s); CPU (<0) is not supported")
    parser.add_argument("--units", "-u", type=int, nargs="+", default=[1024])
    parser.add_argument("--layers", "-l", type=int, default=2)
    parser.add_argument("--activation", "-a", default="relu")
    parser.add_argument("--tdnn-ksize", type=int, nargs="+", default=[5])
    parser.add_argument("--timedelay", type=int, default=0)
    parser.add_argument("--splice", type=int, default=0)
    parser.add_argument("--dropout", "-d", type=float, nargs="+", default=[0])
    parser.add_argument("--ft")
    parser.add_argument("--tri", action="store_true")
    parser.add_argument("--data-dir", default="data/fmllr")
    parser.add_argument("--offset-dir", default="data")
    parser.add_argument("--ivector-dir")
    parser.add_argument("--data", default="data_{}.npy")
    parser.add_argument("--offsets", default="offsets_{}.npy")
    parser.add_argument("--ivectors", default="ivectors_{}.npy")
    parser.add_argument("--fold-data-dir")
    parser.add_argument("--fold-output-dir")
    parser.add_argument("--fold-model-dir")
    parser.add_argument("--fold-output-dev")
    parser.add_argument("--fold-data-pattern", default="data_{}.npy")
    parser.add_argument("--fold-offset-pattern", default="offsets_{}.npy")
    parser.add_argument("--fold-ivector-pattern", default="ivectors_{}.npy")
    parser.add_argument("--fold-output-pattern", default="data_{}.npy")
    parser.add_argument("--fold-network-pattern", default="fold_{}.npz")
    parser.add_argument("--no-progress", action="store_true")
    parser.add_argument("--precision", default=None, help="extension: GEMM precision mode (fp32 | fp16 | bf16, see engine.Precision)")
    return parser


def fold_setup(args):
    """What both fold CLIs derive from the flags: (model, its Classifier, num_classes, recurrent, winlen, ft, gpu)."""
    num_classes = 1909 if args.tri else 39
    model = get_nn(args.network, args.layers, args.units, num_classes, _activation(args.activation),
                   args.tdnn_ksize, args.dropout)
    if args.precision:
        model.precision = args.precision
    model_cls = Classifier(model)
    recurrent = is_nn_recurrent(args.network)
    splice = (sum(args.tdnn_ksize) - len(args.tdnn_ksize)) // 2 if args.network == "tdnn" else args.splice
    winlen = 2 * splice + 1
    ft = None
    if args.ft is not None and args.ft != "-":
        ft = adapt_transform(loadKaldiFeatureTransform(str(Path(args.data_dir, args.ft))), args.network, splice,
                             recurrent)
    gpu = args.gpu if len(args.gpu) > 1 else args.gpu[0]
    return model, model_cls, num_classes, recurrent, winlen, ft, gpu


def main(arg_list=None):
    """predict_folds.py:97-246 -- same flags, same directory conventions, same outputs."""
    parser = fold_arg_parser("B200 network-output step (predict_folds drop-in)")
    args = parser.parse_args(list(map(str, arg_list)) if arg_list is not None else None)

    out_file = Path(args.fold_output_dir, args.fold_output_dev or args.fold_output_pattern)
    out_file.parent.mkdir(exist_ok=True, parents=True)
    model, model_cls, num_classes, recurrent, winlen, ft, gpu = fold_setup(args)

    def fold_models():
        fold = 0
        while True:
            f = Path(args.fold_model_dir, args.fold_network_pattern.format(fold))
            if not f.is_file():
                return
            load_npz(str(f), model_cls)
            print("Predicting fold {} data".format(fold))
            yield fold
            fold += 1

    n_folds = 0
    if args.fold_output_dev is not None:
        x = np.load(str(Path(args.data_dir, args.data.format("dev"))))
        offsets = np.load(str(Path(args.offset_dir, args.offsets.format("dev")))) if recurrent else None
        iv = np.load(str(Path(args.ivector_dir, args.ivectors.format("dev")))) if args.ivector_dir else None
        folds = []
        while True:
            f = Path(args.fold_model_dir, args.fold_network_pattern.format(len(folds)))
            if not f.is_file():
                break
            m = get_nn(args.network, args.layers, args.units, num_classes, _activation(args.activation),
                       args.tdnn_ksize, args.dropout)
            if args.precision:
                m.precision = args.precision
            load_npz(str(f), Classifier(m))
            print("Predicting fold {} data".format(len(folds)))
            folds.append(m)
        n_folds = len(folds)
        if n_folds == 0:
            print("Error: No fold networks found")
            sys.exit(2)
        # predict_folds.py:199-219: mean of the fold LOG-SOFTMAX outputs, renormalised (quirk Q5) -- one pass on the
        # device: K4 normalises every member, averages, and normalises again
        y_out = predict(folds, x, offsets, num_classes, args.network, gpu, winlen, args.timedelay, ft,
                        not args.no_progress, ivectors=iv, head=engine.HeadSpec(pre_normalize=True))
        if recurrent and args.timedelay > 0:
            # quirk Q4 through the reference's averaging: the unwritten (all-zero) tail rows of every fold average to
            # zero and are then renormalised to -log(C) (predict_folds.py:217-219)
            for u in range(len(offsets) - 1):
                y_out[max(int(offsets[u + 1]) - args.timedelay, int(offsets[u])):int(offsets[u + 1])] = -np.log(
                    np.float32(num_classes))
        np.save(str(Path(args.fold_output_dir, args.fold_output_dev)), y_out)
    else:
        for fold in fold_models():
            x = np.load(str(Path(args.fold_data_dir, args.fold_data_pattern.format(fold))))
            offsets = np.load(str(Path(args.fold_data_dir, args.fold_offset_pattern.format(fold)))) if recurrent else None
            iv = (np.load(str(Path(args.fold_data_dir, args.fold_ivector_pattern.format(fold))))
                  if args.ivector_dir else None)
            # np.save(path, y) of predict_folds.py:240, streamed: chunk i goes to the file while chunk i+1 is computed
            sink = NpyFileSink(str(Path(args.fold_output_dir, args.fold_output_pattern.format(fold))), len(x), num_classes)
            try:
                predict(model, x, offsets, num_classes, args.network, gpu, winlen, args.timedelay, ft,
                        not args.no_progress, ivectors=iv, sink=sink)
            except BaseException:
                sink.f.close()
                raise
            sink.close()
            n_folds += 1
        if n_folds == 0:
            print("Error: No fold networks found")
            sys.exit(2)


if __name__ == "__main__":
    main()
