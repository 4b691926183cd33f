"""nnacousticmodeling_b200 -- B200-native network-output hot path of OrcusCZ/NNAcousticModeling.

Feature matrix (+ offsets, i-vectors, Kaldi feature transform) -> per-frame pdf log-likelihoods,
behind the reference's Python surface (get_nn / model specs / predict / evaluateModelTestTri),
and their scores against frame targets (``score``: cross-entropy and frame accuracy, reduced on the device),
computed by hand-written sm_100a CUDA kernels in ``libnnam_b200.so`` (C ABI: include/nnam_b200.h).
There is no CPU fallback.
"""
from ._native import NnamError, build  # noqa: F401
from . import functions as F  # noqa: F401
from .networks import (  # noqa: F401
    GRU, LSTM, MLP, TDNN, Classifier, NetMGRU, PeepholeLSTM, RPL4, ZoneoutDropoutLSTM, ZoneoutLSTM,
    get_nn, is_nn_recurrent, load_npz, save_npz, set_default_precision,
)
from .features import (  # noqa: F401
    adapt_transform, loadBin, loadKaldiFeatureTransform, saveBin, splice_and_transform, splicing,
)
from .engine import empty_pinned, partition_frames, partition_utterances  # noqa: F401
from .engine import HeadSpec  # noqa: F401
from .predict import predict  # noqa: F401
from .score import FrameScore, score  # noqa: F401
from . import evaluate  # noqa: F401
from .evaluate import NNWithRPL, evaluateModelTestTri  # noqa: F401

__version__ = "0.1.0"
