"""Build + load the C-ABI shared library (include/nnam_b200.h).

The library is built IN-TREE with nvcc for sm_100a and loaded with ctypes; there is no CPU
fallback -- if it is missing or fails to load, every op raises ``NnamError``.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import threading
from ctypes import c_char_p, c_float, c_int, c_longlong, c_void_p, POINTER

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libnnam_b200.so")
SOURCES = ["api.cu", "gemm.cu", "gemm_head.cu", "splice.cu", "head.cu", "recurrent.cu", "recurrent_mc.cu", "recurrent_wide.cu", "recurrent_wide_gru.cu", "peephole.cu",
           "host_widen.cpp"]  # .cpp = host-only code, compiled with the host C++ compiler
# measured dead end kept for reference (DSMEM all-gather recurrence); NNAM_WITH_CLUSTER_EXPERIMENT=1 builds it in
EXPERIMENTAL_SOURCES = ["experimental/recurrent_cluster.cu"]
ABI_VERSION = 4
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


class NnamError(RuntimeError):
    pass


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _with_experiments():
    return os.environ.get("NNAM_WITH_CLUSTER_EXPERIMENT", "0") == "1"


def _sources():
    names = SOURCES + (EXPERIMENTAL_SOURCES if _with_experiments() else [])
    return [os.path.join(CSRC, s) for s in names if os.path.exists(os.path.join(CSRC, s))]


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = _sources() + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    deps.append(os.path.join(PKG_DIR, "..", "include", "nnam_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    """Compile every CUDA translation unit for sm_100a into ``libnnam_b200.so`` (in-tree).
    Objects are compiled in parallel (one nvcc per .cu) and linked with ``nvcc -shared``."""
    if not force and not needs_build():
        return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor
    objdir = os.path.join(PKG_DIR, "build")
    os.makedirs(objdir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "-shared"] + (["-Xptxas", "-v"] if verbose else [])
    if _with_experiments():
        flags.append("-DNNAM_WITH_CLUSTER_EXPERIMENT")

    def compile_one(src):
        obj = os.path.join(objdir, os.path.splitext(os.path.basename(src))[0] + ".o")
        if src.endswith(".cpp"):
            cmd = [os.environ.get("CXX", "g++"), "-O3", "-std=c++17", "-fPIC", "-pthread", "-c", "-o", obj, src]
        else:
            cmd = [_nvcc()] + flags + ["-c", "-o", obj, src]
        res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
        if res.returncode != 0:
            raise NnamError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
        if verbose:
            print(res.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as pool:
        objs = list(pool.map(compile_one, _sources()))
    cmd = [_nvcc(), "-shared", "-o", LIB_PATH] + objs + ["-lpthread"]
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise NnamError("link failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    return LIB_PATH


_lib = None
_lock = threading.Lock()

_SIGNATURES = {
    "nnam_abi_version": (c_int, []),
    "nnam_last_error": (c_char_p, []),
    "nnam_sm_count": (c_int, []),
    "nnam_splice_transform": (c_int, [c_void_p, c_longlong, c_longlong, c_longlong, c_int, c_int, c_void_p, c_void_p,
                                      c_void_p, c_int, c_longlong, c_longlong, c_void_p, c_void_p, c_longlong, c_int,
                                      c_void_p]),
    "nnam_convert_f32": (c_int, [c_void_p, c_longlong, c_int, c_longlong, c_void_p, c_void_p, c_longlong, c_int,
                                 c_void_p]),
    "nnam_linear_bias_act": (c_int, [c_void_p, c_void_p, c_longlong, c_void_p, c_void_p, c_longlong, c_void_p,
                                     c_void_p, c_void_p, c_longlong, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                     c_void_p]),
    "nnam_head": (c_int, [POINTER(c_void_p), POINTER(c_float), c_int, c_longlong, c_int, c_void_p, c_void_p, c_void_p,
                          c_void_p, c_float, c_int, c_void_p, c_longlong, c_longlong, c_int, c_void_p]),
    "nnam_head_scatter": (c_int, [POINTER(c_void_p), POINTER(c_float), c_int, c_longlong, c_int, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_float, c_int, c_void_p, c_longlong, c_longlong, c_int, c_void_p,
                                  c_void_p]),
    "nnam_head_f16": (c_int, [POINTER(c_void_p), POINTER(c_float), c_int, c_longlong, c_int, c_void_p, c_void_p, c_void_p,
                              c_void_p, c_float, c_int, c_void_p, c_longlong, c_void_p, c_longlong, c_int, c_void_p,
                              c_void_p]),
    "nnam_linear_logsoftmax": (c_int, [c_void_p, c_void_p, c_longlong, c_void_p, c_void_p, c_longlong, c_void_p, c_void_p,
                                       c_float, c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_void_p, c_int,
                                       c_int, c_int, c_int, c_int, c_void_p]),
    # scoring forms of nnam_head_scatter / nnam_linear_logsoftmax (Chainer's softmax_cross_entropy + accuracy, †)
    "nnam_head_score": (c_int, [POINTER(c_void_p), POINTER(c_float), c_int, c_longlong, c_int, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_float, c_int, c_void_p, c_void_p, c_void_p, c_longlong, c_int,
                                c_void_p, c_void_p]),
    "nnam_linear_logsoftmax_score": (c_int, [c_void_p, c_void_p, c_longlong, c_void_p, c_void_p, c_longlong, c_void_p,
                                             c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                             c_int, c_int, c_int, c_void_p]),
    "nnam_widen_f16_host": (c_int, [c_void_p, c_longlong, c_void_p, c_void_p, c_longlong, c_void_p, c_longlong, c_int,
                                    c_int]),
    "nnam_gather_transform": (c_int, [c_void_p, c_longlong, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                      c_longlong, c_void_p, c_void_p, c_longlong, c_int, c_void_p]),
    "nnam_peephole_cell": (c_int, [c_int, c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_longlong, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_int, c_int, c_int, c_void_p]),
    "nnam_rnn_seq": (c_int, [c_void_p, c_void_p]),
    "nnam_rnn_desc_size": (c_int, []),
    "nnam_rnn_plan": (c_int, [c_int, c_int, c_int, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int),
                              POINTER(c_int)]),
    "nnam_rnn_solo_step_cycles": (c_int, [c_int, c_int, c_int, c_int, POINTER(c_int)]),
}


class RnnDesc(ctypes.Structure):
    """Mirror of ``NnamRnnDesc`` (include/nnam_b200.h)."""

    _fields_ = [
        ("cell", c_int), ("hidden", c_int), ("n_dirs", c_int), ("batch", c_int), ("streams", c_int), ("nsplit", c_int),
        ("flags", c_int), ("elem", c_int),
        ("gx", c_void_p * 2), ("gx_ld", c_longlong),
        ("w_hi", c_void_p * 2), ("w_lo", c_void_p * 2), ("w_ld", c_longlong),
        ("u_bias", c_void_p * 2),
        ("h_hi", c_void_p), ("h_lo", c_void_p), ("h_ld", c_longlong),
        ("xchg_hi", c_void_p), ("xchg_lo", c_void_p),
        ("n_items", c_int), ("item_batch", c_void_p), ("item_dir", c_void_p),
        ("n_groups", c_int), ("group_item_start", c_void_p),
        ("batch_row0", c_void_p), ("batch_steps", c_void_p), ("batch_nutt", c_void_p), ("batch_base_off", c_void_p),
        ("base", c_void_p), ("utt_len", c_void_p),
        ("h0_hi", c_void_p), ("h0_lo", c_void_p), ("c0", c_void_p), ("c_out", c_void_p),
        ("counters", c_void_p), ("started", c_void_p), ("started_tag", ctypes.c_uint), ("debug_cycles", c_void_p),
    ]


EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def lib():
    """Return the loaded ctypes library; fail loudly when it is absent (no CPU fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise NnamError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
                "nnacousticmodeling_b200 has no CPU or PyTorch fallback.")
        try:
            handle = ctypes.CDLL(LIB_PATH)
        except OSError as e:  # pragma: no cover
            raise NnamError(f"cannot load {LIB_PATH}: {e}") from e
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        if handle.nnam_abi_version() != ABI_VERSION:
            raise NnamError("libnnam_b200.so ABI version mismatch; rebuild")
        if handle.nnam_rnn_desc_size() != ctypes.sizeof(RnnDesc):
            raise NnamError("RnnDesc (ctypes) and NnamRnnDesc (include/nnam_b200.h) differ in size; rebuild")
        _lib = handle
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().nnam_last_error()
        raise NnamError(f"nnam_b200 error {rc}: {msg.decode() if msg else '?'}")
