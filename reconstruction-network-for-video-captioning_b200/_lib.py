"""ctypes binding of librecnet_b200.so (C ABI declared in include/recnet_b200.h).

The shared library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a only).  There is no
CPU or PyTorch fallback: if the library is missing, importing a symbol raises, and every compute call
raises RuntimeError on a non-zero status.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librecnet_b200.so")
CSRC = os.path.join(_HERE, "csrc")

PREC_FP32, PREC_BF16 = 0, 1
PRECISIONS = {"fp32": PREC_FP32, "bf16": PREC_BF16}

_STATUS = {
    -1: "RECNET_ERR_BAD_SHAPE", -2: "RECNET_ERR_ALIGNMENT", -3: "RECNET_ERR_UNSUPPORTED_ARCH",
    -4: "RECNET_ERR_UNSUPPORTED", -5: "RECNET_ERR_WORKSPACE", -6: "RECNET_ERR_DRIVER",
}

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/recnet_abi.cu -> librecnet_b200.so for sm_100a (cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [os.path.join(_HERE, "..", "include", "recnet_b200.h")]
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(s) for s in srcs):
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-o", LIB_PATH, os.path.join(CSRC, "recnet_abi.cu")]
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return LIB_PATH


class decoder_desc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("B", "T", "E", "H", "A", "EMB", "V", "L", "precision", "train")] + \
               [(n, C.c_float) for n in ("embedding_scale", "p_emb_drop", "p_out_drop")] + \
               [("cell", C.c_int32), ("n_layers", C.c_int32), ("p_layer_drop", C.c_float)]


CELL_LSTM, CELL_GRU = 0, 1
ATTN_SOFTMAX = 0x100           # OR'd into the descriptors' `cell`: the paper's softmax attention instead of the reference's mean


MAX_LAYERS = 4


class decoder_tensors(C.Structure):
    FIELDS = ("embedding", "attn_W", "attn_U", "attn_b", "attn_w", "w_ih", "w_hh", "b_ih", "b_hh", "out_w", "out_b")
    EXTRA = ("w_ih_x", "w_hh_x", "b_ih_x", "b_hh_x")          # per extra layer l = 1.., in this order in the flat parameter list
    _fields_ = [(n, C.c_void_p) for n in FIELDS] + [(n, C.c_void_p * (MAX_LAYERS - 1)) for n in EXTRA]


class local_desc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("B", "S", "R", "H", "A", "L", "precision", "train")] + [("p_drop", C.c_float), ("cell", C.c_int32), ("dec_layers", C.c_int32)]


class local_tensors(C.Structure):
    FIELDS = ("attn_W", "attn_U", "attn_b", "attn_w", "w_ih", "w_hh", "b_ih", "b_hh", "out_w", "out_b")
    _fields_ = [(n, C.c_void_p) for n in FIELDS]


class global_desc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("B", "L", "R", "H", "T", "precision", "train")] + \
               [("p_drop", C.c_float), ("caption_max_len", C.c_float), ("cell", C.c_int32), ("dec_layers", C.c_int32)]


class global_tensors(C.Structure):
    FIELDS = ("w_ih", "w_hh", "b_ih", "b_hh", "out_w", "out_b")
    _fields_ = [(n, C.c_void_p) for n in FIELDS]


class cider_corpus(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_videos", "n_df", "vocab")] + [("ref_len", C.c_float)] + \
               [(n, C.c_void_p) for n in ("df_keys", "df_log", "video_refs", "ref_entries", "entry_keys", "entry_w", "ref_norm",
                                          "ref_length")]


_p, _i, _l, _f, _u, _d = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint32, C.c_double

# name -> (restype, argtypes); mirrors include/recnet_b200.h one to one
SIGNATURES = {
    "recnet_abi_version": (_i, []),
    "recnet_query_device": (_i, [_i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "recnet_launch_count": (C.c_longlong, []),
    "recnet_profile_enable": (_i, [_i, _i]),
    "recnet_profile_collect": (_i, [_p, _i]),
    "recnet_gemm": (_i, [_i, _p, _l, _i, _p, _l, _i, _p, _l, _p, _l, _p, _i, _i, _i, _i, _l, _i, _i, _p]),
    "recnet_plan_persistent_loops": (_i, [C.POINTER(local_desc), _p]),
    "recnet_plan_batched_gemm": (_i, [_i, _i, _i, _i, _p, _p]),
    "recnet_splitk_reduce": (_i, [_p, _i, _l, _l, _p, _l, _i, _i, _i, _p]),
    "recnet_attn_fwd": (_i, [_i, _p, _i, _l, _p, _l, _l, _p, _p, _p, _l, _l, _i, _i, _i, _i, _i, _p, _p, _p, _l, _f, _p, _u, _l, _p]),
    "recnet_attn_bwd": (_i, [_i, _p, _i, _l, _l, _p, _l, _l, _p, _p, _l, _l, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p, _i, _p, _f, _p, _u, _l, _p]),
    "recnet_attn_bwd_softmax": (_i, [_i, _p, _i, _l, _l, _p, _l, _l, _p, _p, _p, _l, _l, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p, _i, _p, _f, _p,
                                     _u, _l, _p]),
    "recnet_lstm_cell_fwd": (_i, [_i, _p, _i, _l, _l, _p, _l, _p, _p, _p, _i, _i, _p, _p, _p, _l, _p, _l, _p, _l, _p]),
    "recnet_lstm_cell_bwd": (_i, [_i, _p, _l, _p, _p, _l, _p, _i, _l, _l, _i, _p, _i, _l, _l, _p, _i, _p, _p, _p, _i, _i, _p, _l, _p]),
    "recnet_gru_cell_fwd": (_i, [_i, _p, _i, _l, _l, _p, _i, _l, _l, _p, _l, _p, _p, _p, _l, _i, _i, _p, _p, _l, _p, _l, _p]),
    "recnet_gru_cell_bwd": (_i, [_i, _p, _l, _p, _l, _p, _i, _l, _l, _p, _i, _l, _l, _p, _i, _p, _p, _l, _i, _i, _p, _p, _l, _p]),
    "recnet_decoder_workspace_bytes": (_l, [C.POINTER(decoder_desc)]),
    "recnet_decoder_fwd": (_i, [C.POINTER(decoder_desc), C.POINTER(decoder_tensors), _p, _p, _p, _p, _p, _p, _l, _p, _p, _p]),
    "recnet_decoder_fwd_phase": (_i, [C.POINTER(decoder_desc), C.POINTER(decoder_tensors), _p, _p, _p, _p, _p, _p, _l, _p, _p, _i, _p]),
    "recnet_decoder_bwd": (_i, [C.POINTER(decoder_desc), C.POINTER(decoder_tensors), _p, _p, _p, _p, _p, _p, _l, _p, _p, _p,
                                C.POINTER(decoder_tensors), _p]),
    "recnet_decoder_bwd_phase": (_i, [C.POINTER(decoder_desc), C.POINTER(decoder_tensors), _p, _p, _p, _p, _p, _p, _l, _p, _p, _p,
                                      C.POINTER(decoder_tensors), _i, _p]),
    "recnet_decoder_bwd_is_split": (_i, [C.POINTER(decoder_desc)]),
    "recnet_decoder_logits": (_p, [C.POINTER(decoder_desc), _p, C.POINTER(_l)]),
    "recnet_greedy_workspace_bytes": (_l, [C.POINTER(decoder_desc)]),
    "recnet_decoder_greedy": (_i, [C.POINTER(decoder_desc), C.POINTER(decoder_tensors), _p, _i, _p, _l, _p, _p, _p]),
    "recnet_beam_workspace_bytes": (_l, [C.POINTER(decoder_desc), _i, _i]),
    "recnet_decoder_beam": (_i, [C.POINTER(decoder_desc), C.POINTER(decoder_tensors), _p, _i, _i, _l, _p, _l, _p, _p, _p]),
    "recnet_sample_workspace_bytes": (_l, [C.POINTER(decoder_desc), _i]),
    "recnet_decoder_sample": (_i, [C.POINTER(decoder_desc), C.POINTER(decoder_tensors), _p, _i, _f, _l, _p, _p, _p, _l, _p, _p, _p, _p,
                                   _p]),
    "recnet_local_workspace_bytes": (_l, [C.POINTER(local_desc)]),
    "recnet_local_fwd": (_i, [C.POINTER(local_desc), C.POINTER(local_tensors), _p, _p, _p, _p, _l, _p, _p]),
    "recnet_local_bwd": (_i, [C.POINTER(local_desc), C.POINTER(local_tensors), _p, _p, _p, _p, _l, _p,
                              C.POINTER(local_tensors), _p, _p]),
    "recnet_local_bwd_phase": (_i, [C.POINTER(local_desc), C.POINTER(local_tensors), _p, _p, _p, _p, _l, _p,
                                    C.POINTER(local_tensors), _p, _i, _p]),
    "recnet_set_background_ctas": (_i, [_i]),
    "recnet_local_outputs": (_p, [C.POINTER(local_desc), _p]),
    "recnet_global_workspace_bytes": (_l, [C.POINTER(global_desc)]),
    "recnet_global_fwd": (_i, [C.POINTER(global_desc), C.POINTER(global_tensors), _p, _p, _p, _p, _l, _p, _p]),
    "recnet_global_bwd": (_i, [C.POINTER(global_desc), C.POINTER(global_tensors), _p, _p, _p, _p, _l, _p,
                               C.POINTER(global_tensors), _p, _p]),
    "recnet_global_outputs": (_p, [C.POINTER(global_desc), _p]),
    "recnet_decoder_error_offset": (_l, [C.POINTER(decoder_desc)]),
    "recnet_local_error_offset": (_l, [C.POINTER(local_desc)]),
    "recnet_global_error_offset": (_l, [C.POINTER(global_desc)]),
    "recnet_debug_set_timeline": (_i, [_p]),
    "recnet_debug_dropout_mask": (_i, [_p, C.c_uint32, _l, C.c_float, _p, _p]),
    "recnet_param_norms_fwd": (_i, [_p, _p, _i, _p, _p, _i, _p, _p, _p, _p, _p, _p, _p]),
    "recnet_param_norms_partial": (_i, [_p, _p, _p, _p, _i, _p, _p]),
    "recnet_param_norms_finalize": (_i, [_p, _p, _i, _i, _p, _p, _p, _p, _p, _p]),
    "recnet_param_norms_bwd": (_i, [_p, _p, _p, _i, _p, _p, _i, _p, _p, _f, _p, _i, _p]),
    "recnet_cider_d": (_i, [C.POINTER(cider_corpus), _p, _l, _l, _i, _i, _p, _l, _p, _p]),
    "recnet_teacher_forcing_prep": (_i, [_p, _i, _i, _l, _l, _p, _p, _p]),
    "recnet_allreduce_avg": (_i, [_p, _p, _p, _p, _p, _p, _p, _l, _l, _i, _i, _i, _p]),
    "recnet_adam_step": (_i, [_p, _p, _p, _p, _p, _p, _i, _p, _p, _i, _d, _d, _d, _d, _d, _d, _p, _p, _i, _p]),
}

_lib = None


def lib() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built -- there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). recnet_b200 has no CPU/PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)       # AttributeError if the header and the library disagree
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(status: int, what: str = "recnet call") -> None:
    if status == 0:
        return
    if status < 0:
        raise RuntimeError(f"{what} failed: {_STATUS.get(status, status)}")
    raise RuntimeError(f"{what} failed: cudaError_t {status}")


_device_ok = {}


def require_device(index: int) -> None:
    """Refuse to run on anything but an sm_100 device (no other cubin is shipped)."""
    if index in _device_ok:
        return
    sm, ma, mi = C.c_int(), C.c_int(), C.c_int()
    st = lib().recnet_query_device(index, C.byref(sm), C.byref(ma), C.byref(mi))
    if st != 0:
        check(st, f"recnet_query_device (cc {ma.value}.{mi.value})")
    _device_ok[index] = sm.value
