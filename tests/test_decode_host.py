"""CPU checks of the decode entry points' argument checks: recnet_decoder_{greedy,beam,sample} and recnet_{greedy,beam,sample}_workspace_bytes
answer every input below before anything is launched (null buffers, no GPU needed).  Each input is tried with a valid, an unsupported
and a misaligned descriptor, so the table also pins which check comes first when an input is wrong in two ways."""
import ctypes as C

import pytest

from recnet_b200 import _lib as L

BAD, ALIGN, UNSUP = -1, -2, -4
OK = "bytes"                                # a workspace query that answers with a size
SHAPE = dict(B=12, T=5, E=16, H=8, A=8, EMB=8, V=5, L=1)
DESCS = ("valid", "unsupported", "misaligned")
FIX = {"valid": {}, "unsupported": dict(cell=L.CELL_GRU, n_layers=2), "misaligned": dict(E=10)}
PAIR = (C.c_uint64 * 2)(7, 0)               # a (seed, offset) pair in host memory: never read, every call below is refused
P = "pair"
NAN = float("nan")

# (entry point, arguments) -> (answer with a valid, an unsupported, a misaligned descriptor); None: that call would launch, not tried.
# greedy (max_steps,); beam (K, max_steps); sample (max_steps, temperature, noise, rng, train); queries without the run-time arguments.
CASES = [
    ("greedy", (0,), (BAD, BAD, BAD)),
    ("greedy", (65,), (BAD, BAD, BAD)),
    ("greedy", (31,), (None, UNSUP, ALIGN)),
    ("greedy_ws", (), (OK, OK, OK)),
    ("beam", (3, 0), (BAD, UNSUP, ALIGN)),
    ("beam", (3, 65), (BAD, UNSUP, ALIGN)),
    ("beam", (0, 31), (BAD, UNSUP, ALIGN)),
    ("beam", (9, 31), (BAD, UNSUP, ALIGN)),
    ("beam", (6, 31), (BAD, UNSUP, ALIGN)),              # K > V
    ("beam", (5, 31), (BAD, UNSUP, ALIGN)),              # B % K != 0
    ("beam", (0, 65), (BAD, UNSUP, ALIGN)),
    ("beam", (3, 31), (None, UNSUP, ALIGN)),
    ("beam_ws", (3, 0), (BAD, BAD, BAD)),
    ("beam_ws", (3, 65), (BAD, BAD, BAD)),
    ("beam_ws", (0, 31), (BAD, BAD, BAD)),
    ("beam_ws", (9, 31), (BAD, BAD, BAD)),
    ("beam_ws", (6, 31), (OK, OK, OK)),
    ("beam_ws", (5, 31), (OK, OK, OK)),
    ("beam_ws", (3, 31), (OK, OK, OK)),
    ("sample", (0, 1.0, P, None, 0), (BAD, UNSUP, ALIGN)),
    ("sample", (65, 1.0, P, None, 0), (BAD, UNSUP, ALIGN)),
    ("sample", (31, 0.0, P, None, 0), (BAD, UNSUP, ALIGN)),
    ("sample", (31, -1.0, P, None, 0), (BAD, UNSUP, ALIGN)),
    ("sample", (31, NAN, P, None, 0), (BAD, UNSUP, ALIGN)),
    ("sample", (31, 1.0, None, None, 0), (BAD, UNSUP, ALIGN)),
    ("sample", (31, 1.0, P, None, 1), (BAD, UNSUP, ALIGN)),     # train mode without a dropout pair
    ("sample", (65, NAN, None, None, 1), (BAD, UNSUP, ALIGN)),
    ("sample", (31, 1.0, P, P, 1), (None, UNSUP, ALIGN)),
    ("sample_ws", (0,), (BAD, UNSUP, ALIGN)),
    ("sample_ws", (65,), (BAD, UNSUP, ALIGN)),
    ("sample_ws", (31,), (OK, UNSUP, ALIGN)),
]


def _desc(kind, precision, train=0):
    f = dict(SHAPE, cell=L.CELL_LSTM, n_layers=1)
    f.update(FIX[kind])
    return L.decoder_desc(precision=precision, train=train, embedding_scale=1.0, p_emb_drop=0.5, p_out_drop=0.5, p_layer_drop=0.5, **f)


def _call(entry, args, kind, precision):
    lib, w = L.lib(), L.decoder_tensors()
    if entry == "greedy":
        return lib.recnet_decoder_greedy(C.byref(_desc(kind, precision)), C.byref(w), None, args[0], None, 0, None, None, None)
    if entry == "greedy_ws":
        return lib.recnet_greedy_workspace_bytes(C.byref(_desc(kind, precision)))
    if entry == "beam":
        return lib.recnet_decoder_beam(C.byref(_desc(kind, precision)), C.byref(w), None, *args, 2, None, 0, None, None, None)
    if entry == "beam_ws":
        return lib.recnet_beam_workspace_bytes(C.byref(_desc(kind, precision)), *args)
    if entry == "sample_ws":
        return lib.recnet_sample_workspace_bytes(C.byref(_desc(kind, precision, train=1)), *args)
    steps, tau, noise, rng, train = args
    noise, rng = (PAIR if x == P else None for x in (noise, rng))
    return lib.recnet_decoder_sample(C.byref(_desc(kind, precision, train)), C.byref(w), None, steps, tau, 2, rng, noise, None, 0, None,
                                     None, None, None, None)


@pytest.mark.parametrize("precision", [L.PREC_FP32, L.PREC_BF16])
def test_decode_entry_points_answer_bad_arguments_as_recorded(precision):
    got, want = {}, {}
    for entry, args, expected in CASES:
        for kind, code in zip(DESCS, expected):
            if code is None:
                continue
            r = _call(entry, args, kind, precision)
            got[entry, args, kind] = OK if code == OK and r > 0 else r
            want[entry, args, kind] = code
    assert {k: v for k, v in got.items() if v != want[k]} == {}
