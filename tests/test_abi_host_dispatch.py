"""Host-side dispatch of the C ABI, checked on the CPU through ctypes: which plan each descriptor gets (workspace sizes, buffer
offsets, the decoder's split and the persistent-loop layout), how invalid descriptors are rejected, and that the RECNET_* switches
are still read.

GOLDEN was recorded from the library built at commit e069efa, which had the same plans; every query below must keep answering
exactly that.  The queries run in a child process whose environment has no RECNET_* variable, so that a developer's shell cannot
change the answer (the switches are read once per process)."""
import json
import os
import subprocess
import sys

from recnet_b200 import _lib as L

# Runs in a child: loads _lib.py (path in argv[1]) without importing the package, answers argv[2] as JSON on stdout.
_CHILD = r'''
import ctypes as C, importlib.util, json, sys
spec = importlib.util.spec_from_file_location("_recnet_lib", sys.argv[1])
L = importlib.util.module_from_spec(spec)
spec.loader.exec_module(L)
lib = L.lib()
BASE = 4096
PREC = {"fp32": L.PREC_FP32, "bf16": L.PREC_BF16}
CELL = {"LSTM": L.CELL_LSTM, "GRU": L.CELL_GRU}
DEC_SHAPES = {"bench": dict(B=100, T=28, E=1536, H=512, A=128, EMB=468, V=4188, L=31),
              "small": dict(B=4, T=5, E=16, H=8, A=6, EMB=8, V=11, L=3)}          # A = 6: not on the projected-feature path
LOC_SHAPES = {"bench": dict(B=100, S=28, R=1536, H=512, A=128, L=31), "small": dict(B=4, S=5, R=16, H=8, A=6, L=3)}


def dec_desc(shape, prec, cell, layers):
    return L.decoder_desc(precision=prec, train=1, embedding_scale=1.0, p_emb_drop=0.5, p_out_drop=0.5, cell=cell, n_layers=layers,
                          **DEC_SHAPES[shape])


def loc_desc(shape, prec, cell, layers):
    return L.local_desc(precision=prec, train=1, p_drop=0.5, cell=cell, dec_layers=layers, **LOC_SHAPES[shape])


def glob_desc(prec):
    return L.global_desc(B=100, L=31, R=1536, H=512, T=28, precision=prec, train=1, p_drop=0.5, caption_max_len=30.0,
                         cell=L.CELL_LSTM, dec_layers=1)


def off(p):
    return None if p is None else p - BASE


def dec_row(d):
    r = C.byref(d)
    ld = C.c_int64(-1)
    p = lib.recnet_decoder_logits(r, C.c_void_p(BASE), C.byref(ld))
    return [lib.recnet_decoder_workspace_bytes(r), lib.recnet_greedy_workspace_bytes(r), lib.recnet_beam_workspace_bytes(r, 3, 31),
            lib.recnet_decoder_bwd_is_split(r), lib.recnet_decoder_error_offset(r), ld.value, off(p)]


def loc_row(d):
    r = C.byref(d)
    out = (C.c_int32 * 12)()
    st = lib.recnet_plan_persistent_loops(r, out)
    return [lib.recnet_local_workspace_bytes(r), lib.recnet_local_error_offset(r), off(lib.recnet_local_outputs(r, C.c_void_p(BASE))),
            st] + list(out)


def golden():
    t = {}
    for shape in DEC_SHAPES:
        for pn, prec in PREC.items():
            for cn, cell in CELL.items():
                for sm in (0, L.ATTN_SOFTMAX):
                    for layers in (1, 2):
                        k = "%s/%s/%s%s/n%d" % (shape, pn, cn, "+softmax" if sm else "", layers)
                        t["dec/" + k] = dec_row(dec_desc(shape, prec, cell | sm, layers))
                        t["loc/" + k] = loc_row(loc_desc(shape, prec, cell | sm, layers))
    for pn, prec in PREC.items():
        r = C.byref(glob_desc(prec))
        t["glob/" + pn] = [lib.recnet_global_workspace_bytes(r), lib.recnet_global_error_offset(r),
                           off(lib.recnet_global_outputs(r, C.c_void_p(BASE)))]
    return t


def invalid():
    """Every descriptor entry point, once with a null descriptor and once with precision 7."""
    dw, lw, gw = L.decoder_tensors(), L.local_tensors(), L.global_tensors()
    dec = {
        "recnet_decoder_workspace_bytes": lambda d: lib.recnet_decoder_workspace_bytes(d),
        "recnet_greedy_workspace_bytes": lambda d: lib.recnet_greedy_workspace_bytes(d),
        "recnet_beam_workspace_bytes": lambda d: lib.recnet_beam_workspace_bytes(d, 3, 31),
        "recnet_decoder_error_offset": lambda d: lib.recnet_decoder_error_offset(d),
        "recnet_decoder_bwd_is_split": lambda d: lib.recnet_decoder_bwd_is_split(d),
        "recnet_decoder_logits": lambda d: lib.recnet_decoder_logits(d, C.c_void_p(BASE), None),
        "recnet_decoder_fwd": lambda d: lib.recnet_decoder_fwd(d, C.byref(dw), *[None] * 6, 0, None, None, None),
        "recnet_decoder_fwd_phase": lambda d: lib.recnet_decoder_fwd_phase(d, C.byref(dw), *[None] * 6, 0, None, None, 1, None),
        "recnet_decoder_bwd": lambda d: lib.recnet_decoder_bwd(d, C.byref(dw), *[None] * 6, 0, None, None, None, C.byref(dw), None),
        "recnet_decoder_bwd_phase": lambda d: lib.recnet_decoder_bwd_phase(d, C.byref(dw), *[None] * 6, 0, None, None, None, C.byref(dw),
                                                                           1, None),
        "recnet_decoder_greedy": lambda d: lib.recnet_decoder_greedy(d, C.byref(dw), None, 31, None, 0, None, None, None),
        "recnet_decoder_beam": lambda d: lib.recnet_decoder_beam(d, C.byref(dw), None, 3, 31, 2, None, 0, None, None, None),
    }
    loc = {
        "recnet_local_workspace_bytes": lambda d: lib.recnet_local_workspace_bytes(d),
        "recnet_local_error_offset": lambda d: lib.recnet_local_error_offset(d),
        "recnet_local_outputs": lambda d: lib.recnet_local_outputs(d, C.c_void_p(BASE)),
        "recnet_plan_persistent_loops": lambda d: lib.recnet_plan_persistent_loops(d, (C.c_int32 * 12)()),
        "recnet_local_fwd": lambda d: lib.recnet_local_fwd(d, C.byref(lw), None, None, None, None, 0, None, None),
        "recnet_local_bwd": lambda d: lib.recnet_local_bwd(d, C.byref(lw), None, None, None, None, 0, None, C.byref(lw), None, None),
        "recnet_local_bwd_phase": lambda d: lib.recnet_local_bwd_phase(d, C.byref(lw), None, None, None, None, 0, None, C.byref(lw), None,
                                                                       1, None),
    }
    glob = {
        "recnet_global_workspace_bytes": lambda d: lib.recnet_global_workspace_bytes(d),
        "recnet_global_error_offset": lambda d: lib.recnet_global_error_offset(d),
        "recnet_global_outputs": lambda d: lib.recnet_global_outputs(d, C.c_void_p(BASE)),
        "recnet_global_fwd": lambda d: lib.recnet_global_fwd(d, C.byref(gw), None, None, None, None, 0, None, None),
        "recnet_global_bwd": lambda d: lib.recnet_global_bwd(d, C.byref(gw), None, None, None, None, 0, None, C.byref(gw), None, None),
    }
    res = {}
    for calls, make in ((dec, lambda: dec_desc("bench", 7, L.CELL_LSTM, 1)), (loc, lambda: loc_desc("bench", 7, L.CELL_LSTM, 1)),
                        (glob, lambda: glob_desc(7))):
        for name, f in calls.items():
            res[name] = [f(None), f(C.byref(make()))]
    return res


def switches():
    d = C.byref(dec_desc("bench", L.PREC_BF16, L.CELL_LSTM, 1))
    out = (C.c_int32 * 12)()
    lib.recnet_plan_persistent_loops(C.byref(loc_desc("bench", L.PREC_BF16, L.CELL_LSTM, 1)), out)
    return {"bwd_is_split": lib.recnet_decoder_bwd_is_split(d), "decoder_workspace_bytes": lib.recnet_decoder_workspace_bytes(d),
            "persistent_loops": list(out)}


print(json.dumps(globals()[sys.argv[2]]()))
'''


def _child(what, **switches):
    env = {k: v for k, v in os.environ.items() if not k.startswith("RECNET_")}
    env.update(switches)
    r = subprocess.run([sys.executable, "-c", _CHILD, L.__file__, what], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    return json.loads(r.stdout)


# decoder rows: decoder_workspace_bytes, greedy_workspace_bytes, beam_workspace_bytes(., 3, 31), decoder_bwd_is_split,
#               decoder_error_offset, logits ld, logits offset from the workspace base
# local rows:   local_workspace_bytes, local_error_offset, local_outputs offset, plan_persistent_loops status, its 12 outputs
# global rows:  global_workspace_bytes, global_error_offset, global_outputs offset
GOLDEN = {
    'dec/bench/bf16/GRU+softmax/n1': [266208000, 94646016, 94673808, 0, 266207488, 4188, 116458752],
    'dec/bench/bf16/GRU+softmax/n2': [315663104, 107237120, 107264912, 0, 266207488, 4188, 116458752],
    'dec/bench/bf16/GRU/n1': [266208000, 94646016, 94673808, 0, 266207488, 4188, 116458752],
    'dec/bench/bf16/GRU/n2': [315663104, 107237120, 107264912, 0, 266207488, 4188, 116458752],
    'dec/bench/bf16/LSTM+softmax/n1': [271622912, 104257024, 80440976, 1, 271622400, 4188, 93316352],
    'dec/bench/bf16/LSTM+softmax/n2': [292214272, 93004288, 93032080, 0, 242758656, 4188, 108267008],
    'dec/bench/bf16/LSTM/n1': [271622912, 104257024, 80440976, 1, 271622400, 4188, 93316352],
    'dec/bench/bf16/LSTM/n2': [292214272, 93004288, 93032080, 0, 242758656, 4188, 108267008],
    'dec/bench/fp32/GRU+softmax/n1': [357117440, 111539712, 111567504, 0, 357116928, 4188, 162288128],
    'dec/bench/fp32/GRU+softmax/n2': [439848448, 126686720, 126714512, 0, 357116928, 4188, 162288128],
    'dec/bench/fp32/GRU/n1': [357117440, 111539712, 111567504, 0, 357116928, 4188, 162288128],
    'dec/bench/fp32/GRU/n2': [439848448, 126686720, 126714512, 0, 357116928, 4188, 162288128],
    'dec/bench/fp32/LSTM+softmax/n1': [375434752, 100686080, 100713872, 1, 375434240, 4188, 146928128],
    'dec/bench/fp32/LSTM+softmax/n2': [410562816, 115833088, 115860880, 0, 327831296, 4188, 156963584],
    'dec/bench/fp32/LSTM/n1': [375434752, 100686080, 100713872, 1, 375434240, 4188, 146928128],
    'dec/bench/fp32/LSTM/n2': [410562816, 115833088, 115860880, 0, 327831296, 4188, 156963584],
    'dec/small/bf16/GRU+softmax/n1': [19432192, 19425408, 19427856, 0, 19431680, 12, 23040],
    'dec/small/bf16/GRU+softmax/n2': [19436160, 19427968, 19430416, 0, 19431680, 12, 23040],
    'dec/small/bf16/GRU/n1': [19432192, 19425408, 19427856, 0, 19431680, 12, 23040],
    'dec/small/bf16/GRU/n2': [19436160, 19427968, 19430416, 0, 19431680, 12, 23040],
    'dec/small/bf16/LSTM+softmax/n1': [19431424, 19425152, 19427600, 0, 19430912, 12, 22784],
    'dec/small/bf16/LSTM+softmax/n2': [19435392, 19427712, 19430160, 0, 19430912, 12, 22784],
    'dec/small/bf16/LSTM/n1': [19431424, 19425152, 19427600, 0, 19430912, 12, 22784],
    'dec/small/bf16/LSTM/n2': [19435392, 19427712, 19430160, 0, 19430912, 12, 22784],
    'dec/small/fp32/GRU+softmax/n1': [19431680, 19425152, 19427600, 0, 19431168, 12, 23040],
    'dec/small/fp32/GRU+softmax/n2': [19438720, 19429504, 19431952, 0, 19431168, 12, 23040],
    'dec/small/fp32/GRU/n1': [19431680, 19425152, 19427600, 0, 19431168, 12, 23040],
    'dec/small/fp32/GRU/n2': [19438720, 19429504, 19431952, 0, 19431168, 12, 23040],
    'dec/small/fp32/LSTM+softmax/n1': [19430400, 19424640, 19427088, 0, 19429888, 12, 22784],
    'dec/small/fp32/LSTM+softmax/n2': [19437440, 19428992, 19431440, 0, 19429888, 12, 22784],
    'dec/small/fp32/LSTM/n1': [19430400, 19424640, 19427088, 0, 19429888, 12, 22784],
    'dec/small/fp32/LSTM/n2': [19437440, 19428992, 19431440, 0, 19429888, 12, 22784],
    'glob/bf16': [327876352, 320486144, 193871872],
    'glob/fp32': [449966080, 449948416, 279404544],
    'loc/bench/bf16/GRU+softmax/n1': [294982400, 294963968, 118666496, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/bench/bf16/GRU+softmax/n2': [495984896, 478763776, 188981504, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/bench/bf16/GRU/n1': [294982400, 294963968, 118666496, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/bench/bf16/GRU/n2': [495984896, 478763776, 188981504, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/bench/bf16/LSTM+softmax/n1': [254483456, 244583936, 108836352, 0, 1, 3, 48, 11, 3, 144, 1, 9, 16, 11, 3, 144],
    'loc/bench/bf16/LSTM+softmax/n2': [419800064, 402578944, 179151360, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/bench/bf16/LSTM/n1': [254483456, 244583936, 108836352, 0, 1, 3, 48, 11, 3, 144, 1, 9, 16, 11, 3, 144],
    'loc/bench/bf16/LSTM/n2': [419800064, 402578944, 179151360, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/bench/fp32/GRU+softmax/n1': [432885504, 432867072, 189932800, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/bench/fp32/GRU+softmax/n2': [770464000, 736039680, 309297408, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/bench/fp32/GRU/n1': [432885504, 432867072, 189932800, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/bench/fp32/GRU/n2': [770464000, 736039680, 309297408, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/bench/fp32/LSTM+softmax/n1': [359977472, 359959040, 183789056, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/bench/fp32/LSTM+softmax/n2': [645946368, 611522048, 303153664, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/bench/fp32/LSTM/n1': [359977472, 359959040, 183789056, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/bench/fp32/LSTM/n2': [645946368, 611522048, 303153664, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/bf16/GRU+softmax/n1': [38843136, 38824704, 13056, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/bf16/GRU+softmax/n2': [38860032, 38840576, 19712, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/bf16/GRU/n1': [38843136, 38824704, 13056, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/bf16/GRU/n2': [38860032, 38840576, 19712, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/bf16/LSTM+softmax/n1': [38840832, 38822400, 12544, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/bf16/LSTM+softmax/n2': [38855936, 38836480, 19200, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/bf16/LSTM/n1': [38840832, 38822400, 12544, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/bf16/LSTM/n2': [38855936, 38836480, 19200, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/fp32/GRU+softmax/n1': [38856192, 38837760, 20736, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/fp32/GRU+softmax/n2': [38883328, 38862848, 30976, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/fp32/GRU/n1': [38856192, 38837760, 20736, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/fp32/GRU/n2': [38883328, 38862848, 30976, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/fp32/LSTM+softmax/n1': [38852096, 38833664, 20224, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/fp32/LSTM+softmax/n2': [38875392, 38854912, 30464, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/fp32/LSTM/n1': [38852096, 38833664, 20224, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
    'loc/small/fp32/LSTM/n2': [38875392, 38854912, 30464, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0],
}

# decoder_workspace_bytes of the bench decoder (bf16, LSTM, one layer) under RECNET_PF=0: the general plan's size
GOLDEN_PF_OFF = 242759168

BAD_SHAPE, UNSUPPORTED = -1, -4


def test_plans_match_the_recorded_table():
    got = _child("golden")
    assert sorted(got) == sorted(GOLDEN)
    assert {k: v for k, v in got.items() if v != GOLDEN[k]} == {}


def test_invalid_descriptors_are_rejected_alike():
    got = _child("invalid")
    for name, (null, bad_prec) in got.items():
        if name == "recnet_decoder_bwd_is_split":              # a yes/no query: an invalid descriptor is not split
            assert (null, bad_prec) == (0, 0), name
        elif name in ("recnet_decoder_logits", "recnet_local_outputs", "recnet_global_outputs"):
            assert (null, bad_prec) == (None, None), name
        else:
            assert (null, bad_prec) == (BAD_SHAPE, UNSUPPORTED), name
    assert len(got) == 24


def test_switches_are_still_read():
    default = _child("switches")
    assert default["bwd_is_split"] == 1 and default["decoder_workspace_bytes"] == GOLDEN["dec/bench/bf16/LSTM/n1"][0]
    no_pf = _child("switches", RECNET_PF="0")
    assert no_pf["bwd_is_split"] == 0 and no_pf["decoder_workspace_bytes"] == GOLDEN_PF_OFF
    no_bwd = _child("switches", RECNET_PERSIST_BWD="0")
    assert default["persistent_loops"][0] == 1 and default["persistent_loops"][6] == 1
    assert no_bwd["persistent_loops"][6] == 0 and no_bwd["persistent_loops"][:6] == default["persistent_loops"][:6]
