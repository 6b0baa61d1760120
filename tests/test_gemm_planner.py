"""The tile / split-K plan of the batched GEMMs (csrc/runtime.cuh:plan_gemm_full<bf16>) is host code: pin its decisions for the shapes of the
MSVD train step to what the sweeps on the B200 found best (profiles/r2_h_gemm_sweep.md, r1_g_gemm_sweep.md).  No GPU needed."""
import ctypes as C

import pytest

import recnet_b200  # noqa: F401
from recnet_b200 import _lib as L
from tests.test_gpu_loop_shapes import REC_CASES as LOOP_CASES

B, T, E, H, A, V, Lr, R = 100, 28, 1536, 512, 128, 4188, 31, 1536
LB, BT, SB, GR = Lr * B, B * T, 28 * B, 4 * R


def plan(M, N, K, prec=L.PREC_BF16):
    bn, splits = C.c_int32(), C.c_int32()
    L.check(L.lib().recnet_plan_batched_gemm(prec, M, N, K, C.byref(bn), C.byref(splits)), "recnet_plan_batched_gemm")
    return bn.value, splits.value


@pytest.mark.parametrize("name,shape,expect", [
    ("rec.dW_hh: the one GEMM with >= 1.5 rounds of pair tiles and a long K loop", (GR, R, SB), 2256),
    ("dec.logits: K = 512, many tiles", (LB, V, H), 1256),
    ("dec.Gx", (LB, 4 * H, 512), 1256),
    ("dec.VW", (BT, 4 * H, E), 1256),
    ("rec.out", (SB, R, R), 1256),
    ("rec.dW_ih: 96 tiles of 256", (GR, H, SB), 1256),
    ("dec.dW_ctx", (4 * H, E, LB), 1256),
    ("rec.out_w: 72 tiles of 256 -> 128-wide", (R, R, SB), 1128),
    ("dec.out_w", (V, H, LB), 1128),
    ("dec.dHext", (LB, H, 4192), 1128),
    ("dec.dXe", (LB, 468, 4 * H), 1128),
])
def test_persistent_kernel_plans(name, shape, expect):
    bn, splits = plan(*shape)
    assert (bn, splits) == (expect, 1), name


@pytest.mark.parametrize("name,shape", [
    ("dec.dW_a", (A, H, LB)), ("dec.dU", (A, E, BT)), ("rec.attn_W", (A, R, SB)), ("rec.attn_U", (A, H, LB)),
])
def test_skinny_attention_gradients_stay_on_split_k(name, shape):
    bn, splits = plan(*shape)
    assert bn == 64 and splits >= 4, (name, bn, splits)


@pytest.mark.parametrize("shape", [(BT, A, E), (LB, A, H)])
def test_128_column_key_projections_stay_on_the_one_tile_kernel(shape):
    bn, splits = plan(*shape)
    assert bn in (64, 128) and splits == 1


def test_background_budget_limits_split_k_plans():
    lib = L.lib()
    free = plan(A, R, SB)
    L.check(lib.recnet_set_background_ctas(48), "recnet_set_background_ctas")
    try:
        bn, splits = plan(A, R, SB)
        assert bn in (64, 128) and -(-R // bn) * splits <= 48, (bn, splits)   # N-tiles x splits within the lane's budget
        assert plan(GR, R, SB) == (2256, 1)                                  # persistent kernels are capped at launch, not re-planned
    finally:
        lib.recnet_set_background_ctas(0)
    assert plan(A, R, SB) == free
    assert lib.recnet_set_background_ctas(-1) < 0


def test_rejects_empty_shapes():
    bn, splits = C.c_int32(), C.c_int32()
    assert L.lib().recnet_plan_batched_gemm(L.PREC_BF16, 0, 8, 8, C.byref(bn), C.byref(splits)) < 0


def _loops(**kw):
    base = dict(B=100, S=28, R=1536, H=512, A=128, L=31, precision=L.PREC_BF16, train=1, p_drop=0.5, cell=L.CELL_LSTM, dec_layers=1)
    base.update(kw)
    d = L.local_desc(**base)
    out = (C.c_int32 * 12)()
    L.check(L.lib().recnet_plan_persistent_loops(C.byref(d), out), "recnet_plan_persistent_loops")
    return list(out)


def test_persistent_loop_layout_of_the_msvd_shape():
    """DESIGN.md 3a: 144 CTAs = 48 unit groups x 3 K-splits forward (11 resident k-blocks = 176 KB of weights per CTA), 16 column groups x 9
    gate-row splits backward."""
    o = _loops()
    assert o[:4] == [1, 3, 48, 11] and o[4] >= 3 and o[5] == 144
    assert o[6:10] == [1, 9, 16, 11] and o[10] >= 2 and o[11] == 144


@pytest.mark.parametrize("kw", [dict(R=3584, H=512), dict(precision=L.PREC_FP32), dict(cell=L.CELL_GRU), dict(A=256), dict(L=40), dict(B=200),
                                dict(dec_layers=2)])
def test_shapes_outside_the_persistent_loops_take_the_kernel_per_phase_path(kw):
    o = _loops(**kw)
    assert o[0] == 0 and o[6] == 0, (kw, o)


def _global_loops(B, L_, R, H):
    d = L.global_desc(B=B, L=L_, R=R, H=H, T=28, precision=L.PREC_BF16, train=1, p_drop=0.5, caption_max_len=30.0, cell=L.CELL_LSTM,
                      dec_layers=1)
    out = (C.c_int32 * 12)()
    L.check(L.lib().recnet_plan_global_loops(C.byref(d), out), "recnet_plan_global_loops")
    return list(out)


@pytest.mark.parametrize("cid", sorted(LOOP_CASES))
def test_loop_shape_cases_keep_the_layout_the_gpu_tests_expect(cid):
    """tests/test_gpu_loop_shapes.py asserts on the GPU which loop each case runs and with how many CTAs; the planners decide that on the
    host, so a planner change that moves a case fails here first."""
    c = LOOP_CASES[cid]
    if c.kind == "local":
        o = _loops(B=c.B, S=c.S, R=c.R, H=c.H, A=128, L=c.L)
    else:
        o = _global_loops(c.B, c.L, c.R, c.H)
    assert (bool(o[0]), bool(o[6])) == (c.fwd is not None, c.bwd is not None), (cid, o)
    if c.fwd:
        assert (o[1], o[5]) == c.fwd and o[5] == o[2] * o[1] <= 148 and o[4] >= 2, (cid, o)
    if c.bwd:
        assert (o[7], o[11]) == c.bwd and o[11] == o[8] * o[7] <= 148 and o[10] >= 2, (cid, o)


def test_loop_shape_cases_reach_the_edges_they_are_named_for():
    R3, R4, R5, G2 = (LOOP_CASES[k] for k in ("R3", "R4", "R5", "G2"))
    assert _loops(B=R3.B, R=R3.R, H=R3.H)[4] == 2                                   # 2-stage ring at B > 112
    assert R4.B == 128 and R4.L == 32
    assert R5.B == R5.fwd[1] and _loops(B=R5.B + 1, R=R5.R, H=R5.H)[0] == 0        # B = UG x KS is the local forward's last batch
    assert G2.B > G2.fwd[1] and _loops(B=G2.B, R=G2.R, H=0, L=G2.L)[0] == 0       # only global mode runs B > UG x KS
    assert _global_loops(129, 31, 1536, 512)[0] == 0 and _global_loops(129, 31, 1536, 512)[6] == 0


def test_global_loop_probe_rejects_bad_descriptors():
    out = (C.c_int32 * 12)()
    assert L.lib().recnet_plan_global_loops(None, out) < 0
    d = L.global_desc(B=8, L=4, R=512, H=128, T=4, precision=7, train=0, p_drop=0.0, caption_max_len=30.0, cell=L.CELL_LSTM, dec_layers=1)
    assert L.lib().recnet_plan_global_loops(C.byref(d), out) == -4                 # RECNET_ERR_UNSUPPORTED
    d.precision = L.PREC_FP32
    assert L.lib().recnet_plan_global_loops(C.byref(d), out) == 0 and list(out) == [0] * 12


def test_smaller_batches_and_widths_stay_covered():
    assert _loops(B=64)[0] == 1 and _loops(B=64)[6] == 1
    o = _loops(R=1024, H=512, B=64)             # (B = 100 at R = 1024 is NOT covered: the forward needs B <= unit groups x K-splits = 96)
    assert o[0] == 1 and o[5] <= 148 and o[6] == 1 and o[11] <= 148
    assert _loops(R=1024, H=512)[0] == 0
