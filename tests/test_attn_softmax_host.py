"""CPU checks of the opt-in softmax attention (``attn_softmax``): the fp64 oracle restatement against an independent one and against
autograd's numerical gradient, the Python surface (constructors, state_dict, config, builders) and the C-ABI flag handling."""
import ctypes as C

import pytest
import torch

import recnet_b200
from recnet_b200 import _lib as L
from recnet_b200 import models as M
from recnet_b200 import train as T
from recnet_b200.config import TrainConfig
from oracle import recnet_oracle as O
from tests import attn_softmax_oracle as S


def _dec_params(NL, model_name="LSTM", dtype=torch.float64):
    return O.init_decoder_params(11, 5, 6, 4, 3, n_layers=NL, model_name=model_name, seed=7, dtype=dtype)


@pytest.mark.parametrize("NL", [1, 2])
def test_oracle_decoder_step_equals_functional_softmax_restatement(NL):
    P = _dec_params(NL)
    g = torch.Generator().manual_seed(NL)
    feats = torch.randn(2, 5, 6, generator=g, dtype=torch.float64)
    hidden = (torch.randn(NL, 2, 4, generator=g, dtype=torch.float64), torch.randn(NL, 2, 4, generator=g, dtype=torch.float64))
    tok = torch.tensor([[3, 7]])
    logits, (h, c) = S.decoder_step(P, tok, hidden, feats, n_layers=NL, attn_softmax=True)
    # independent restatement: scores per frame, torch.nn.functional.softmax, context as a batched matrix product
    scores = torch.stack([torch.tanh(hidden[0][-1] @ P["attn_W.weight"].t() + feats[:, t] @ P["attn_U.weight"].t() + P["attn_b"])
                          @ P["attn_w.weight"][0] for t in range(5)], dim=1)                     # (B,T)
    ctx = torch.bmm(torch.nn.functional.softmax(scores, dim=1).unsqueeze(1), feats).squeeze(1)
    x = torch.cat((P["embedding.weight"][tok[0]], ctx), dim=1)
    hs, cs = [], []
    for l in range(NL):
        pre = x @ P[f"rnn.weight_ih_l{l}"].t() + P[f"rnn.bias_ih_l{l}"] + hidden[0][l] @ P[f"rnn.weight_hh_l{l}"].t() + P[f"rnn.bias_hh_l{l}"]
        i, f, gg, o = pre.chunk(4, dim=1)
        cl = torch.sigmoid(f) * hidden[1][l] + torch.sigmoid(i) * torch.tanh(gg)
        x = torch.sigmoid(o) * torch.tanh(cl)
        hs.append(x); cs.append(cl)
    assert torch.allclose(h, torch.stack(hs), atol=1e-12) and torch.allclose(c, torch.stack(cs), atol=1e-12)
    assert torch.allclose(logits, x @ P["out.weight"].t() + P["out.bias"], atol=1e-12)
    # and it is NOT the reference's mean attention
    ref_logits, _ = O.decoder_step(P, tok, hidden, feats, n_layers=NL)
    assert not torch.allclose(logits, ref_logits)


@pytest.mark.parametrize("NLd", [1, 2])
def test_oracle_local_step_equals_functional_softmax_restatement(NLd):
    Q = O.init_reconstructor_params("local", 4, 6, 3, seed=2, dtype=torch.float64)
    g = torch.Generator().manual_seed(10 + NLd)
    dh = torch.randn(5, NLd, 2, 4, generator=g, dtype=torch.float64)          # (L, NLdec, B, H)
    hidden = (torch.randn(1, 2, 6, generator=g, dtype=torch.float64), torch.randn(1, 2, 6, generator=g, dtype=torch.float64))
    out, _ = S.local_reconstructor_step(Q, hidden, dh, attn_softmax=True)
    q = hidden[0][-1] @ Q["attn_W.weight"].t()
    xs = []
    for j in range(NLd):                                                        # one softmax over L per decoder layer
        sc = torch.stack([torch.tanh(q + dh[l, j] @ Q["attn_U.weight"].t() + Q["attn_b"]) @ Q["attn_w.weight"][0] for l in range(5)], 1)
        xs.append(torch.bmm(torch.nn.functional.softmax(sc, dim=1).unsqueeze(1), dh[:, j].transpose(0, 1)).squeeze(1))
    pre = xs[0] @ Q["rnn.weight_ih_l0"].t() + Q["rnn.bias_ih_l0"] + hidden[0][0] @ Q["rnn.weight_hh_l0"].t() + Q["rnn.bias_hh_l0"]
    i, f, gg, o = pre.chunk(4, dim=1)
    h1 = torch.sigmoid(o) * torch.tanh(torch.sigmoid(f) * hidden[1][0] + torch.sigmoid(i) * torch.tanh(gg))
    assert torch.allclose(out, h1 @ Q["out.weight"].t() + Q["out.bias"], atol=1e-12)


def test_oracle_softmax_steps_pass_gradcheck():
    P = _dec_params(1)
    names = ["attn_W.weight", "attn_U.weight", "attn_b", "attn_w.weight", "rnn.weight_ih_l0"]
    g = torch.Generator().manual_seed(3)
    feats = torch.randn(2, 4, 6, generator=g, dtype=torch.float64, requires_grad=True)
    h0 = torch.randn(1, 2, 4, generator=g, dtype=torch.float64)
    c0 = torch.randn(1, 2, 4, generator=g, dtype=torch.float64)

    def dec_fn(f, *ws):
        Q = dict(P, **dict(zip(names, ws)))
        return S.decoder_step(Q, torch.tensor([[1, 2]]), (h0, c0), f, attn_softmax=True)[0]

    assert torch.autograd.gradcheck(dec_fn, (feats, *[P[n].clone().requires_grad_(True) for n in names]))
    R = O.init_reconstructor_params("local", 4, 5, 3, seed=4, dtype=torch.float64)
    rnames = ["attn_W.weight", "attn_U.weight", "attn_b", "attn_w.weight"]
    dh = torch.randn(4, 1, 2, 4, generator=g, dtype=torch.float64, requires_grad=True)
    hr = (torch.randn(1, 2, 5, generator=g, dtype=torch.float64), torch.randn(1, 2, 5, generator=g, dtype=torch.float64))

    def loc_fn(d, *ws):
        Q = dict(R, **dict(zip(rnames, ws)))
        return S.local_reconstructor_step(Q, hr, d, attn_softmax=True)[0]

    assert torch.autograd.gradcheck(loc_fn, (dh, *[R[n].clone().requires_grad_(True) for n in rnames]))


def test_oracle_flag_off_is_the_oracle():
    assert S.decoder_step(_dec_params(1), torch.tensor([[1]]), O.zero_hidden("LSTM", 1, 1, 4, torch.zeros(1, dtype=torch.float64)),
                          torch.ones(1, 3, 6, dtype=torch.float64))[0].shape == (1, 11)
    assert O.decoder_step is not S.decoder_step_softmax and O.local_reconstructor_step is not S.local_reconstructor_step_softmax


def _dec(flag, name="LSTM", NL=1):
    return M.Decoder(name, NL, 16, 8, 1, 8, 4, 20, 0.5, 0.5, 0.5, precision="fp32", attn_softmax=flag)


def _loc(flag):
    return M.LocalReconstructor("LSTM", 1, 8, 16, 0.5, 0.5, 4, precision="fp32", attn_softmax=flag)


@pytest.mark.parametrize("name,NL", [("LSTM", 1), ("LSTM", 2), ("GRU", 1)])
def test_modules_construct_on_cpu_with_identical_state_dicts(name, NL):
    a, b = _dec(False, name, NL), _dec(True, name, NL)
    assert not a.attn_softmax and b.attn_softmax
    assert {k: v.shape for k, v in a.state_dict().items()} == {k: v.shape for k, v in b.state_dict().items()}
    b.load_state_dict(a.state_dict())                                          # checkpoints interchangeable both ways
    a.load_state_dict(b.state_dict())
    assert b.uses_fused_sequence == a.uses_fused_sequence                      # every fused driver has the softmax variant
    ra, rb = _loc(False), _loc(True)
    assert {k: v.shape for k, v in ra.state_dict().items()} == {k: v.shape for k, v in rb.state_dict().items()}
    h = torch.zeros(5, NL, 2, 8)
    assert ra._fused_ok(h) == rb._fused_ok(h)
    assert b._meta()["cell"] == a._meta()["cell"] | L.ATTN_SOFTMAX


def test_positional_signature_is_the_references():
    d = M.Decoder("LSTM", 1, 16, 8, 1, 8, 4, 20, 0.5, 0.5, 0.5, "fp32")       # precision still the 12th positional argument
    assert d.precision == "fp32" and not d.attn_softmax


def test_config_defaults_are_the_reference_attention():
    assert TrainConfig.decoder_attn_softmax is False and TrainConfig.reconstructor_attn_softmax is False


@pytest.mark.parametrize("flag", [False, True])
def test_builders_pass_the_flags_through(flag, monkeypatch):
    C_ = T.C
    for k, v in dict(device="cpu", decoder_attn_softmax=flag, reconstructor_attn_softmax=not flag, reconstructor_type="local",
                     decoder_model="LSTM", reconstructor_model="LSTM", optimizer_impl="torch").items():
        monkeypatch.setattr(C_, k, v, raising=False)
    monkeypatch.setenv("RECNET_OPTIMIZER", "torch")
    try:
        dec = T.build_decoder(50)
        rec = T.build_reconstructor()
    except RuntimeError as e:                   # an optimiser that insists on CUDA tensors: the module was built before it
        pytest.skip(f"optimiser needs CUDA: {e}")
    assert dec["model"].attn_softmax is flag and rec["model"].attn_softmax is (not flag)


# ---- C ABI ------------------------------------------------------------------------------------------------------
def _local_desc(cell):
    return L.local_desc(B=100, S=28, R=1536, H=512, A=128, L=31, precision=L.PREC_BF16, train=1, p_drop=0.5, cell=cell, dec_layers=1)


def _dec_desc(cell, precision=L.PREC_BF16):
    return L.decoder_desc(B=100, T=28, E=1536, H=512, A=128, EMB=468, V=4188, L=31, precision=precision, train=1, embedding_scale=1.0,
                          p_emb_drop=0.5, p_out_drop=0.5, cell=cell, n_layers=1, p_layer_drop=0.0)


def test_abi_constants():
    assert L.ATTN_SOFTMAX == 0x100 and L.lib().recnet_abi_version() == 1


def test_persistent_loop_planner_covers_the_bench_configuration_with_softmax():
    lib = L.lib()
    a, b = (C.c_int32 * 12)(), (C.c_int32 * 12)()
    assert lib.recnet_plan_persistent_loops(C.byref(_local_desc(L.CELL_LSTM)), a) == 0
    assert lib.recnet_plan_persistent_loops(C.byref(_local_desc(L.CELL_LSTM | L.ATTN_SOFTMAX)), b) == 0
    assert list(a) == list(b) and a[0] == 1 and a[6] == 1


@pytest.mark.parametrize("precision", [L.PREC_FP32, L.PREC_BF16])
def test_workspace_queries_accept_the_flag(precision):
    lib = L.lib()
    for cell in (L.CELL_LSTM, L.CELL_GRU):
        d0, d1 = _dec_desc(cell, precision), _dec_desc(cell | L.ATTN_SOFTMAX, precision)
        assert lib.recnet_decoder_workspace_bytes(C.byref(d1)) == lib.recnet_decoder_workspace_bytes(C.byref(d0)) > 0
        assert lib.recnet_greedy_workspace_bytes(C.byref(d1)) == lib.recnet_greedy_workspace_bytes(C.byref(d0)) > 0
        assert lib.recnet_beam_workspace_bytes(C.byref(d1), 5, 31) == lib.recnet_beam_workspace_bytes(C.byref(d0), 5, 31) > 0
        assert lib.recnet_decoder_bwd_is_split(C.byref(d1)) == lib.recnet_decoder_bwd_is_split(C.byref(d0))
    l0, l1 = _local_desc(L.CELL_LSTM), _local_desc(L.CELL_LSTM | L.ATTN_SOFTMAX)
    l0.precision = l1.precision = precision
    assert lib.recnet_local_workspace_bytes(C.byref(l1)) == lib.recnet_local_workspace_bytes(C.byref(l0)) > 0
    assert lib.recnet_local_error_offset(C.byref(l1)) == lib.recnet_local_error_offset(C.byref(l0))


@pytest.mark.parametrize("bad", [0x200, 0x10000, 0x100 | 0x400])
def test_unknown_flag_bits_are_unsupported(bad):
    lib = L.lib()
    out = (C.c_int32 * 12)()
    assert lib.recnet_plan_persistent_loops(C.byref(_local_desc(L.CELL_LSTM | bad)), out) == -4
    assert lib.recnet_local_workspace_bytes(C.byref(_local_desc(L.CELL_LSTM | bad))) == -4
    assert lib.recnet_decoder_workspace_bytes(C.byref(_dec_desc(L.CELL_LSTM | bad))) == -4
    assert lib.recnet_greedy_workspace_bytes(C.byref(_dec_desc(L.CELL_LSTM | bad))) == -4
    assert lib.recnet_beam_workspace_bytes(C.byref(_dec_desc(L.CELL_LSTM | bad)), 3, 31) == -4


def test_softmax_backward_symbol_is_declared_and_bound():
    from tests.test_abi import _declared
    decl = _declared()
    assert decl["recnet_attn_bwd_softmax"] == decl["recnet_attn_bwd"] + 1 == len(L.SIGNATURES["recnet_attn_bwd_softmax"][1])
    assert hasattr(C.CDLL(L.LIB_PATH), "recnet_attn_bwd_softmax")
