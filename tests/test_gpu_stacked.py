"""GPU parity of stacked LSTM decoders (n_layers = 2..4) on the fused kernel-per-phase drivers (csrc/seq_decoder.cuh, the
stacked branches of csrc/seq_recon.cuh) against the fp64 CPU oracle, through the public modules:
  * depth: 3 and 4 layers in eval mode -- the middle layers run code that 2 layers never reach (the forward's write into the
    input slot of the layer above, the backward's non-top layers >= 1, the local reconstructor over an odd number of layers);
  * train mode with the kernels' Philox masks at every site, including the inter-layer dropout (sites 17, 18) that the
    oracle restates in tests/stacked_oracle.py;
  * the benchmarked step (bench.py msrvtt_stress): 2 layers, local reconstructor, train.train_step as bench.py runs it.
Tolerances as everywhere: fp32 1e-3, bf16 2e-2 relative to the tensor's max.  Each case prints its worst relative error."""
import pytest
import torch

import recnet_b200
from recnet_b200 import functional as Fn
from recnet_b200 import train as T
from oracle import recnet_oracle as O
from tests import stacked_oracle as SO
from tests.test_gpu_parity import TOL, build, dev, rel

pytestmark = pytest.mark.gpu

D = torch.float64
# odd batch, 19 frames, ragged captions (seed 7: the loop stops after 12 of the 13 steps)
MID = dict(B=13, T=19, E=512, H=256, A=128, EMB=96, V=700, cap_len=12, rec_layers=1, dec_model="LSTM", rec_model="LSTM")
# bench.py msrvtt_stress widths at the full caption length; batch 8 and V = 600 keep the oracle at ~11 s
STRESS = dict(B=8, T=40, E=3584, H=512, A=128, EMB=468, V=600, cap_len=30, dec_layers=2, rec_layers=1, dec_model="LSTM",
              rec_model="LSTM")
SEEDS = {"dec": 0xDEC0, "local": 0x10CA, "global": 0x610B}


def _problem(m, kind, seed, full_length_first):
    feats, targets, masks = O.synthetic_batch(m["B"], m["T"], m["E"], m["V"], m["cap_len"], seed=seed, full_length_first=full_length_first,
                                              dtype=D)
    P = O.init_decoder_params(m["V"], m["EMB"], m["E"], m["H"], m["A"], n_layers=m["dec_layers"], seed=4, dtype=D)
    Q = O.init_reconstructor_params(kind, m["H"], m["E"], m["A"], seed=5, dtype=D) if kind != "none" else {}
    return (feats, targets, masks), P, Q


def _masks(m, kind):
    return SO.train_mode_masks(T.C, SEEDS, kind, L=m["cap_len"] + 1, B=m["B"], EMB=m["EMB"], V=m["V"], H=m["H"], S=m["T"],
                               n_layers=m["dec_layers"])


def _oracle(m, kind, inputs, P, Q, drops=None):
    """fp64 losses, hiddens, logits and gradients; drops = train_mode_masks(...) or None (eval mode)."""
    feats, targets, masks = inputs
    d = drops or {}
    Pr = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    Qr = {k: v.clone().requires_grad_(True) for k, v in Q.items()}
    dl, hid, _, aux = SO.forward_decoder(Pr, feats, targets, masks, n_layers=m["dec_layers"], caption_max_len=m["cap_len"],
                                         drop_emb=d.get("emb"), drop_logits=d.get("logits"), drop_layer=d.get("layer"))
    rl = None
    if kind == "local":
        rl, _ = O.forward_local_reconstructor(Qr, hid, feats, drop_x=d.get("x"))
    elif kind == "global":
        rl, _ = O.forward_global_reconstructor(Qr, hid, feats, caption_max_len=m["cap_len"], drop_mp=d.get("mp"))
    (dl if rl is None else dl + rl).backward()
    return dict(dl=dl.detach(), rl=None if rl is None else rl.detach(), hid=hid.detach(), logits=aux["logits"].detach(),
                gP={k: v.grad for k, v in Pr.items()}, gQ={k: v.grad for k, v in Qr.items()})


_CACHE = {}


def _case(NL, kind, train):
    """Inputs, weights and oracle of one mid-shape case, shared by its fp32 and bf16 runs."""
    key = (NL, kind, train)
    if key not in _CACHE:
        m = dict(MID, dec_layers=NL)
        inputs, P, Q = _problem(m, kind, seed=7, full_length_first=False)
        _CACHE[key] = (m, inputs, P, Q, _oracle(m, kind, inputs, P, Q, _masks(m, kind) if train else None))
    return _CACHE[key]


def _build(m, precision, kind, P, Q, train):
    dec, rec = build(m, precision, kind, P, Q)
    assert dec["model"].n_layers == m["dec_layers"] and dec["model"].uses_fused_sequence
    if rec is not None:
        assert rec["model"]._fused_ok(torch.empty(1, m["dec_layers"], 1, 1))
    if train:
        C = T.C
        assert min(C.embedding_dropout, C.decoder_out_dropout, C.decoder_dropout, C.reconstructor_decoder_dropout) > 0
        assert dec["model"].dropout_p == C.decoder_dropout
        dec["model"].train(); dec["model"].seed_dropout(SEEDS["dec"])
        if rec is not None:
            rec["model"].train(); rec["model"].seed_dropout(SEEDS[kind])
    return dec, rec


def _errors(o, dloss, rloss, dec, rec, hiddens=None):
    errs = {"dec_loss": rel(dloss, o["dl"])}
    if hiddens is not None:
        assert hiddens.shape == o["hid"].shape, (hiddens.shape, o["hid"].shape)
        errs["hiddens"] = rel(hiddens, o["hid"])
    if rec is not None:
        errs["rec_loss"] = rel(rloss, o["rl"])
    named = {"dec." + k: (p, o["gP"][k]) for k, p in dec["model"].named_parameters()}
    if rec is not None:
        named.update({"rec." + k: (p, o["gQ"][k]) for k, p in rec["model"].named_parameters()})
    assert {k[4:] for k in named if k.startswith("dec.")} == set(o["gP"])
    for k, (p, ref) in named.items():
        assert p.grad is not None, k
        errs[k] = rel(p.grad, ref)
    return errs


def _check(tag, errs, tol):
    worst = max(errs, key=errs.get)
    print(f"[stacked] {tag}: worst rel err {errs[worst]:.3e} ({worst})")
    assert errs[worst] < tol, (worst, errs[worst])


def _step(m, kind, precision, inputs, P, Q, train):
    dec, rec = _build(m, precision, kind, P, Q, train)
    feats, targets, masks = (x.to(dev()) for x in inputs)
    feats = feats.float()
    dloss, hiddens, _ = T.forward_decoder(dec, feats, targets, masks, 1.0)
    rloss = T.forward_reconstructor_for(kind)(hiddens, feats, rec) if rec is not None else None
    (dloss if rloss is None else dloss + rloss).backward()
    Fn.check_loop_status()
    return dec, rec, feats, targets, dloss, rloss, hiddens


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", ["none", "global", "local"])
@pytest.mark.parametrize("NL", [3, 4])
def test_deep_decoder_eval_mode_matches_the_fp64_oracle(NL, kind, precision):
    m, inputs, P, Q, o = _case(NL, kind, train=False)
    dec, rec, feats, targets, dloss, rloss, hiddens = _step(m, kind, precision, inputs, P, Q, train=False)
    errs = _errors(o, dloss, rloss, dec, rec, hiddens)
    assert all(f"dec.rnn.weight_ih_l{l}" in errs for l in range(NL))
    if kind == "none":
        Lsteps = o["hid"].shape[0]
        tokens_in = torch.cat((torch.ones(1, m["B"], dtype=torch.long, device=dev()), targets[: Lsteps - 1]), 0)
        logits, hid2 = dec["model"].teacher_forced_logits(tokens_in, feats)
        errs["teacher_forced_logits"] = rel(logits, o["logits"])
        errs["teacher_forced_hiddens"] = rel(hid2, o["hid"])
    _check(f"NL={NL} {kind} {precision} eval", errs, TOL[precision])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", ["none", "global", "local"])
@pytest.mark.parametrize("NL", [2, 3])
def test_train_mode_with_the_same_masks_matches_the_fp64_oracle(NL, kind, precision):
    """Dropout at every site: embedding, logits, the decoder's inter-layer sites 17 (and 18), the local reconstructor's input over
    (S, NLd, B, H) or the global one's pooled state over (L, B, H)."""
    m, inputs, P, Q, o = _case(NL, kind, train=True)
    dec, rec, _, _, dloss, rloss, hiddens = _step(m, kind, precision, inputs, P, Q, train=True)
    _check(f"NL={NL} {kind} {precision} train", _errors(o, dloss, rloss, dec, rec, hiddens), TOL[precision])


@pytest.fixture(scope="module")
def stress_case():
    m = STRESS
    inputs, P, Q = _problem(m, "local", seed=9, full_length_first=True)
    assert int(inputs[2].any(dim=1).sum()) == m["cap_len"] + 1                # 31 decoder steps, as bench.py runs them
    return m, inputs, P, Q, _oracle(m, "local", inputs, P, Q, _masks(m, "local"))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_benchmarked_stacked_train_step_matches_the_fp64_oracle(stress_case, precision):
    """bench.py msrvtt_stress: train.train_step with the default environment (split decoder forward, background lane), the
    optimiser step left out so that the gradients can be read; the same masks in the oracle."""
    m, inputs, P, Q, o = stress_case
    dec, rec = _build(m, precision, "local", P, Q, train=True)
    feats, targets, _ = (x.to(dev()) for x in inputs)
    _, dloss, rloss = T.train_step(dec, rec, feats.float(), targets, n_steps=m["cap_len"] + 1, optimizer_step=False)
    torch.cuda.synchronize()
    Fn.check_loop_status()
    _check(f"msrvtt_stress NL=2 local {precision} train_step", _errors(o, dloss, rloss, dec, rec), TOL[precision])
