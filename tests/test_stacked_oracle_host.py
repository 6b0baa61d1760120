"""The train-mode stacked-decoder oracle (tests/stacked_oracle.py) checked without a GPU:
  * all-ones masks give O.forward_decoder bit for bit (loss, hiddens, every gradient), NL = 2, 3, 4;
  * Philox masks give what an independent formulation gives: one single-layer fp64 nn.LSTM per layer, masks multiplied in between;
  * the masks matter: at the shape of the train-mode GPU cases the masked result is farther from eval mode and from every
    near miss of the mask convention (site, offset, step) than 10x the bf16 tolerance of those tests -- so a kernel that slips
    one of them cannot pass tests/test_gpu_stacked.py.
"""
import pytest
import torch

from oracle import recnet_oracle as O
from tests import stacked_oracle as SO
from tests.philox_ref import SITE_LAYER0

D = torch.float64
SMALL = dict(B=5, T=7, E=24, H=16, A=8, EMB=12, V=40, cap=6)
# the shape and inputs of the train-mode GPU cases (tests/test_gpu_stacked.py); seed 5 (SMALL) and 7 (MID) give a loop that stops
# before caption_max_len + 1 steps
MID = dict(B=13, T=19, E=512, H=256, A=128, EMB=96, V=700, cap=12)
P_LAYER, SEED = 0.5, 0xDEC0
BF16_TOL = 2e-2


def _setup(m, NL, seed):
    feats, targets, masks = O.synthetic_batch(m["B"], m["T"], m["E"], m["V"], m["cap"], seed=seed, dtype=D, full_length_first=False)
    P = O.init_decoder_params(m["V"], m["EMB"], m["E"], m["H"], m["A"], n_layers=NL, seed=4, dtype=D)
    return feats, targets, masks, P


def _run(P, feats, targets, masks, NL, cap, fn=SO.forward_decoder, **kw):
    """(loss, hiddens, logits, grads) of fn on fresh leaves."""
    Pr = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    loss, hid, _, aux = fn(Pr, feats, targets, masks, n_layers=NL, caption_max_len=cap, **kw)
    loss.backward()
    return loss.detach(), hid.detach(), aux["logits"].detach(), {k: v.grad for k, v in Pr.items()}


def _rel(a, b):
    return float((a - b).abs().max() / (b.abs().max() + 1e-300))


@pytest.mark.parametrize("NL", [2, 3, 4])
def test_all_ones_masks_reproduce_the_eval_oracle_bit_for_bit(NL):
    m = SMALL
    feats, targets, masks, P = _setup(m, NL, seed=5)
    ones = torch.ones(m["cap"] + 1, NL - 1, m["B"], m["H"], dtype=D)
    oracle_step = O.decoder_step
    ref = _run(P, feats, targets, masks, NL, m["cap"], fn=O.forward_decoder)
    got = _run(P, feats, targets, masks, NL, m["cap"], drop_layer=ones)
    assert O.decoder_step is oracle_step                                    # the swap is undone
    assert ref[1].shape[1] == NL and ref[1].shape[0] < m["cap"] + 1          # ragged: the loop stops early
    for a, b in zip(got[:3], ref[:3]):
        assert torch.equal(a, b)
    assert got[3].keys() == ref[3].keys()
    for k in ref[3]:
        assert torch.equal(got[3][k], ref[3][k]), k


def _independent(P, feats, targets, masks, NL, drop_layer, lambda_reg=1e-3):
    """Stacked decoder built from one single-layer nn.LSTM per layer (fp64), the inter-layer masks multiplied between them;
    attention (decoder.py:50-61), vocabulary projection and the reference's loss (train.py:41-70) written out here."""
    B, H = feats.shape[0], P["rnn.weight_hh_l0"].shape[1]
    leaf = {k: v.clone().requires_grad_(True) for k, v in P.items() if not k.startswith("rnn.")}
    lstms = []
    for l in range(NL):
        cell = torch.nn.LSTM(P[f"rnn.weight_ih_l{l}"].shape[1], H).to(D)
        with torch.no_grad():
            for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
                getattr(cell, n + "_l0").copy_(P[f"rnn.{n}_l{l}"])
        lstms.append(cell)
    L = int(masks.any(dim=1).sum())                      # captions are prefix-shaped: the loop runs while a row is non-empty
    h = [torch.zeros(1, B, H, dtype=D) for _ in range(NL)]
    c = [torch.zeros(1, B, H, dtype=D) for _ in range(NL)]
    tok = torch.full((B,), O.SOS, dtype=torch.long)
    ce, n_tok, hiddens = 0.0, 0, []
    for t in range(L):
        emb = leaf["embedding.weight"][tok]
        score = torch.tanh((h[-1][0] @ leaf["attn_W.weight"].t()).unsqueeze(1) + feats @ leaf["attn_U.weight"].t() + leaf["attn_b"])
        ctx = (score @ leaf["attn_w.weight"].t() * feats).mean(dim=1)
        x = torch.cat((emb, ctx), dim=1).unsqueeze(0)
        for l in range(NL):
            out, (h[l], c[l]) = lstms[l](x, (h[l], c[l]))
            x = out * drop_layer[t, l] if l + 1 < NL else out
        logits = x[0] @ leaf["out.weight"].t() + leaf["out.bias"]
        sel = masks[t]
        ce = ce + torch.nn.functional.cross_entropy(logits[sel], targets[t][sel])
        n_tok += int(sel.sum())
        hiddens.append(torch.cat(h, 0))
        tok = targets[t]
    params = dict(leaf)
    for l in range(NL):
        for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
            params[f"rnn.{n}_l{l}"] = getattr(lstms[l], n + "_l0")
    loss = ce / n_tok + lambda_reg * sum(torch.linalg.vector_norm(p) for p in params.values())
    loss.backward()
    return loss.detach(), torch.stack(hiddens).detach(), {k: p.grad for k, p in params.items()}


@pytest.mark.parametrize("NL", [2, 3, 4])
def test_philox_masks_match_a_chain_of_single_layer_nn_lstms(NL):
    m = SMALL
    feats, targets, masks, P = _setup(m, NL, seed=5)
    drop = SO.layer_drop_masks(SEED, NL, m["cap"] + 1, m["B"], m["H"], P_LAYER)
    assert set(drop.unique().tolist()) == {0.0, 1.0 / (1.0 - P_LAYER)}
    loss, hid, _, grads = _run(P, feats, targets, masks, NL, m["cap"], drop_layer=drop)
    ref_loss, ref_hid, ref_grads = _independent(P, feats, targets, masks, NL, drop)
    assert hid.shape == ref_hid.shape
    errs = {"loss": _rel(loss, ref_loss), "hiddens": _rel(hid, ref_hid)}
    errs.update({k: _rel(grads[k], ref_grads[k]) for k in ref_grads})
    assert grads.keys() == ref_grads.keys()
    worst = max(errs, key=errs.get)
    assert errs[worst] < 1e-12, (worst, errs[worst])


def _worst(a, b):
    """The largest relative error over what the GPU tests compare: loss, hiddens, every gradient."""
    errs = {"loss": _rel(a[0], b[0]), "hiddens": _rel(a[1], b[1])}
    errs.update({k: _rel(a[3][k], b[3][k]) for k in b[3]})
    worst = max(errs, key=errs.get)
    return errs[worst], worst


@pytest.mark.parametrize("NL", [2, 3])
def test_the_masks_matter_far_beyond_the_bf16_tolerance(NL):
    m = MID
    feats, targets, masks, P = _setup(m, NL, seed=7)
    Lmax, B, H = m["cap"] + 1, m["B"], m["H"]
    drop = SO.layer_drop_masks(SEED, NL, Lmax, B, H, P_LAYER)
    masked = _run(P, feats, targets, masks, NL, m["cap"], drop_layer=drop)
    near_misses = {
        "eval mode": None,
        "site + 1": SO.layer_drop_masks(SEED, NL, Lmax, B, H, P_LAYER, site0=SITE_LAYER0 + 1),
        "site - 1": SO.layer_drop_masks(SEED, NL, Lmax, B, H, P_LAYER, site0=SITE_LAYER0 - 1),
        "offset + 1": SO.layer_drop_masks(SEED, NL, Lmax, B, H, P_LAYER, offset=2),
        "drop_base of step t + 1": SO.layer_drop_masks(SEED, NL, Lmax + 1, B, H, P_LAYER)[1:],
    }
    for name, other in near_misses.items():
        err, where = _worst(_run(P, feats, targets, masks, NL, m["cap"], drop_layer=other), masked)
        print(f"[stacked oracle] NL={NL} {name}: worst rel difference {err:.3f} ({where})")
        assert err > 10 * BF16_TOL, (name, where, err)
