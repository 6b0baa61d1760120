"""GPU parity of greedy and beam decoding of stacked LSTM decoders (n_layers 2-4) on the device loops (recnet_decoder_greedy /
recnet_decoder_beam: one C call, the stacked step's upper layers ping-ponged between two state blocks):
  * fp32 greedy ids and stop step bit-exact against the fp64 oracle, at the mid shape of test_gpu_stacked.py and at BASELINE config 4;
  * bf16 greedy against the per-step Decoder.forward and the oracle, each fed the device's own tokens;
  * fp32 beam search (widths 1-8) against the oracle's restatement and against the per-step loop (RECNET_BEAM_DEVICE=0);
  * the public entry points take the device loop (Decoder.forward is never called); stacked GRU decoders still step;
  * the paper's softmax attention over a 2-layer stack;
  * train.forward_decoder with teacher_forcing_ratio 0, whose fed-back tokens continue after an all-<PAD> step as the reference's do.
Each case prints its worst error or smallest top-2 logit margin."""
import pytest
import torch

import recnet_b200
from recnet_b200 import eval as E
from recnet_b200 import models as M
from recnet_b200 import train as T
from oracle import recnet_oracle as O
from tests import attn_softmax_oracle as S
from tests.golden_util import load_golden
from tests.test_gpu_attn_softmax import build_sm
from tests.test_gpu_parity import FULL, TOL, _Vocab, _full_inputs, build, dev, rel
from tests.test_gpu_stacked import MID

pytestmark = pytest.mark.gpu

D = torch.float64
STEPS = MID["cap_len"] + 1


def _m(NL, **kw):
    return dict(MID, dec_layers=NL, **kw)


def _inputs(seed=7):
    return O.synthetic_batch(MID["B"], MID["T"], MID["E"], MID["V"], MID["cap_len"], seed=seed, full_length_first=True, dtype=D)


def _params(NL, logit_scale=1.0, pad_boost=0.0, eos_boost=0.0):
    """fp64 decoder weights; logit_scale spreads the (near-flat) default-init logits, the boosts lift <PAD> / <EOS>."""
    P = O.init_decoder_params(MID["V"], MID["EMB"], MID["E"], MID["H"], MID["A"], n_layers=NL, seed=4, dtype=D)
    P["out.weight"] = P["out.weight"] * logit_scale
    P["out.bias"] = P["out.bias"].clone()
    P["out.bias"][0] += pad_boost
    P["out.bias"][2] += eos_boost
    return P


def _forced_logits(P, feats, ids, NL, softmax=False):
    """fp64 oracle logits of every step with the tokens `ids` (steps, B) fed back (step t sees ids[t-1])."""
    n, B = ids.shape
    masks = torch.ones(n + 1, B, dtype=torch.bool)
    targets = torch.cat((ids.cpu(), torch.zeros(1, B, dtype=torch.long)))
    _, _, _, aux = S.forward_decoder(P, feats, targets, masks, n_layers=NL, caption_max_len=n - 1, attn_softmax=softmax)
    return aux["logits"]


def _margin(logits):
    top2 = logits.topk(2, dim=-1).values
    return float((top2[..., 0] - top2[..., 1]).min())


def _tok_hid(B, NL, H):
    z = torch.zeros(NL, B, H, device=dev())
    return torch.full((1, B), 1, dtype=torch.long, device=dev()), (z, z.clone())


def _first_mismatch(got, ref):
    diff = (got != ref).nonzero()
    return None if diff.numel() == 0 else tuple(int(x) for x in diff[0])


# ---- 1. fp32 greedy, bit-exact ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("NL", [2, 3, 4])
def test_fp32_greedy_is_bit_exact_against_the_fp64_oracle(NL):
    feats, _, _ = _inputs()
    P = _params(NL)
    ref = O.greedy_search(P, feats, n_layers=NL, caption_max_len=MID["cap_len"])
    dec, _ = build(_m(NL), "fp32", "none", P, {})
    assert dec["model"].uses_fused_sequence
    ids, n = dec["model"].greedy(feats.float().to(dev()), STEPS)
    got = ids[: int(n)].cpu()
    margin = _margin(_forced_logits(P, feats, ref, NL))
    print(f"[stacked decode] fp32 greedy NL={NL}: steps {int(n)} / oracle {ref.shape[0]}, smallest oracle top-2 logit margin "
          f"{margin:.3e}, first mismatch {_first_mismatch(got, ref) if got.shape == ref.shape else 'shape'}")
    assert int(n) == ref.shape[0]
    assert torch.equal(got, ref)


def test_fp32_greedy_bit_exact_at_the_batch1024_shape_two_layers():
    """BASELINE config 4 (batch 1024, 28 frames, max len 30) with a 2-layer decoder, by the criterion of
    test_full_size_greedy_bit_exact_fp32_batch1024_shape: every id and the stop step."""
    B = 1024
    feats, _, _ = _full_inputs(B, seed=77)
    P = O.init_decoder_params(FULL["V"], FULL["EMB"], FULL["E"], FULL["H"], FULL["A"], n_layers=2, seed=0)
    P["out.bias"][0] += 3.0                     # random weights never emit <PAD>; nudge it so the PAD-stop rule is exercised
    ref = O.greedy_search(P, feats, n_layers=2)
    dec, _ = build(dict(FULL, B=B, dec_layers=2), "fp32", "none", P, {})
    ids, n = dec["model"].greedy(feats.to(dev()), 31)
    got = ids[: int(n)].cpu()
    print(f"[stacked decode] fp32 greedy B=1024 NL=2: steps {int(n)} / oracle {ref.shape[0]}, first mismatch "
          f"{_first_mismatch(got, ref) if got.shape == ref.shape else 'shape'}")
    assert int(n) == ref.shape[0]
    assert torch.equal(got, ref)


# ---- 2. bf16 greedy -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("NL", [2, 3, 4])
def test_bf16_greedy_agrees_with_the_per_step_api_and_the_oracle(NL):
    """The bf16 device loop against the per-step Decoder.forward (operator kernels) and the fp64 oracle, both fed the device's own tokens
    so that one near-tie does not change the rest of a caption; the allowance of
    test_bf16_greedy_on_projected_feature_kernels_agrees_with_the_per_step_api (first step equal, >= 90 % of the ids)."""
    feats, _, _ = _inputs()
    P = _params(NL, logit_scale=12.0)
    dec, _ = build(_m(NL), "bf16", "none", P, {})
    model = dec["model"]
    f = feats.float().to(dev())
    ids, n = model.greedy(f, STEPS)
    ids = ids[: int(n)]
    B = f.shape[0]
    tok, hid = _tok_hid(B, NL, MID["H"])
    pred = []
    with torch.no_grad(), model.cached_uv(f):
        for t in range(int(n)):
            logits, hid = model(tok, hid, f)
            pred.append(logits.argmax(dim=1))
            tok = ids[t].view(1, -1)
    pred = torch.stack(pred)
    oracle = _forced_logits(P, feats, ids, NL).argmax(dim=-1)
    agree_api = float((pred == ids).float().mean())
    agree_oracle = float((oracle == ids.cpu()).float().mean())
    print(f"[stacked decode] bf16 greedy NL={NL}: {int(n)} steps, agreement with the per-step API {agree_api:.3f}, with the oracle "
          f"{agree_oracle:.3f}")
    assert torch.equal(ids[0], pred[0]), (ids[0], pred[0])
    assert agree_api >= 0.9 and agree_oracle >= 0.9, (agree_api, agree_oracle)


# ---- 3. beam search ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("NL", [2, 3, 4])
def test_fp32_beam_matches_the_oracle_and_the_per_step_loop(NL, monkeypatch):
    """Logits spread (out.weight x 12) and <EOS> lifted (+1.5) as in the beam fixtures, so that the length rule is exercised."""
    feats, _, _ = _inputs()
    P = _params(NL, logit_scale=12.0, eos_boost=1.5)
    dec, _ = build(_m(NL), "fp32", "none", P, {})
    model = dec["model"]
    f = feats.float().to(dev())
    B = f.shape[0]
    T.C.batch_size = B
    vocab = _Vocab(MID["V"])
    for width in (1, 3, 5, 8):
        ref = O.beam_search(P, feats, width, n_layers=NL, caption_max_len=MID["cap_len"])
        assert sum(2 in s[:-1] for s in ref) > 0                   # some caption has <EOS> before its end
        tok, hid = _tok_hid(B, NL, MID["H"])
        assert E._device_beam_applies(model, width, tok, hid, vocab)
        got = E.beam_search(T.C, width, vocab, model, tok, hid, f)
        with monkeypatch.context() as mp:
            mp.setenv("RECNET_BEAM_DEVICE", "0")
            loop = E.beam_search(T.C, width, vocab, model, tok, hid, f)
        bad = [b for b in range(B) if got[b] != ref[b]]
        print(f"[stacked decode] fp32 beam NL={NL} width {width}: {len(ref[0])} steps, samples differing from the oracle {bad}, "
              f"from the per-step loop {[b for b in range(B) if got[b] != loop[b]]}")
        assert got == ref, (width, bad)
        assert got == loop, width


# ---- 4. the public entry points take the device loop ----------------------------------------------------------------------------
def test_public_entry_points_decode_a_two_layer_lstm_without_decoder_forward(monkeypatch):
    g = load_golden("tiny_lstm_2layer")
    m = g["meta"]
    dec, _ = build(m, "fp32", "none", g["dec"], {})
    model = dec["model"]
    feats = g["feats"].float().to(dev())
    B = feats.shape[0]
    T.C.batch_size = B

    def no_forward(*a, **kw):
        raise AssertionError("Decoder.forward called")

    monkeypatch.setattr(M.Decoder, "forward", no_forward)
    tok, hid = _tok_hid(B, 2, m["H"])
    ids = E.greedy_search(T.C, model, tok, hid, feats)
    assert torch.equal(torch.tensor(ids), g["greedy_ids"])
    for width in (3, 5):          # sequences themselves: test_fp32_beam_matches_the_oracle_and_the_per_step_loop
        got = E.beam_search(T.C, width, _Vocab(m["V"]), model, tok, hid, feats)
        assert len(got) == B and len({len(s) for s in got}) == 1 and 1 <= len(got[0]) <= m["cap_len"] + 1, got


def test_two_layer_gru_decoder_still_steps_through_forward(monkeypatch):
    g = load_golden("tiny_gru_2layer")
    m = g["meta"]
    dec, _ = build(m, "fp32", "none", g["dec"], {})
    model = dec["model"]
    assert not model.uses_fused_sequence
    feats = g["feats"].float().to(dev())
    B = feats.shape[0]
    T.C.batch_size = B
    calls = []
    forward = M.Decoder.forward

    def counted(self, *a, **kw):
        calls.append(1)
        return forward(self, *a, **kw)

    monkeypatch.setattr(M.Decoder, "forward", counted)
    tok = torch.full((1, B), 1, dtype=torch.long, device=dev())
    hid = torch.zeros(2, B, m["H"], device=dev())
    ids = E.greedy_search(T.C, model, tok, hid, feats)
    assert torch.equal(torch.tensor(ids), g["greedy_ids"]) and len(calls) == len(ids)
    assert not E._device_beam_applies(model, 3, tok, hid, _Vocab(m["V"]))
    del calls[:]
    got = E.beam_search(T.C, 3, _Vocab(m["V"]), model, tok, hid, feats)
    assert len(got) == B and len(calls) == 3 * (len(got[0]) - 1) + 1          # one beam at step 0, three after


# ---- 5. softmax attention -----------------------------------------------------------------------------------------------------
def test_softmax_attention_two_layer_greedy_and_beam_against_the_oracle():
    NL = 2
    feats, _, _ = _inputs()
    f = feats.float().to(dev())
    B = f.shape[0]
    P = _params(NL)
    dec, _ = build_sm(_m(NL), "fp32", P, None)
    ref = S.greedy_search(P, feats, n_layers=NL, caption_max_len=MID["cap_len"], attn_softmax=True)
    ids, n = dec["model"].greedy(f, STEPS)
    got = ids[: int(n)].cpu()
    margin = _margin(_forced_logits(P, feats, ref, NL, softmax=True))
    print(f"[stacked decode] softmax greedy NL=2: steps {int(n)} / oracle {ref.shape[0]}, smallest oracle top-2 logit margin "
          f"{margin:.3e}, first mismatch {_first_mismatch(got, ref) if got.shape == ref.shape else 'shape'}")
    assert int(n) == ref.shape[0] and torch.equal(got, ref)
    Pb = _params(NL, logit_scale=12.0, eos_boost=1.5)
    dec, _ = build_sm(_m(NL), "fp32", Pb, None)
    T.C.batch_size = B
    for width in (3, 5):
        ref = S.beam_search(Pb, feats, width, n_layers=NL, caption_max_len=MID["cap_len"], attn_softmax=True)
        tok, hid = _tok_hid(B, NL, MID["H"])
        got = E.beam_search(T.C, width, _Vocab(MID["V"]), dec["model"], tok, hid, f)
        print(f"[stacked decode] softmax beam NL=2 width {width}: samples differing from the oracle "
              f"{[b for b in range(B) if got[b] != ref[b]]}")
        assert got == ref, width


# ---- 6. train.forward_decoder with argmax feedback ------------------------------------------------------------------------------
# <PAD> lifts (chosen on the fp64 oracle) under which every sample emits <PAD> at step 0 and some sample emits another token later
PAD_BOOST = {2: 0.1, 3: 0.15, 4: 0.05}


@pytest.mark.parametrize("NL", [2, 3, 4])
def test_forward_decoder_without_teacher_forcing_continues_after_an_all_pad_step(NL):
    feats, targets, masks = _inputs()
    P = _params(NL, pad_boost=PAD_BOOST[NL])
    Pr = {k: v.clone() for k, v in P.items()}
    dl, hid, idx, aux = O.forward_decoder(Pr, feats, targets, masks, n_layers=NL, caption_max_len=MID["cap_len"], teacher_forcing=False)
    ref_ids = torch.stack(idx)
    nonpad = (ref_ids != 0).sum(dim=1)
    assert ref_ids.shape[0] == STEPS and int(nonpad[0]) == 0 and int(nonpad[1:].sum()) > 0, nonpad.tolist()
    dec, _ = build(_m(NL), "fp32", "none", P, {})
    loss, hiddens, out_idx = T.forward_decoder(dec, feats.float().to(dev()), targets.to(dev()), masks.to(dev()), 0.0)
    errs = {"loss": rel(loss, dl), "hiddens": rel(hiddens, hid)}
    worst = max(errs, key=errs.get)
    print(f"[stacked decode] forward_decoder ratio 0 NL={NL}: non-<PAD> ids per step {nonpad.tolist()}, smallest oracle top-2 logit "
          f"margin {_margin(aux['logits']):.3e}, first id mismatch {_first_mismatch(out_idx, ref_ids)}, worst rel err "
          f"{errs[worst]:.3e} ({worst})")
    assert torch.equal(out_idx, ref_ids)
    assert errs[worst] < TOL["fp32"], (worst, errs[worst])
