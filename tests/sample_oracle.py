"""fp64 CPU oracle of the device sampler (``Decoder.sample`` / recnet_decoder_sample) and of the self-critical replay -- test
infrastructure.

A free-running loop over ``O.decoder_step`` (``stacked_oracle.decoder_step`` with the inter-layer masks in a stack,
``attn_softmax_oracle`` for the paper's attention) that feeds back its own samples.  Conventions (the kernels', csrc/seq_decoder.cuh):
  * train mode: the dropout masks of the sequence forward, element (t*B + row)*D + j of every site, drawn from the decoder's
    (seed, offset) pair -- embedding (site 1, D = EMB), logits (site 2, D = V), input of stacked layer l (site 16 + l, D = H);
  * Gumbel noise g = -log(-log u), u = ((w >> 8) + 0.5) 2^-24, w = Philox word of element (t*B + row)*V + v of site 5 (SITE_SAMPLE),
    keyed by the separate noise (seed, offset) pair;
  * row token = arg-max of logits'/tau + g (lowest index on ties), logp = log_softmax(logits'/tau)[token];
  * a row finishes once it emits <EOS> or <PAD>; afterwards it emits <PAD> with logp 0; lengths = tokens up to the finishing one;
    the loop ends once every row has finished (n = that step + 1) or after max_steps.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from oracle import recnet_oracle as O
from tests import attn_softmax_oracle as S
from tests import stacked_oracle as SO
from tests.golden_util import philox_scales
from tests.philox_ref import SITE_EMB, SITE_LOGITS, philox4x32_10

SITE_SAMPLE = 5
PAD, SOS, EOS = 0, 1, 2


def gumbel(seed: int, offset: int, t: int, B: int, V: int) -> torch.Tensor:
    """(B, V) fp64 Gumbel noise of step t."""
    row = np.arange(B, dtype=np.uint64)[:, None]
    v = np.arange(V, dtype=np.uint64)[None, :]
    idx = ((np.uint64(t * B) + row) * np.uint64(V) + v).ravel()
    words = philox4x32_10(idx >> np.uint64(2), (int(offset) << 8) | SITE_SAMPLE, int(seed))
    w = np.choose((idx & np.uint64(3)).astype(np.int64), words)
    u = ((w >> np.uint64(8)).astype(np.float64) + 0.5) / 16777216.0
    return torch.from_numpy(-np.log(-np.log(u))).view(B, V)


class Drops:
    """Train-mode dropout scales of a decoder for steps 0..L-1 at batch B (None everywhere = eval mode)."""

    def __init__(self, seed, offset, *, L, B, EMB, V, H, n_layers, p_emb, p_out, p_layer):
        self.emb = philox_scales(seed, offset, SITE_EMB, (L, B, EMB), p_emb)
        self.logits = philox_scales(seed, offset, SITE_LOGITS, (L, B, V), p_out)
        self.layer = SO.layer_drop_masks(seed, n_layers, L, B, H, p_layer, offset=offset) if n_layers > 1 else None


def _step(P, tok, hidden, feats, t, *, model_name, n_layers, embedding_scale, drops: Optional[Drops], attn_softmax):
    de = None if drops is None else drops.emb[t]
    dl = None if drops is None else drops.logits[t]
    if attn_softmax:
        assert n_layers == 1
        return S.decoder_step(P, tok, hidden, feats, model_name=model_name, n_layers=1, embedding_scale=embedding_scale,
                              drop_emb=de, drop_logits=dl, attn_softmax=True)
    dly = None if (drops is None or drops.layer is None) else drops.layer[t]
    return SO.decoder_step(P, tok, hidden, feats, model_name=model_name, n_layers=n_layers, embedding_scale=embedding_scale,
                           drop_emb=de, drop_logits=dl, drop_layer=dly)


@torch.no_grad()
def sample(P, feats, *, max_steps, tau=1.0, noise=(0, 0), model_name="LSTM", n_layers=1, embedding_scale=1.0,
           drops: Optional[Drops] = None, attn_softmax=False, eos=EOS, zero_noise=False):
    """feats (N, T, E) fp64, rows already tiled.  Returns dict(ids (max_steps, N), logp (max_steps, N), lengths (N,), n,
    gap (max_steps, N): top-2 gap of the noisy values, +inf where the row had finished)."""
    N = feats.shape[0]
    H = P["rnn.weight_hh_l0"].shape[1]
    V = P["out.weight"].shape[0]
    tok = torch.full((1, N), SOS, dtype=torch.long)
    hidden = O.zero_hidden(model_name, n_layers, N, H, feats)
    ids = torch.zeros(max_steps, N, dtype=torch.long)
    logp = torch.zeros(max_steps, N, dtype=torch.float64)
    gap = torch.full((max_steps, N), float("inf"), dtype=torch.float64)
    lengths = torch.full((N,), max_steps, dtype=torch.int32)
    done = torch.zeros(N, dtype=torch.bool)
    n = max_steps
    for t in range(max_steps):
        logits, hidden = _step(P, tok, hidden, feats, t, model_name=model_name, n_layers=n_layers, embedding_scale=embedding_scale,
                               drops=drops, attn_softmax=attn_softmax)
        x = logits / tau
        y = x if zero_noise else x + gumbel(noise[0], noise[1], t, N, V)
        v = y.argmax(dim=1)                                              # first maximal index on ties
        top2 = y.topk(2, dim=1).values
        lp = torch.log_softmax(x, dim=1).gather(1, v.view(-1, 1)).squeeze(1)
        live = ~done
        ids[t] = torch.where(live, v, torch.zeros_like(v))
        logp[t] = torch.where(live, lp, torch.zeros_like(lp))
        gap[t] = torch.where(live, top2[:, 0] - top2[:, 1], gap[t])
        fin = live & ((v == eos) | (v == PAD))
        lengths[fin] = t + 1
        tok = torch.where(done, torch.zeros_like(v), v).view(1, -1)      # <PAD> after the finishing token has been fed back
        done = done | fin
        if bool(done.all()):
            n = t + 1
            break
    return {"ids": ids, "logp": logp, "lengths": lengths, "n": n, "gap": gap}


def replay_loss(P, feats, tokens_in, targets, ce_weight, *, model_name="LSTM", n_layers=1, embedding_scale=1.0,
                drops: Optional[Drops] = None, attn_softmax=False, lambda_reg=1e-3):
    """Teacher-forced loss of the self-critical replay: sum_{t,row} ce_weight * (-log_softmax(logits')[targets]) + lambda * sum ||p||."""
    N = feats.shape[0]
    H = P["rnn.weight_hh_l0"].shape[1]
    hidden = O.zero_hidden(model_name, n_layers, N, H, feats)
    loss = feats.new_zeros(())
    for t in range(tokens_in.shape[0]):
        logits, hidden = _step(P, tokens_in[t:t + 1], hidden, feats, t, model_name=model_name, n_layers=n_layers,
                               embedding_scale=embedding_scale, drops=drops, attn_softmax=attn_softmax)
        lp = torch.log_softmax(logits, dim=1).gather(1, targets[t].view(-1, 1)).squeeze(1)
        loss = loss - (ce_weight[t] * lp).sum()
    return loss + lambda_reg * O.param_norm_sum(P)
