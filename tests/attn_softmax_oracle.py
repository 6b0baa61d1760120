"""fp64 CPU oracle of the RecNet paper's softmax attention (opt-in ``attn_softmax``) -- test infrastructure.

The reference never calls its ``attn_softmax`` module (SURVEY.md 0.1), so no reference-generated golden exists for this
variant; this restatement is the authority.  It reuses ``oracle/recnet_oracle.py`` unchanged: only the two attention steps are
restated, and the sequence loops / searches of the oracle run over them.  With ``attn_softmax=False`` every function here IS the
oracle's.

    decoder, step t, sample b:        alpha_t[b,tau] = softmax_tau(e_t[b,tau]),  ctx_t[b] = sum_tau alpha_t[b,tau] v[b,tau]
    local reconstructor, step s:      beta_s[l] = softmax_l(score) per decoder layer,  x_s = sum_l beta_s[l] h_l   (all L steps)
"""
from __future__ import annotations

import contextlib
from typing import Optional

import torch

from oracle import recnet_oracle as O


def decoder_step_softmax(P, tok, hidden, feats, *, model_name="LSTM", n_layers=1, embedding_scale=1.0,
                         drop_emb: Optional[torch.Tensor] = None, drop_logits: Optional[torch.Tensor] = None):
    """O.decoder_step with the paper's attention (decoder.py:55-62 with the softmax the reference builds but never calls)."""
    emb = P["embedding.weight"][tok[0]] * embedding_scale
    if drop_emb is not None:
        emb = emb * drop_emb
    top_h = hidden[0][-1] if model_name == "LSTM" else hidden[-1]
    Uv = feats @ P["attn_U.weight"].t()                                  # (B,T,A)
    Wh = (top_h @ P["attn_W.weight"].t()).unsqueeze(1)
    e = torch.tanh(Wh + Uv + P["attn_b"]) @ P["attn_w.weight"].t()       # (B,T,1)
    alpha = torch.softmax(e, dim=1)                                      # over the T frames
    ctx = (alpha * feats).sum(dim=1)                                     # weighted sum, no 1/T
    x = torch.cat((emb, ctx), dim=1)
    outs, hidden = O._rnn_layers(P, "rnn", model_name, n_layers, [x], hidden)
    logits = outs[0] @ P["out.weight"].t() + P["out.bias"]
    if drop_logits is not None:
        logits = logits * drop_logits
    return logits, hidden


def local_reconstructor_step_softmax(P, hidden, decoder_hiddens, *, model_name="LSTM", n_layers=1,
                                     drop_x: Optional[torch.Tensor] = None):
    """O.local_reconstructor_step with the paper's attention: one softmax over the L steps per decoder layer."""
    top_h = hidden[0][-1] if model_name == "LSTM" else hidden[-1]
    Uv = decoder_hiddens @ P["attn_U.weight"].t()                        # (L,NLdec,B,A)
    Wh = top_h @ P["attn_W.weight"].t()
    score = torch.tanh(Wh + Uv + P["attn_b"]) @ P["attn_w.weight"].t()   # (L,NLdec,B,1)
    beta = torch.softmax(score, dim=0)                                   # over the L decoder steps, per layer and sample
    x = (beta * decoder_hiddens).sum(dim=0)                              # (NLdec,B,H)
    if drop_x is not None:
        x = x * drop_x                                                   # dropout after the weighted sum, as in the reference
    outs, hidden = O._rnn_layers(P, "rnn", model_name, n_layers, list(x.unbind(0)), hidden)
    out = outs[0] @ P["out.weight"].t() + P["out.bias"]
    return out, hidden


@contextlib.contextmanager
def _softmax_steps(on: bool):
    """The oracle's loops look their step functions up at call time: run them over the softmax steps."""
    if not on:
        yield
        return
    saved = O.decoder_step, O.local_reconstructor_step
    O.decoder_step, O.local_reconstructor_step = decoder_step_softmax, local_reconstructor_step_softmax
    try:
        yield
    finally:
        O.decoder_step, O.local_reconstructor_step = saved


def decoder_step(*args, attn_softmax=False, **kw):
    return (decoder_step_softmax if attn_softmax else O.decoder_step)(*args, **kw)


def local_reconstructor_step(*args, attn_softmax=False, **kw):
    return (local_reconstructor_step_softmax if attn_softmax else O.local_reconstructor_step)(*args, **kw)


def forward_decoder(*args, attn_softmax=False, **kw):
    with _softmax_steps(attn_softmax):
        return O.forward_decoder(*args, **kw)


def forward_local_reconstructor(*args, attn_softmax=False, **kw):
    with _softmax_steps(attn_softmax):
        return O.forward_local_reconstructor(*args, **kw)


def greedy_search(*args, attn_softmax=False, **kw):
    with _softmax_steps(attn_softmax):
        return O.greedy_search(*args, **kw)


def beam_search(*args, attn_softmax=False, **kw):
    with _softmax_steps(attn_softmax):
        return O.beam_search(*args, **kw)
