"""CPU oracle of a stacked LSTM decoder in TRAIN mode: the inter-layer dropout of nn.LSTM(num_layers=NL, dropout=p) -- test
infrastructure.

``oracle/recnet_oracle.py`` runs stacked decoders in eval mode only (``_rnn_layers``: inter-layer dropout off).  This module
restates ``O.decoder_step`` with the inter-layer masks and runs ``O.forward_decoder`` over it, the way
``tests/attn_softmax_oracle.py`` swaps in its attention; the oracle itself is unchanged.  With ``drop_layer=None`` the functions
here ARE the oracle's.  Callers pass float64 tensors to get an fp64 reference.

Mask convention (the kernels', csrc/seq_decoder.cuh):
    input of layer l at step t  =  h^{l-1}_t * m_l[t],   1 <= l <= NL-1,
    m_l = the Philox scales of site SITE_LAYER0 + l over (L, B, H) (element (t, b, j) = index t*B*H + b*H + j), drawn from the
    decoder's (seed, offset): offset 1 on the first training forward after ``seed_dropout``.
The mask multiplies only the copy fed to layer l: the returned hiddens, the layer's own recurrent state and the attention query
(the top layer's h) are unmasked.

The reconstructors need no restatement: ``O.forward_local_reconstructor`` takes drop_x (S, NLd, B, H) over a stacked decoder
(site 3, pseudo-step q = t*NLd + l) and ``O.forward_global_reconstructor`` drop_mp (L, B, H) (site 4).
"""
from __future__ import annotations

import contextlib
from typing import Dict, Optional

import torch

from oracle import recnet_oracle as O
from tests.golden_util import philox_scales
from tests.philox_ref import SITE_EMB, SITE_GLOBAL_MP, SITE_LAYER0, SITE_LOCAL_X, SITE_LOGITS


def decoder_step(P, tok, hidden, feats, *, model_name="LSTM", n_layers=1, embedding_scale=1.0,
                 drop_emb: Optional[torch.Tensor] = None, drop_logits: Optional[torch.Tensor] = None,
                 drop_layer: Optional[torch.Tensor] = None):
    """O.decoder_step (decoder.py:45-70) with this step's inter-layer scales drop_layer (NL-1, B, H); None = eval mode."""
    if drop_layer is None:
        return O.decoder_step(P, tok, hidden, feats, model_name=model_name, n_layers=n_layers, embedding_scale=embedding_scale,
                              drop_emb=drop_emb, drop_logits=drop_logits)
    if model_name != "LSTM":
        raise NotImplementedError("inter-layer dropout is restated for LSTM decoders only (stacked GRU decoders have no fused driver)")
    assert drop_layer.shape[0] == n_layers - 1, (tuple(drop_layer.shape), n_layers)
    emb = P["embedding.weight"][tok[0]] * embedding_scale
    if drop_emb is not None:
        emb = emb * drop_emb
    top_h = hidden[0][-1]
    Uv = feats @ P["attn_U.weight"].t()
    Wh = (top_h @ P["attn_W.weight"].t()).unsqueeze(1)
    e = torch.tanh(Wh + Uv + P["attn_b"]) @ P["attn_w.weight"].t()
    ctx = (e * feats).mean(dim=1)
    x = torch.cat((emb, ctx), dim=1)
    hs, cs = [], []
    for l in range(n_layers):
        h, c = O.lstm_cell(x, hidden[0][l], hidden[1][l], P[f"rnn.weight_ih_l{l}"], P[f"rnn.weight_hh_l{l}"],
                           P[f"rnn.bias_ih_l{l}"], P[f"rnn.bias_hh_l{l}"])
        hs.append(h)
        cs.append(c)
        x = h * drop_layer[l] if l + 1 < n_layers else h          # nn.LSTM: dropout on every layer's output except the last
    logits = x @ P["out.weight"].t() + P["out.bias"]
    if drop_logits is not None:
        logits = logits * drop_logits
    return logits, (torch.stack(hs), torch.stack(cs))


@contextlib.contextmanager
def _layer_drop_steps(drop_layer: Optional[torch.Tensor]):
    """O.forward_decoder looks O.decoder_step up at call time, once per step in order: feed it row t of drop_layer."""
    if drop_layer is None:
        yield
        return
    rows = iter(drop_layer.unbind(0))
    saved = O.decoder_step
    O.decoder_step = lambda *a, **kw: decoder_step(*a, drop_layer=next(rows), **kw)
    try:
        yield
    finally:
        O.decoder_step = saved


def forward_decoder(*args, drop_layer: Optional[torch.Tensor] = None, **kw):
    """O.forward_decoder; drop_layer (>= L, NL-1, B, H) holds the inter-layer scales of every step (None = eval mode)."""
    with _layer_drop_steps(drop_layer):
        return O.forward_decoder(*args, **kw)


def layer_drop_masks(seed: int, n_layers: int, L: int, B: int, H: int, p: float, offset: int = 1, site0: int = SITE_LAYER0,
                     dtype=torch.float64) -> torch.Tensor:
    """(L, NL-1, B, H): column l-1 holds the scales of site site0 + l, the input of layer l."""
    return torch.stack([philox_scales(seed, offset, site0 + l, (L, B, H), p, dtype) for l in range(1, n_layers)], 1)


def train_mode_masks(C, seeds: Dict[str, int], kind: str, *, L: int, B: int, EMB: int, V: int, H: int, S: int, n_layers: int,
                     dtype=torch.float64) -> Dict[str, torch.Tensor]:
    """Every dropout scale tensor of one training step, as the kernels draw them on the first training forward after
    ``seed_dropout(seeds[...])`` (offset 1).  L is the longest caption + 1; steps beyond the actual loop length are unused.
    Keys: emb (L,B,EMB), logits (L,B,V), layer (L,NL-1,B,H); x (S,NL,B,H) for kind = local, mp (L,B,H) for kind = global."""
    out = {"emb": philox_scales(seeds["dec"], 1, SITE_EMB, (L, B, EMB), C.embedding_dropout, dtype),
           "logits": philox_scales(seeds["dec"], 1, SITE_LOGITS, (L, B, V), C.decoder_out_dropout, dtype),
           "layer": layer_drop_masks(seeds["dec"], n_layers, L, B, H, C.decoder_dropout, dtype=dtype)}
    if kind == "local":
        out["x"] = philox_scales(seeds["local"], 1, SITE_LOCAL_X, (S, n_layers, B, H), C.reconstructor_decoder_dropout, dtype)
    elif kind == "global":
        out["mp"] = philox_scales(seeds["global"], 1, SITE_GLOBAL_MP, (L, B, H), C.reconstructor_decoder_dropout, dtype)
    return out
