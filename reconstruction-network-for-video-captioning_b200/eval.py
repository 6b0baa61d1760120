"""Inference mirrors of the reference's eval.greedy_search (eval.py:19-33) and eval.beam_search (eval.py:36-120)."""
from __future__ import annotations

import torch


def greedy_search(config, decoder, input, hidden, encoder_outputs):
    """Same signature and return value as eval.greedy_search: a list (one entry per generated step) of lists of
    B token ids.  ``input`` must be the <SOS> row and ``hidden`` the zero state (what eval.evaluate passes,
    eval.py:130-140); the argmax feedback loop runs entirely on the device (one host read at the end instead of
    B per step, eval.py:25)."""
    if not bool((input == 1).all()):
        raise NotImplementedError("greedy_search: the device loop starts from <SOS>; use Decoder.forward for custom starts")
    ids, n = decoder.greedy(encoder_outputs, config.caption_max_len + 1)
    n = int(n.item())
    return ids[:n].tolist()


@torch.no_grad()
def beam_search(config, beam_width, vocab, decoder, input, hidden, encoder_outputs):
    """eval.beam_search (eval.py:36-120) with the same signature and return value (top-1 id list per sample).

    Same scoring quirks as the reference: token scores are log(sigmoid(logit)) (eval.py:61); the running score of a
    beam is divided by len**0.7 at EVERY step before the new term is added (eval.py:53-59), len = position of the
    (last) <EOS> + 1 once the beam has emitted one, else t + 1; the loop stops when every fed token is <PAD>
    (eval.py:116).  The decoder steps run on our kernels (Decoder.forward); beam bookkeeping (top-k over
    beams x vocab, state gather, sequence-length tracking) is batched tensor work on the device: one host sync per
    step (the stop test) instead of the reference's B x beam Python loops."""
    n_vocabs = vocab.n_vocabs
    eos = vocab.word2idx['<EOS>']
    B = encoder_outputs.shape[0]
    dev = encoder_outputs.device
    is_lstm = config.decoder_model == "LSTM"
    if _device_beam_applies(decoder, beam_width, input, hidden, vocab):
        # the whole loop on the device (recnet_decoder_beam): one host read at the end instead of one per step
        seqs, n = decoder.beam(encoder_outputs, beam_width, config.caption_max_len + 1, eos_id=eos)
        return seqs[:, : int(n.item())].tolist()
    inputs = [input]                                             # list over beams of (1,B)
    hiddens = [hidden]
    cum = [torch.zeros(B, dtype=torch.float32, device=dev)]      # log(1.)
    seqs = torch.zeros(B, 1, 0, dtype=torch.long, device=dev)    # (B, beams, t) ids so far
    last_eos = torch.full((B, 1), -1, dtype=torch.long, device=dev)   # position of the last <EOS> per (b, beam), -1 = none
    import contextlib
    scope = decoder.cached_uv(encoder_outputs) if hasattr(decoder, "cached_uv") else contextlib.nullcontext()
    with scope:                       # U.v once for this batch (decoder.py:54 recomputes it every step); nothing survives the block
        seqs = _beam_loop(config, beam_width, n_vocabs, eos, decoder, inputs, hiddens, cum, seqs, last_eos, encoder_outputs, is_lstm)
    return seqs[:, 0].tolist()


def _device_beam_applies(decoder, beam_width, input, hidden, vocab) -> bool:
    """recnet_decoder_beam covers what eval.evaluate passes (eval.py:130-140): a decoder with a fused driver (LSTM with 1-4 layers,
    single-layer GRU), <SOS> start, zero state, <= 8 beams."""
    import os
    if os.environ.get("RECNET_BEAM_DEVICE", "1") != "1" or not hasattr(decoder, "beam"):
        return False
    if not getattr(decoder, "uses_fused_sequence", False) or not 1 <= beam_width <= 8:
        return False
    if not input.is_cuda or vocab.word2idx.get('<PAD>', 0) != 0:
        return False
    hs = hidden if isinstance(hidden, (tuple, list)) else (hidden,)
    return bool((input == vocab.word2idx['<SOS>']).all()) and all(bool((h == 0).all()) for h in hs)


def _beam_loop(config, beam_width, n_vocabs, eos, decoder, inputs, hiddens, cum, seqs, last_eos, encoder_outputs, is_lstm):
    B = encoder_outputs.shape[0]
    dev = encoder_outputs.device
    for t in range(config.caption_max_len + 1):
        cand, next_hiddens = [], []
        for i, (tok, hid, cp) in enumerate(zip(inputs, hiddens, cum)):
            logits, nh = decoder(tok, hid, encoder_outputs)
            next_hiddens.append(nh)
            seq_len = torch.where(last_eos[:, i] >= 0, last_eos[:, i] + 1, torch.full_like(last_eos[:, i], t + 1)).to(torch.float32)
            cand.append(torch.log(torch.sigmoid(logits.float())) + (cp / seq_len ** 0.7).unsqueeze(1))
        flat = torch.cat(cand, dim=1)                            # (B, beams * V)
        top_p, top_i = flat.topk(beam_width, dim=1)              # (B, k)
        tok_ids, src = top_i % n_vocabs, top_i // n_vocabs       # new token and the beam it extends
        ar = torch.arange(B, device=dev)
        if is_lstm:
            H = torch.stack([h[0] for h in next_hiddens])        # (beams, NL, B, Hd)
            Cc = torch.stack([h[1] for h in next_hiddens])
            new_hiddens = [(H[src[:, k], :, ar].transpose(0, 1).contiguous(), Cc[src[:, k], :, ar].transpose(0, 1).contiguous())
                           for k in range(beam_width)]
        else:
            H = torch.stack(next_hiddens)
            new_hiddens = [H[src[:, k], :, ar].transpose(0, 1).contiguous() for k in range(beam_width)]
        prev = seqs[ar.unsqueeze(1), src]                        # (B, k, t)
        seqs = torch.cat((prev, tok_ids.unsqueeze(2)), dim=2)
        prev_eos = last_eos[ar.unsqueeze(1), src]
        last_eos = torch.where(tok_ids == eos, torch.full_like(prev_eos, t), prev_eos)
        inputs = [tok_ids[:, k].view(1, -1) for k in range(beam_width)]
        hiddens, cum = new_hiddens, [top_p[:, k] for k in range(beam_width)]
        if t == config.caption_max_len or bool((tok_ids == 0).all()):
            break
    return seqs


def save_checkpoint(path, iteration, decoder, reconstructor=None, loss=None, config=None):
    """Write the reference's checkpoint layout (train.py:398-420): keys 'iteration', 'dec', 'rec', 'dec_opt', 'rec_opt',
    'loss', 'config' -- so reference tooling (eval.main, eval.py:173-204) can load what this package trained."""
    blob = {'iteration': iteration, 'dec': decoder['model'].state_dict(), 'dec_opt': decoder['optimizer'].state_dict(),
            'loss': loss, 'config': config}
    if reconstructor is not None:
        blob['rec'] = reconstructor['model'].state_dict()
        blob['rec_opt'] = reconstructor['optimizer'].state_dict()
    torch.save(blob, path)


def load_checkpoint(path, decoder, reconstructor=None, map_location=None, restore_optimizers=True):
    """Load a reference-format checkpoint (also ones written by the reference itself) into our modules; the optimiser
    states ('dec_opt' / 'rec_opt', torch.optim.Adam layout) are restored too unless ``restore_optimizers=False``."""
    blob = torch.load(path, map_location=map_location, weights_only=False)
    decoder['model'].load_state_dict(blob['dec'])
    if restore_optimizers and blob.get('dec_opt') is not None and decoder.get('optimizer') is not None:
        decoder['optimizer'].load_state_dict(blob['dec_opt'])            # Adam moments, amsgrad max, step count (train.py:409)
    if reconstructor is not None and 'rec' in blob:
        reconstructor['model'].load_state_dict(blob['rec'])
        if restore_optimizers and blob.get('rec_opt') is not None and reconstructor.get('optimizer') is not None:
            reconstructor['optimizer'].load_state_dict(blob['rec_opt'])
    return blob.get('iteration')
