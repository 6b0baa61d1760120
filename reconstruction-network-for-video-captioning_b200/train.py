"""Step drivers and losses: mirrors of the reference's train.forward_decoder / forward_global_reconstructor /
forward_local_reconstructor / build_decoder / build_reconstructor (train.py:17-197), same names, same
arguments, same return values, same module-dict convention {'model','loss','optimizer','lambda_reg'} and the
same global config object ``C`` -- but each driver is ONE call into the CUDA sequence kernels instead of a
Python loop of ~400 ATen ops per step.
"""
from __future__ import annotations

import os
import random

import torch

from .config import TrainConfig as C
from . import functional as Fn
from .models import Decoder, GlobalReconstructor, LocalReconstructor
from .optim import ClipAdam


def _optimizer_impl() -> str:
    impl = os.environ.get("RECNET_OPTIMIZER") or getattr(C, "optimizer_impl", "recnet")
    if impl not in ("torch", "recnet"):
        raise ValueError(f"optimizer_impl must be 'torch' or 'recnet', got {impl!r}")
    return impl


def _num_steps(target_masks: torch.Tensor, caption_max_len: int) -> int:
    """Loop length of train.py:41,66: stop after step t when masks[t+1] is all False (one host read,
    the reference does two per step)."""
    any_t = target_masks.any(dim=1)
    n = int(any_t[: caption_max_len + 1].sum().item()) if bool(any_t[0]) else 0
    # masks are prefix-shaped (PAD only after EOS, dataset/MSVD.py:111-117) so the count of non-empty rows is L
    return max(1, min(n, caption_max_len + 1))


def forward_decoder(decoder, encoder_outputs, targets, target_masks, teacher_forcing_ratio=0., n_steps=None):
    """train.py:17-75.  Returns (loss, hiddens (L,NL,B,H), output_indices).
    ``target_masks`` is ``targets > <PAD>`` as the reference builds it (train.py:246); it may be None when ``n_steps`` is given.
    ``n_steps``: optional static loop length (skips the host read; needed under CUDA-graph capture)."""
    pad, sos_id = C.init_word2idx['<PAD>'], C.init_word2idx['<SOS>']
    if target_masks is None and n_steps is None:
        target_masks = targets > pad                               # the host-side loop length needs it
    model = decoder['model']
    L = n_steps if n_steps is not None else _num_steps(target_masks, C.caption_max_len)
    B = encoder_outputs.shape[0]
    dev = encoder_outputs.device
    use_teacher_forcing = random.random() <= teacher_forcing_ratio                                          # train.py:38
    output_indices = torch.empty(0, dtype=torch.long)
    if use_teacher_forcing and targets.is_cuda:
        # <SOS> row + shifted targets (train.py:25,44-45) and the CE weights mask / (n_t * sum_t n_t) (train.py:54-60,68): one launch
        tokens_in, ce_weight = Fn.teacher_forcing_inputs(targets, L, pad, sos_id)
    else:
        sos = torch.full((1, B), sos_id, dtype=torch.long, device=dev)                                      # train.py:25
        if use_teacher_forcing:
            tokens_in = torch.cat((sos, targets[: L - 1]), dim=0)                                           # train.py:44-45
        else:
            # argmax feedback (train.py:47-51): decode greedily on device, then replay those tokens through the
            # differentiable sequence kernel (identical arithmetic in eval mode, where validation uses it, train.py:329).
            # KNOWN DIFFERENCE in train mode with teacher_forcing_ratio < 1 (the reference's default is 1.0, config.py:71): the
            # reference feeds back the argmax of the SAME pass's dropout-perturbed logits; here the tokens come from a dropout-free
            # greedy pass, so the fed-back tokens follow the eval-mode distribution.  Losses / gradients for a GIVEN token sequence
            # are identical.  The device greedy keeps feeding the argmax back after an all-<PAD> step, as the reference does.
            # (The step-wise greedy of the decoders without a fused driver -- stacked GRU, > 4 layers -- stops once every token is
            # <PAD> and leaves the remaining rows 0 = <PAD>, which is what the reference would decode from an all-<PAD> row only by
            # accident.)
            ids, _ = model.greedy(encoder_outputs, L)
            tokens_in = torch.cat((sos, ids[: L - 1]), dim=0)
            output_indices = ids[:L].cpu()
        if target_masks is None:
            target_masks = targets > pad
        m = target_masks[:L].to(torch.float32)
        n_t = m.sum(dim=1, keepdim=True)                                                                    # train.py:57
        ce_weight = m / (n_t.clamp_min(1.0) * n_t.sum())                                                    # mean over n_t, then / sum n_t (train.py:54-60,68)
    # loss = CE + lambda_reg * sum_p ||p|| (train.py:69-70), assembled inside the sequence call
    loss, hiddens, _ = model.forward_sequence(tokens_in, targets[:L], ce_weight, encoder_outputs, lambda_reg=decoder['lambda_reg'])
    return loss, hiddens, output_indices                                                                    # (L,NL,B,H), train.py:73-75


def self_critical_weights(rewards, baseline, lengths, n_steps):
    """ce_weight (n_steps, K*B0) of self-critical training: (rewards[row] - baseline[row % B0]) * [t < lengths[row]] / (K*B0).
    With it the cross entropy of forward_sequence is -sum_row advantage_row / N * sum_t log p(ids[t, row]), the policy-gradient loss."""
    N = rewards.shape[0]
    B0 = baseline.shape[0]
    adv = rewards.float() - baseline.float().repeat(N // B0)                      # row k * B0 + b is sample k of video b
    steps = torch.arange(n_steps, device=lengths.device).unsqueeze(1)
    mask = (steps < lengths.long().unsqueeze(0)).float()
    return mask * (adv / N).unsqueeze(0), adv


def forward_decoder_self_critical(decoder, encoder_outputs, reward_fn, n_samples=1, temperature=1.0, max_steps=None):
    """Self-critical sequence training (Rennie et al., 2017), one forward: sample ``n_samples`` captions per video on the device in the
    module's current mode (``Decoder.sample``), decode the greedy baseline (``Decoder.greedy``), score both with
    ``reward_fn(sample_ids (n, K*B0), greedy_ids (max_steps, B0)) -> (rewards (K*B0,), baseline (B0,))``, then replay the samples
    through the fused sequence kernels with ce_weight = advantage * step mask / (K*B0) (``self_critical_weights``), the dropout pair
    the sampler read and ``+ lambda_reg * reg`` as in ``forward_decoder``.  Returns (loss, hiddens (n, NL, K*B0, H), info) with info =
    {rewards, baseline, advantage, ids, lengths, logp}; the caller runs backward and the optimiser step (or adds a reconstructor loss on
    ``hiddens`` over the features tiled K times) as in ``train_step``.
    The replay computes the sampler's logits again with other kernels: in fp32 they agree to fp32 rounding; in bf16 the replay runs
    the training kernels (the cluster / projected-feature loop and the batched vocabulary GEMM) rather than the sampler's per-step
    kernels, so they agree to bf16 rounding only."""
    sos_id, eos_id = C.init_word2idx['<SOS>'], C.init_word2idx['<EOS>']
    model = decoder['model']
    L = max_steps if max_steps is not None else C.caption_max_len + 1
    K = int(n_samples)
    ids, logp, lengths, n = model.sample(encoder_outputs, K, max_steps=L, temperature=temperature, eos_id=eos_id)
    rng = model._rng.clone()               # the pair the sampler read; the buffer itself moves on with the next training forward
    greedy_ids, _ = model.greedy(encoder_outputs, L)
    n = int(n)
    ids, logp = ids[:n], logp[:n]
    rewards, baseline = reward_fn(ids, greedy_ids)
    ce_weight, adv = self_critical_weights(rewards, baseline, lengths, n)
    N = ids.shape[1]
    tokens_in = torch.cat((torch.full((1, N), sos_id, dtype=torch.long, device=ids.device), ids[:-1]), dim=0)
    meta = model._meta()
    meta["lambda_reg"] = decoder['lambda_reg']
    feats = encoder_outputs.repeat(K, 1, 1).contiguous()
    loss, hiddens, _ = Fn.DecoderSequenceFn.apply(meta, feats, tokens_in, ids, ce_weight.contiguous(), rng, *model._params())
    return loss, hiddens, {"rewards": rewards, "baseline": baseline, "advantage": adv, "ids": ids, "lengths": lengths, "logp": logp}


def forward_global_reconstructor(decoder_hiddens, encoder_outputs, reconstructor):
    """train.py:78-105."""
    model = reconstructor['model']
    loss, _ = model.forward_sequence(decoder_hiddens, encoder_outputs, lambda_reg=reconstructor['lambda_reg'])    # incl. /L (train.py:100) and + lambda * reg (:101-102)
    return loss


def forward_local_reconstructor(decoder_hiddens, encoder_outputs, reconstructor):
    """train.py:108-131."""
    model = reconstructor['model']
    loss, _ = model.forward_sequence(decoder_hiddens, encoder_outputs, lambda_reg=reconstructor['lambda_reg'])    # incl. + lambda * reg (train.py:129-130)
    return loss


def build_decoder(n_vocabs):
    """train.py:134-160."""
    model = Decoder(
        model_name=C.decoder_model, n_layers=C.decoder_n_layers, encoder_size=C.encoder_output_size,
        embedding_size=C.embedding_size, embedding_scale=C.embedding_scale, hidden_size=C.decoder_hidden_size,
        attn_size=C.decoder_attn_size, output_size=n_vocabs, embedding_dropout=C.embedding_dropout,
        dropout=C.decoder_dropout, out_dropout=C.decoder_out_dropout, precision=C.precision,
        attn_softmax=C.decoder_attn_softmax).to(C.device)
    if _optimizer_impl() == "recnet":      # clip (train.py:269-270) folded into the Adam pass
        optimizer = ClipAdam(model.parameters(), lr=C.decoder_learning_rate, weight_decay=C.decoder_weight_decay,
                             amsgrad=C.decoder_use_amsgrad, max_grad_norm=C.gradient_clip if C.use_gradient_clip else None)
    else:
        optimizer = torch.optim.Adam(model.parameters(), lr=C.decoder_learning_rate, weight_decay=C.decoder_weight_decay,
                                     amsgrad=C.decoder_use_amsgrad, fused=True, capturable=True)
    lambda_reg = torch.tensor(0.001, device=C.device)
    return {'model': model, 'loss': torch.nn.CrossEntropyLoss(), 'optimizer': optimizer, 'lambda_reg': lambda_reg}


def build_reconstructor():
    """train.py:163-197."""
    if C.reconstructor_type == "local":
        model = LocalReconstructor(
            model_name=C.reconstructor_model, n_layers=C.reconstructor_n_layers, decoder_hidden_size=C.decoder_hidden_size,
            hidden_size=C.reconstructor_hidden_size, dropout=C.reconstructor_dropout,
            decoder_dropout=C.reconstructor_decoder_dropout, attn_size=C.reconstructor_attn_size, precision=C.precision,
            attn_softmax=C.reconstructor_attn_softmax)
    elif C.reconstructor_type == "global":
        model = GlobalReconstructor(
            model_name=C.reconstructor_model, n_layers=C.reconstructor_n_layers, decoder_hidden_size=C.decoder_hidden_size,
            hidden_size=C.reconstructor_hidden_size, dropout=C.reconstructor_dropout,
            decoder_dropout=C.reconstructor_decoder_dropout, caption_max_len=C.caption_max_len, precision=C.precision)
    else:
        raise NotImplementedError("Unknown reconstructor: {}".format(C.reconstructor_type))
    model = model.to(C.device)
    if _optimizer_impl() == "recnet":
        optimizer = ClipAdam(model.parameters(), lr=C.reconstructor_learning_rate, weight_decay=C.reconstructor_weight_decay,
                             amsgrad=C.reconstructor_use_amsgrad)
    else:
        optimizer = torch.optim.Adam(model.parameters(), lr=C.reconstructor_learning_rate,
                                     weight_decay=C.reconstructor_weight_decay, amsgrad=C.reconstructor_use_amsgrad,
                                     fused=True, capturable=True)
    lambda_reg = torch.tensor(0.01, device=C.device)
    return {'model': model, 'loss': torch.nn.MSELoss(), 'optimizer': optimizer, 'lambda_reg': lambda_reg}


def forward_reconstructor_for(kind):
    if kind == "global":
        return forward_global_reconstructor
    if kind == "local":
        return forward_local_reconstructor
    raise NotImplementedError("Unknown reconstructor type '{}'".format(kind))          # train.py:240


def train_step(decoder, reconstructor, encoder_outputs, targets, n_steps=None, lambda_recon=1.0, zero_grad=True,
               optimizer_step=True, grad_hook=None, reducer=None):
    """One iteration of the reference's loop body (train.py:243-273): decoder + reconstructor forward, combined
    loss, backward, clip, two Adam steps.  ``grad_hook`` (if given) runs between backward and clip -- the
    data-parallel gradient all-reduce plugs in there.  ``reducer`` (parallel.make_reducer(...), modules in the order
    [reconstructor, decoder]) does the same with overlap: the reconstructor's optimiser step runs while the decoder's gradients
    are still being averaged (the two steps are independent; the clip, train.py:269-270, only concerns the decoder).
    Returns (loss, decoder_loss, recon_loss) device scalars."""
    # train.py:246 (the fused path derives the mask from the targets itself; the host-side loop length needs it when n_steps is None)
    target_masks = None if (n_steps is not None and targets.is_cuda) else targets > C.init_word2idx['<PAD>']
    if (grad_hook is None and targets.is_cuda and os.environ.get("RECNET_BG_WGRAD", "1") == "1"
            and os.environ.get("RECNET_BG_NORMS", "1") == "1"):                    # (also in data-parallel steps: no reducer involved)
        # the regularisers' squared norms depend on the parameters only: on the lane, underneath the decoder's forward loop
        Fn.prefetch_param_norms(*[m._params() for m in (decoder['model'], reconstructor['model'] if reconstructor else None)
                                  if m is not None and hasattr(m, "_params") and getattr(m, "uses_fused_sequence", True)])
    decoder['model'].train()
    split_fwd = (grad_hook is None and reconstructor is not None and targets.is_cuda and os.environ.get("RECNET_BG_WGRAD", "1") == "1"
                 and os.environ.get("RECNET_BG_FWD", "1") == "1")
    with Fn.split_decoder_forward(enabled=split_fwd):      # vocabulary projection + CE on the lane, next to the reconstructor's staging
        dec_loss, hiddens, _ = forward_decoder(decoder, encoder_outputs, targets, target_masks,
                                               C.decoder_teacher_forcing_ratio, n_steps=n_steps)
    rec_loss = None
    if reconstructor is not None:
        reconstructor['model'].train()
        rec_loss = forward_reconstructor_for(C.reconstructor_type)(hiddens, encoder_outputs, reconstructor)
    Fn.wait_forward_tail()                                 # the decoder's loss is final on the main stream from here on
    if reconstructor is not None:
        loss = dec_loss + rec_loss if lambda_recon == 1.0 else dec_loss + lambda_recon * rec_loss           # train.py:260
    else:
        loss = dec_loss
    if zero_grad:
        decoder['optimizer'].zero_grad(set_to_none=True)
        if reconstructor is not None:
            reconstructor['optimizer'].zero_grad(set_to_none=True)
    # Background lane (functional.deferred_weight_grads), single-GPU runs: the local reconstructor's weight-gradient GEMMs, its
    # regulariser gradient + optimiser step and the decoder's vocabulary-projection gradients run on a second stream underneath /
    # next to the decoder's backward; joined at the end of this function.  Data-parallel runs keep the plain order: there the
    # reducer overlaps the reconstructor's all-reduce with the decoder's backward and its optimiser step with the decoder's
    # all-reduce, and a third tenant on the SMs (measured at N = 2, profiles/r2_j_step_timeline.md) costs more than it hides.
    use_bg = _background_ok(grad_hook, reducer)
    local_rec = reconstructor is not None and isinstance(reconstructor['model'], LocalReconstructor)
    tail = _background_tail(reconstructor) if (use_bg and optimizer_step and local_rec) else None
    with Fn.deferred_weight_grads(enabled=use_bg):
        loss.backward()                                                                                     # train.py:268
    if grad_hook is not None:
        grad_hook()
    rec_stepped = tail.disarm() if tail is not None else False
    if reducer is not None:
        if reconstructor is not None and optimizer_step:
            reducer.wait_first()                       # reconstructor gradients averaged; the decoder's go out underneath ...
            reconstructor['optimizer'].step()          # ... the reconstructor's Adam step (train.py:273; order of :271-273 is immaterial)
            rec_stepped = True
        reducer.wait()
    if optimizer_step:
        own_clip = isinstance(decoder['optimizer'], ClipAdam) and decoder['optimizer'].param_groups[0].get('max_grad_norm')
        if C.use_gradient_clip and not own_clip:
            torch.nn.utils.clip_grad_norm_(decoder['model'].parameters(), C.gradient_clip, foreach=True)    # train.py:269-270
        decoder['optimizer'].step()
        if reconstructor is not None and not rec_stepped:
            Fn.join_background()
            reconstructor['optimizer'].step()
    Fn.join_background()
    return loss, dec_loss, rec_loss


def _background_ok(grad_hook, reducer) -> bool:
    return grad_hook is None and reducer is None and os.environ.get("RECNET_BG_WGRAD", "1") == "1"


class _BackgroundTail:
    """Fires once every reconstructor gradient of this backward has been accumulated: queues the reconstructor's optimiser step
    (train.py:273) on the background lane (functional.py: ``late`` slot, behind the regulariser gradient)."""

    def __init__(self, reconstructor):
        self.params = [p for p in reconstructor['model'].parameters() if p.requires_grad]
        self.optimizer = reconstructor['optimizer']
        self.armed = False
        self.fired = False
        self.count = 0
        self.hooks = [p.register_post_accumulate_grad_hook(self._hook) for p in self.params]

    def _hook(self, _p):
        if not self.armed:
            return
        self.count += 1
        if self.count < len(self.params):
            return
        self.count = 0
        if not Fn.background_pending():                # the backward did not defer anything (e.g. a stacked decoder)
            return
        Fn.background_late(self.optimizer.step)
        self.fired = True

    def arm(self):
        self.armed, self.fired, self.count = True, False, 0
        return self

    def disarm(self) -> bool:
        self.armed = False
        return self.fired


def _background_tail(reconstructor):
    t = reconstructor.get('_bg_tail')
    if t is None or t.optimizer is not reconstructor['optimizer']:
        t = reconstructor['_bg_tail'] = _BackgroundTail(reconstructor)
    return t.arm()
