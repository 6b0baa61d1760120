"""Drop-in mirrors of the reference's three nn.Modules (SURVEY.md section 8b).

Same constructor kwargs, same per-step ``forward`` signatures, same ``state_dict`` keys / shapes / gate order
as models/decoder.py, models/global_reconstructor.py and models/local_reconstructor.py of the reference, so a
reference checkpoint loads with ``load_state_dict``.  The arithmetic runs in librecnet_b200.so:

* ``forward`` (one timestep, models/decoder.py:45) -> operator-level kernels (``ops.py``)
* ``forward_sequence`` (whole teacher-forced loop, what train.forward_* use) -> one C call (``functional.py``)

Extra constructor kwargs after the reference's: ``precision`` ("bf16" | "fp32") and, on Decoder and LocalReconstructor,
``attn_softmax`` (default False = the reference's attention: raw scores, mean over frames / steps; True = the RecNet paper's
softmax-normalised scores and weighted sum).  ``state_dict`` keys and shapes do not depend on either.

Every (cell, n_layers) combination the reference's constructors accept runs on our kernels:
* fused sequence drivers (one C call per loop): LSTM decoder with 1-4 layers, GRU decoder with 1 layer, 1-layer LSTM
  reconstructors over any such decoder, 1-layer GRU reconstructors over a 1-layer decoder -- the configurations the
  reference's config.py / published runs use, and everything bench.py measures.  The same decoders also decode in one C
  call each (``greedy``, ``beam``);
* every other variant (stacked GRU decoder, GRU reconstructor over a stacked decoder, multi-layer reconstructors, > 4
  decoder layers) runs ``forward_sequence`` as a Python loop over the per-step ``forward`` -- the same operator-level
  CUDA kernels (ops.py), autograd glue in between; such decoders also decode step by step.  Slower, never silent:
  ``uses_fused_sequence`` says which one runs.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib as L
from . import functional as Fn
from . import ops
from .rnn_params import RNNParams


def _precision_id(p) -> int:
    if isinstance(p, int):
        return p
    if p not in L.PRECISIONS:
        raise ValueError(f"precision must be one of {list(L.PRECISIONS)}, got {p!r}")
    return L.PRECISIONS[p]


class _RngMixin:
    """(seed, offset) pair living on the device; the offset is bumped once per forward so that every
    iteration draws fresh Philox dropout masks, also under CUDA-graph replay."""

    def _init_rng(self, seed: int = 0x5EED):
        self.register_buffer("_rng", torch.tensor([seed, 0], dtype=torch.int64), persistent=False)

    def _next_rng(self) -> torch.Tensor:
        if self.training:
            self._rng[1] += 1
        return self._rng

    def seed_dropout(self, seed: int):
        self._rng[0] = int(seed)
        self._rng[1] = 0


def _is_lstm(model_name: str) -> bool:
    return model_name == "LSTM"            # models/decoder.py:32-35: anything else is a GRU


def _cell_code(model_name, attn_softmax=False) -> int:
    """The descriptors' `cell` field: recnet_cell, | ATTN_SOFTMAX for the paper's attention."""
    return (L.CELL_LSTM if _is_lstm(model_name) else L.CELL_GRU) | (L.ATTN_SOFTMAX if attn_softmax else 0)


def _attention(Wh, Uv, attn_b, attn_w, V, p, softmax):
    """ops.additive_attention; the reference's mean attention is the plain six-argument call."""
    if softmax:
        return ops.additive_attention(Wh, Uv, attn_b, attn_w, V, p, softmax=True)
    return ops.additive_attention(Wh, Uv, attn_b, attn_w, V, p)


def _zero_state(model_name, n_layers, B, size, device):
    """train.py:28-35 / 82-89 / 112-119: zero (h, c) for LSTM, zero h for GRU."""
    z = lambda: torch.zeros(n_layers, B, size, device=device)
    return (z(), z()) if _is_lstm(model_name) else z()


def _rnn_stack_step(rnn: RNNParams, x, hidden, p, training):
    """One time step through all layers of an nn.LSTM / nn.GRU-shaped stack (inter-layer dropout in train mode).
    x (B,In); hidden ((NL,B,R),(NL,B,R)) [LSTM] or (NL,B,R) [GRU] -> (top-layer output (B,R), new hidden)."""
    is_lstm = rnn.mode == "LSTM"
    hs, cs = [], []
    for l in range(rnn.num_layers):
        w_ih, w_hh, b_ih, b_hh = rnn.layer(l)
        h_prev = hidden[0][l] if is_lstm else hidden[l]
        gi, gh = ops.linear(x, w_ih, b_ih, p), ops.linear(h_prev, w_hh, b_hh, p)
        if is_lstm:
            hl, cl = ops.lstm_cell(gi + gh, hidden[1][l], p)
            cs.append(cl)
        else:
            hl = ops.gru_cell(gi, gh, h_prev, p)
        hs.append(hl)
        x = torch.nn.functional.dropout(hl, rnn.dropout, training) if l < rnn.num_layers - 1 else hl
    return hs[-1], ((torch.stack(hs), torch.stack(cs)) if is_lstm else torch.stack(hs))


def _hiddens4(decoder_hiddens: torch.Tensor) -> torch.Tensor:
    """(L,B,H) -> (L,1,B,H); (L,NLdec,B,H) passes through (train.py:73: hiddens = stack of (NLdec,B,H))."""
    if decoder_hiddens.dim() == 3:
        return decoder_hiddens.unsqueeze(1)
    if decoder_hiddens.dim() != 4:
        raise ValueError(f"decoder_hiddens must be (L,B,H) or (L,n_layers,B,H), got {tuple(decoder_hiddens.shape)}")
    return decoder_hiddens


class Decoder(nn.Module, _RngMixin):
    """models/decoder.py:6-70."""

    def __init__(self, model_name, n_layers, encoder_size, embedding_size, embedding_scale, hidden_size,
                 attn_size, output_size, embedding_dropout, dropout, out_dropout, precision="bf16", attn_softmax=False):
        super().__init__()
        self.model_name = model_name
        self.n_layers = n_layers
        self.encoder_size = encoder_size
        self.embedding_size = embedding_size
        self.embedding_scale = embedding_scale
        self.hidden_size = hidden_size
        self.attn_size = attn_size
        self.output_size = output_size
        self.embedding_dropout_p = embedding_dropout
        self.dropout_p = dropout
        self.out_dropout_p = out_dropout
        self.precision = precision
        self.attn_softmax = bool(attn_softmax)

        # parameter holders, created in the reference's order (decoder.py:22-42) so equal seeds give equal draws
        self.embedding = nn.Embedding(output_size, embedding_size)
        self.attn_W = nn.Linear(hidden_size, attn_size, bias=False)
        self.attn_U = nn.Linear(encoder_size, attn_size, bias=False)
        self.attn_b = nn.Parameter(torch.ones(attn_size), requires_grad=True)
        self.attn_w = nn.Linear(attn_size, 1, bias=False)
        self.rnn = RNNParams(model_name, embedding_size + encoder_size, hidden_size, n_layers, dropout)
        self.out = nn.Linear(hidden_size, output_size)
        self._init_rng(0xDEC0)
        self._uv_scope = None          # [encoder_outputs, U.v or None] while a cached_uv() scope is open

    # ---- helpers ----
    def _params(self):
        w_ih, w_hh, b_ih, b_hh = self.rnn.layer(0)
        base = (self.embedding.weight, self.attn_W.weight, self.attn_U.weight, self.attn_b, self.attn_w.weight,
                w_ih, w_hh, b_ih, b_hh, self.out.weight, self.out.bias)
        extra = tuple(t for l in range(1, self.n_layers) for t in self.rnn.layer(l))       # stacked layers 1..NL-1
        return base + extra

    def _meta(self):
        return dict(H=self.hidden_size, A=self.attn_size, EMB=self.embedding_size, V=self.output_size,
                    precision=_precision_id(self.precision), train=self.training, embedding_scale=self.embedding_scale,
                    p_emb=self.embedding_dropout_p, p_out=self.out_dropout_p, p_layer=self.dropout_p,
                    cell=_cell_code(self.model_name, self.attn_softmax))                   # decoder.py:32-35

    @property
    def uses_fused_sequence(self) -> bool:
        """True when forward_sequence / greedy are ONE C call (csrc/seq_decoder*.cuh); False = per-step kernels in a Python loop."""
        if _is_lstm(self.model_name):
            return 1 <= self.n_layers <= L.MAX_LAYERS
        return self.n_layers == 1

    def cached_uv(self, encoder_outputs):
        """Context manager: inside it, per-step ``forward`` calls on exactly this ``encoder_outputs`` tensor compute
        U.v (decoder.py:54) once instead of once per step.  Nothing is remembered after the block."""
        dec = self

        class _Scope:
            def __enter__(self_):
                self_.prev = dec._uv_scope
                dec._uv_scope = [encoder_outputs, None]
                return dec

            def __exit__(self_, *exc):
                dec._uv_scope = self_.prev
                return False

        return _Scope()

    # ---- whole teacher-forced loop ----
    def forward_sequence(self, tokens_in, targets, ce_weight, encoder_outputs, lambda_reg=None):
        """tokens_in/targets (L,B) int64, ce_weight (L,B) f32 -> (ce scalar, hiddens (L,NL,B,H), reg = sum_p ||p||).
        With ``lambda_reg`` (the module dict's device scalar) output 0 is the assembled loss ce + lambda_reg * reg (train.py:70),
        computed inside the regulariser kernel; reg is then returned for inspection only."""
        if not self.uses_fused_sequence:
            ce, hiddens, reg = self._forward_sequence_stepwise(tokens_in, targets, ce_weight, encoder_outputs)
            return (ce if lambda_reg is None else ce + lambda_reg * reg), hiddens, reg
        meta = self._meta()
        meta["lambda_reg"] = lambda_reg
        return Fn.DecoderSequenceFn.apply(meta, encoder_outputs, tokens_in, targets, ce_weight, self._next_rng(), *self._params())

    def _forward_sequence_stepwise(self, tokens_in, targets, ce_weight, encoder_outputs):
        """The loop body of train.forward_decoder (train.py:41-66) over the per-step ``forward`` (our operator kernels)."""
        Lsteps, B = tokens_in.shape
        hidden = _zero_state(self.model_name, self.n_layers, B, self.hidden_size, encoder_outputs.device)      # train.py:28-35
        ce = 0.0
        hiddens = []
        for t in range(Lsteps):
            logits, hidden = self.forward(tokens_in[t:t + 1], hidden, encoder_outputs)
            if targets is not None and ce_weight is not None:
                lg = logits if logits.dtype == torch.float64 else logits.float()
                logp = torch.log_softmax(lg, dim=1).gather(1, targets[t].unsqueeze(1)).squeeze(1)
                ce = ce - (ce_weight[t] * logp).sum()                                                           # train.py:54-60,68
            hiddens.append(hidden[0] if _is_lstm(self.model_name) else hidden)                                  # train.py:61-64
        reg = Fn.param_norm_sum([p for p in self.parameters()])                                                 # train.py:69
        if not torch.is_tensor(ce):
            ce = torch.zeros((), dtype=torch.float32, device=encoder_outputs.device)
        return ce, torch.stack(hiddens), reg

    @torch.no_grad()
    def teacher_forced_logits(self, tokens_in, encoder_outputs):
        if not self.uses_fused_sequence:
            Lsteps, B = tokens_in.shape
            hidden = _zero_state(self.model_name, self.n_layers, B, self.hidden_size, encoder_outputs.device)
            logits, hiddens = [], []
            with self.cached_uv(encoder_outputs):
                for t in range(Lsteps):
                    lg, hidden = self.forward(tokens_in[t:t + 1], hidden, encoder_outputs)
                    logits.append(lg)
                    hiddens.append(hidden[0] if _is_lstm(self.model_name) else hidden)
            return torch.stack(logits), torch.stack(hiddens)
        return Fn.decoder_teacher_forced_logits(self._meta(), encoder_outputs, tokens_in, self._rng, self._params())

    @torch.no_grad()
    def greedy(self, encoder_outputs, max_steps):
        """eval.greedy_search (eval.py:19-33) on device: returns (ids (max_steps,B) int64 on device, n).  One C call for the decoders
        with a fused driver (LSTM with 1-4 layers, single-layer GRU); the others step through ``forward``."""
        if not self.uses_fused_sequence:
            return self._greedy_stepwise(encoder_outputs, max_steps)
        feats = Fn._f32c(encoder_outputs, "encoder_outputs")
        B = feats.shape[0]
        ids = torch.empty(max_steps, B, dtype=torch.int64, device=feats.device)
        n = torch.zeros(1, dtype=torch.int32, device=feats.device)
        self._decode("greedy", feats, False, (), (max_steps,), (ids, n))
        return ids, n

    @torch.no_grad()
    def _greedy_stepwise(self, encoder_outputs, max_steps):
        """``greedy`` step by step through Decoder.forward (our kernels), arg-max feedback on device, one host read per step; stops
        after the first all-<PAD> step and leaves the remaining rows 0."""
        B = encoder_outputs.shape[0]
        dev = encoder_outputs.device
        hid = _zero_state(self.model_name, self.n_layers, B, self.hidden_size, dev)
        tok = torch.ones(1, B, dtype=torch.long, device=dev)
        was_training = self.training
        self.eval()
        ids = torch.zeros(max_steps, B, dtype=torch.long, device=dev)
        n = max_steps
        with self.cached_uv(encoder_outputs):
            for t in range(max_steps):
                logits, hid = self.forward(tok, hid, encoder_outputs)
                tok = logits.argmax(dim=1).view(1, -1)
                ids[t] = tok[0]
                if bool((tok == 0).all()):
                    n = t + 1
                    break
        self.train(was_training)
        return ids, torch.tensor([n], dtype=torch.int32, device=dev)

    @torch.no_grad()
    def beam(self, encoder_outputs, beam_width, max_steps, eos_id=2):
        """eval.beam_search (eval.py:36-120) as ONE C call: the whole loop, top-k and state gather included, runs on the device.
        Returns (seqs (B, max_steps) int64 on device: top-1 beam per sample, -1 beyond n; n device int32)."""
        feats = Fn._f32c(encoder_outputs, "encoder_outputs")
        B0 = feats.shape[0]
        K = int(beam_width)
        tiled = feats.repeat(K, 1, 1).contiguous()                 # row k * B0 + b = beam k of sample b
        seqs = torch.empty(B0, max_steps, dtype=torch.int64, device=feats.device)
        n = torch.zeros(1, dtype=torch.int32, device=feats.device)
        self._decode("beam", tiled, False, (K, max_steps), (K, max_steps, int(eos_id)), (seqs, n))
        return seqs, n

    @torch.no_grad()
    def sample(self, encoder_outputs, n_samples=1, *, max_steps, temperature=1.0, eos_id=2, seed=None):
        """Stochastic decoding on the device, ONE C call (recnet_decoder_sample): each row draws its tokens from
        softmax(logits / temperature) by Gumbel-max until it emits <EOS> (or <PAD>), then emits <PAD>.  In train mode the logits are
        those of the module's training forward, dropout included (one ``_next_rng()`` per call), so ``forward_sequence`` over
        ``[<SOS>; ids[:-1]]`` with that dropout pair differentiates exactly the distribution the tokens were drawn from.
        Rows are tiled like ``beam``: row k * B0 + b is sample k of video b.  The Gumbel noise pair is (seed, 0), or drawn from torch's
        default generator when ``seed`` is None (reproducible under ``torch.manual_seed``, different on every call).
        Returns (ids (max_steps, K*B0) int64, logp (max_steps, K*B0) f32 = log-prob of each id (0 after the row finished),
        lengths (K*B0,) int32 = tokens up to and including the finishing one, n device int32 = steps until every row finished)."""
        if not self.uses_fused_sequence:
            raise NotImplementedError(f"Decoder.sample: no device sampler for a {self.n_layers}-layer {self.model_name} decoder "
                                      f"(LSTM with 1-{L.MAX_LAYERS} layers and single-layer GRU have one)")
        if seed is None:
            noise = torch.randint(0, 2 ** 62, (2,), dtype=torch.int64)
        else:
            noise = torch.tensor([int(seed), 0], dtype=torch.int64)
        feats = Fn._f32c(encoder_outputs, "encoder_outputs")
        tiled = feats.repeat(int(n_samples), 1, 1).contiguous()
        return self._sample(tiled, max_steps, temperature, eos_id, noise.to(feats.device))

    def _sample(self, feats, max_steps, temperature, eos_id, noise):
        """``sample`` on rows that are already tiled, with the Gumbel (seed, offset) pair `noise` given as a device int64 (2,) tensor."""
        N = feats.shape[0]
        dev = feats.device
        ids = torch.empty(max_steps, N, dtype=torch.int64, device=dev)
        logp = torch.empty(max_steps, N, dtype=torch.float32, device=dev)
        lengths = torch.empty(N, dtype=torch.int32, device=dev)
        n = torch.zeros(1, dtype=torch.int32, device=dev)
        rng = self._next_rng() if self.training else None
        self._decode("sample", feats, self.training, (int(max_steps),),
                     (int(max_steps), float(temperature), int(eos_id), Fn._ptr(rng), noise.data_ptr()), (ids, logp, lengths, n))
        return ids, logp, lengths, n

    def _decode(self, kind, feats, train, query_args, args, outs):
        """One device decode call on the rows of ``feats`` (kind: greedy, beam or sample): the descriptor (L = 1, train mode only when
        ``train``), a workspace sized by recnet_<kind>_workspace_bytes(desc, *query_args), the packed parameters, then
        recnet_decoder_<kind>(desc, params, feats, *args, workspace, its size, *outs, stream)."""
        import ctypes as C
        lib = L.lib()
        N, T, E = feats.shape
        meta = self._meta()
        d = L.decoder_desc(B=N, T=T, E=E, H=meta["H"], A=meta["A"], EMB=meta["EMB"], V=meta["V"], L=1,
                           precision=meta["precision"], train=int(train), embedding_scale=float(meta["embedding_scale"]),
                           p_emb_drop=float(meta["p_emb"]), p_out_drop=float(meta["p_out"]), cell=meta["cell"], n_layers=self.n_layers,
                           p_layer_drop=float(meta["p_layer"]))
        query = f"recnet_{kind}_workspace_bytes"
        nbytes = getattr(lib, query)(C.byref(d), *query_args)
        if nbytes < 0:
            L.check(int(nbytes), query)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=feats.device)
        params = tuple(Fn._f32c(p, "param") for p in self._params())
        w = Fn._pack(L.decoder_tensors, params)
        L.check(getattr(lib, f"recnet_decoder_{kind}")(C.byref(d), C.byref(w), feats.data_ptr(), *args, ws.data_ptr(), nbytes,
                                                      *(t.data_ptr() for t in outs), Fn._stream()), f"recnet_decoder_{kind}")

    # ---- single timestep (reference API) ----
    def forward(self, input, hidden, encoder_outputs):
        """input (1,B) int64; hidden ((NL,B,H),(NL,B,H)) [LSTM] or (NL,B,H) [GRU]; encoder_outputs (B,T,E) -> (logits (B,V), hidden)."""
        p = _precision_id(self.precision)
        h = hidden[0][-1] if _is_lstm(self.model_name) else hidden[-1]                                     # decoder.py:50-53: top layer
        emb = torch.nn.functional.embedding(input[0], self.embedding.weight) * self.embedding_scale      # decoder.py:46-47
        emb = torch.nn.functional.dropout(emb, self.embedding_dropout_p, self.training)                   # decoder.py:48
        # U.v is time-invariant (the reference recomputes it every step, decoder.py:54).  It is recomputed here on every call
        # unless the caller opened an explicit scope for ONE sequence (``with decoder.cached_uv(encoder_outputs):`` -- what
        # the greedy / beam loops over this method do); the scope is tied to the identity of that tensor, holds a reference
        # to it (so the allocator cannot hand its address to another batch), and ends with the ``with`` block.  The training
        # hot path (forward_sequence) hoists the projection out of the loop altogether.
        B, T, E = encoder_outputs.shape
        scope = self._uv_scope
        if scope is not None and scope[0] is encoder_outputs and not (torch.is_grad_enabled() and self.attn_U.weight.requires_grad):
            if scope[1] is None:
                scope[1] = ops.linear(encoder_outputs.reshape(B * T, E), self.attn_U.weight, None, p).view(B, T, -1)
            Uv = scope[1]
        else:
            Uv = ops.linear(encoder_outputs.reshape(B * T, E), self.attn_U.weight, None, p).view(B, T, -1)
        Wh = ops.linear(h, self.attn_W.weight, None, p)                                                   # decoder.py:51
        ctx = _attention(Wh, Uv, self.attn_b, self.attn_w.weight, encoder_outputs, p, self.attn_softmax)          # decoder.py:55-61
        # layer 0 takes [emb ; ctx], layer l the (dropped-out) output of layer l-1 (nn.LSTM / nn.GRU, decoder.py:64-66)
        h_top, hidden = _rnn_stack_step(self.rnn, torch.cat((emb, ctx), dim=1), hidden, p, self.training)
        logits = ops.linear(h_top, self.out.weight, self.out.bias, p)                                     # decoder.py:68
        logits = torch.nn.functional.dropout(logits, self.out_dropout_p, self.training)                    # decoder.py:69
        return logits, hidden


class _ReconstructorBase(nn.Module, _RngMixin):
    def _fused_ok(self, decoder_hiddens) -> bool:
        """One C call (csrc/seq_recon*.cuh) for 1-layer reconstructors: LSTM cells over any decoder depth <= 4, GRU cells over a
        1-layer decoder; everything else loops over the per-step ``forward``."""
        nld = decoder_hiddens.size(1) if decoder_hiddens.dim() == 4 else 1
        if self.n_layers != 1:
            return False
        return nld <= L.MAX_LAYERS if _is_lstm(self.model_name) else nld == 1

    def _all_params(self):
        return [p for p in self.parameters()]


class GlobalReconstructor(_ReconstructorBase):
    """models/global_reconstructor.py:6-46."""

    def __init__(self, model_name, n_layers, decoder_hidden_size, hidden_size, dropout, decoder_dropout, caption_max_len,
                 precision="bf16"):
        super().__init__()
        self.model_name = model_name
        self.n_layers = n_layers
        self.decoder_hidden_size = decoder_hidden_size
        self.hidden_size = hidden_size
        self.dropout_p = dropout
        self.decoder_dropout_p = decoder_dropout
        self.caption_max_len = caption_max_len
        self.precision = precision
        self.rnn = RNNParams(model_name, decoder_hidden_size * 2, hidden_size, n_layers, dropout)
        self.out = nn.Linear(hidden_size, hidden_size)
        self._init_rng(0x610B)

    def _params(self):
        w_ih, w_hh, b_ih, b_hh = self.rnn.layer(0)
        return (w_ih, w_hh, b_ih, b_hh, self.out.weight, self.out.bias)

    def forward_sequence(self, decoder_hiddens, encoder_outputs, lambda_reg=None):
        """decoder_hiddens (L,NLdec,B,H) or (L,B,H); encoder_outputs (B,T,R) -> (MSE(mean_t out, mean_tau feats) / L, reg = sum_p ||p||).
        With ``lambda_reg`` output 0 is the assembled loss (train.py:100-102)."""
        if not self._fused_ok(decoder_hiddens):
            loss, reg = self._forward_sequence_stepwise(decoder_hiddens, encoder_outputs)
            return (loss if lambda_reg is None else loss + lambda_reg * reg), reg
        hid = _sequence_hiddens(decoder_hiddens)
        meta = dict(precision=_precision_id(self.precision), train=self.training, p_drop=self.decoder_dropout_p, lambda_reg=lambda_reg,
                    caption_max_len=self.caption_max_len, cell=L.CELL_LSTM if self.model_name == "LSTM" else L.CELL_GRU)
        return Fn.GlobalReconstructorFn.apply(meta, hid, encoder_outputs, self._next_rng(), *self._params())

    def _forward_sequence_stepwise(self, decoder_hiddens, encoder_outputs):
        """train.forward_global_reconstructor (train.py:78-105) over the per-step ``forward``."""
        hid = _hiddens4(decoder_hiddens)
        Lsteps, B = hid.size(0), hid.size(2)
        hidden = _zero_state(self.model_name, self.n_layers, B, self.hidden_size, hid.device)               # train.py:82-89
        outs = []
        for t in range(Lsteps):
            out, hidden = self.forward(hid[t], hidden, hid)                                                 # train.py:93-95
            outs.append(out)
        loss = torch.nn.functional.mse_loss(torch.stack(outs).mean(0), encoder_outputs.mean(1)) / Lsteps   # train.py:96-100
        return loss, Fn.param_norm_sum(self._all_params())                                                  # train.py:101

    def forward(self, input, hidden, decoder_hiddens):
        """input (NLdec,B,H) = decoder_hiddens[t]; hidden ((NL,B,R),(NL,B,R)) [LSTM] or (NL,B,R) [GRU]; decoder_hiddens (L,NLdec,B,H)."""
        p = _precision_id(self.precision)
        hid = _hiddens4(decoder_hiddens)
        Lsteps = hid.size(0)
        mp = hid.mean(dim=(0, 1)) / Lsteps * self.caption_max_len                        # global_reconstructor.py:33-37
        mp = torch.nn.functional.dropout(mp, self.decoder_dropout_p, self.training)      # :38
        x = torch.cat((input[0], mp), 1)                                                 # :40 (layer-0 state of step t)
        h_top, hidden = _rnn_stack_step(self.rnn, x, hidden, p, self.training)           # :43
        out = ops.linear(h_top, self.out.weight, self.out.bias, p)                       # :45
        return out, hidden


class LocalReconstructor(_ReconstructorBase):
    """models/local_reconstructor.py:6-55."""

    def __init__(self, model_name, n_layers, decoder_hidden_size, hidden_size, dropout, decoder_dropout, attn_size,
                 precision="bf16", attn_softmax=False):
        super().__init__()
        self.model_name = model_name
        self.n_layers = n_layers
        self.decoder_hidden_size = decoder_hidden_size
        self.hidden_size = hidden_size
        self.dropout_p = dropout
        self.decoder_dropout_p = decoder_dropout
        self.attn_size = attn_size
        self.precision = precision
        self.attn_softmax = bool(attn_softmax)
        self.attn_W = nn.Linear(hidden_size, attn_size, bias=False)
        self.attn_U = nn.Linear(decoder_hidden_size, attn_size, bias=False)
        self.attn_b = nn.Parameter(torch.ones(attn_size), requires_grad=True)
        self.attn_w = nn.Linear(attn_size, 1, bias=False)
        self.rnn = RNNParams(model_name, decoder_hidden_size, hidden_size, n_layers, dropout)
        self.out = nn.Linear(hidden_size, hidden_size)
        self._init_rng(0x10CA)

    def _params(self):
        w_ih, w_hh, b_ih, b_hh = self.rnn.layer(0)
        return (self.attn_W.weight, self.attn_U.weight, self.attn_b, self.attn_w.weight, w_ih, w_hh, b_ih, b_hh,
                self.out.weight, self.out.bias)

    def forward_sequence(self, decoder_hiddens, encoder_outputs, lambda_reg=None):
        """decoder_hiddens (L,NLdec,B,H) or (L,B,H); encoder_outputs (B,S,R) -> (MSELoss(outputs^T, encoder_outputs), reg = sum_p ||p||).
        With ``lambda_reg`` output 0 is the assembled loss (train.py:128-130)."""
        if not self._fused_ok(decoder_hiddens):
            loss, reg = self._forward_sequence_stepwise(decoder_hiddens, encoder_outputs)
            return (loss if lambda_reg is None else loss + lambda_reg * reg), reg
        hid = _sequence_hiddens(decoder_hiddens)
        meta = dict(A=self.attn_size, precision=_precision_id(self.precision), train=self.training, lambda_reg=lambda_reg,
                    p_drop=self.decoder_dropout_p, cell=_cell_code(self.model_name, self.attn_softmax))
        return Fn.LocalReconstructorFn.apply(meta, hid, encoder_outputs, self._next_rng(), *self._params())

    def _forward_sequence_stepwise(self, decoder_hiddens, encoder_outputs):
        """train.forward_local_reconstructor (train.py:108-131) over the per-step ``forward``."""
        hid = _hiddens4(decoder_hiddens)
        B, S = hid.size(2), encoder_outputs.size(1)
        hidden = _zero_state(self.model_name, self.n_layers, B, self.hidden_size, hid.device)               # train.py:112-119
        outs = []
        for _ in range(S):                                                                                  # train.py:122-124
            out, hidden = self.forward(hidden, hid)
            outs.append(out)
        loss = torch.nn.functional.mse_loss(torch.stack(outs).transpose(0, 1), encoder_outputs)             # train.py:125-128
        return loss, Fn.param_norm_sum(self._all_params())                                                  # train.py:129

    def forward(self, hidden, decoder_hiddens):
        """hidden ((NL,B,R),(NL,B,R)) [LSTM] or (NL,B,R) [GRU]; decoder_hiddens (L,NLdec,B,H) -> (out (B,R), hidden)."""
        p = _precision_id(self.precision)
        h_prev = hidden[0][-1] if _is_lstm(self.model_name) else hidden[-1]
        hid = _hiddens4(decoder_hiddens)                                                 # (L,NLdec,B,H)
        Lsteps, NLd, B, H = hid.shape
        Wh = ops.linear(h_prev, self.attn_W.weight, None, p)                             # local_reconstructor.py:39-42
        xs = []
        for j in range(NLd):             # the same query attends over the L states of every decoder layer (:43-49), mean (or softmax) over L
            hj = hid[:, j]
            Uv = ops.linear(hj.reshape(Lsteps * B, H), self.attn_U.weight, None, p).view(Lsteps, B, -1).transpose(0, 1)
            xs.append(_attention(Wh, Uv.contiguous(), self.attn_b, self.attn_w.weight, hj.transpose(0, 1).contiguous(), p,
                                 self.attn_softmax))
        x = torch.nn.functional.dropout(torch.stack(xs), self.decoder_dropout_p, self.training)      # (NLdec,B,H)  :50
        # nn.LSTM / nn.GRU read dim 0 of its input as TIME: NLdec pseudo-steps (:52); the output of the FIRST one is projected (:54)
        first = None
        for j in range(NLd):
            h_top, hidden = _rnn_stack_step(self.rnn, x[j], hidden, p, self.training)
            if j == 0:
                first = h_top
        out = ops.linear(first, self.out.weight, self.out.bias, p)                       # :54
        return out, hidden


def _sequence_hiddens(decoder_hiddens: torch.Tensor) -> torch.Tensor:
    """(L,1,B,H) -> (L,B,H); a stacked decoder's (L,NLdec,B,H) passes through to the fused drivers."""
    if decoder_hiddens.dim() == 4 and decoder_hiddens.size(1) == 1:
        return decoder_hiddens[:, 0]
    return decoder_hiddens
