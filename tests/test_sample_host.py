"""CPU checks of the device sampler and of self-critical training: the C entry points' argument checks (answered before any launch,
null buffers, no GPU), the sample workspace against the greedy one, the fp64 sampling oracle (tests/sample_oracle.py) against a direct
Philox evaluation and against the oracle's greedy search, Decoder.sample's refusal of decoders without a fused driver, and the
assembly of the self-critical loss weights around a stub decoder."""
import ctypes as C

import numpy as np
import pytest
import torch

import recnet_b200
from recnet_b200 import _lib as L
from recnet_b200 import functional as Fn
from recnet_b200 import train as T
from oracle import recnet_oracle as O
from tests import sample_oracle as SM
from tests.philox_ref import philox4x32_10

BAD_SHAPE, ALIGNMENT, UNSUPPORTED = -1, -2, -4
SMALL = dict(B=6, T=5, E=16, H=8, A=8, EMB=8, V=11, L=1)
DEC_SHAPES = {"bench": dict(B=100, T=28, E=1536, H=512, A=128, EMB=468, V=4188, L=31),
              "small": dict(B=4, T=5, E=16, H=8, A=6, EMB=8, V=11, L=3)}


def _desc(cell=L.CELL_LSTM, n_layers=1, precision=L.PREC_FP32, train=0, shape=SMALL):
    return L.decoder_desc(precision=precision, train=train, embedding_scale=1.0, p_emb_drop=0.5, p_out_drop=0.5, cell=cell,
                          n_layers=n_layers, p_layer_drop=0.5, **shape)


def _sample_call(d, max_steps=31, temperature=1.0):
    w = L.decoder_tensors()
    return L.lib().recnet_decoder_sample(d, C.byref(w), None, max_steps, temperature, 2, None, None, None, 0, None, None, None, None, None)


@pytest.mark.parametrize("precision", [L.PREC_FP32, L.PREC_BF16])
def test_sample_entry_points_refuse_bad_arguments_before_any_launch(precision):
    lib = L.lib()
    for f in (lambda d: lib.recnet_sample_workspace_bytes(d, 31), _sample_call):
        assert f(None) == BAD_SHAPE
        assert f(C.byref(_desc(precision=7))) == UNSUPPORTED
        for sm in (0, L.ATTN_SOFTMAX):
            assert f(C.byref(_desc(L.CELL_GRU | sm, 2, precision))) == UNSUPPORTED
            assert f(C.byref(_desc(L.CELL_LSTM | sm, L.MAX_LAYERS + 1, precision))) == UNSUPPORTED
    d = C.byref(_desc(precision=precision, train=1))
    for steps in (0, 65):
        assert lib.recnet_sample_workspace_bytes(d, steps) == BAD_SHAPE
        assert _sample_call(d, max_steps=steps) == BAD_SHAPE
    for tau in (0.0, -1.0, float("nan")):
        assert _sample_call(d, temperature=tau) == BAD_SHAPE
    assert lib.recnet_sample_workspace_bytes(d, 64) > 0


def test_sample_workspace_covers_the_greedy_plan():
    """The sampler's plan extends the greedy plan of the general step path.  recnet_greedy_workspace_bytes of a bf16 single-layer LSTM
    also reserves room for the projected-feature greedy driver, which the sampler never runs; that case is left out.  The small pinned
    shape has A = 6, which no decode loop runs (A must be a multiple of 4): the sampler's query says so."""
    lib = L.lib()
    assert lib.recnet_sample_workspace_bytes(C.byref(_desc(shape=DEC_SHAPES["small"])), 64) == ALIGNMENT
    for shape in (DEC_SHAPES["bench"], dict(DEC_SHAPES["small"], A=8)):
        for prec in (L.PREC_FP32, L.PREC_BF16):
            for cell, layers in ((L.CELL_LSTM, 1), (L.CELL_LSTM, 2), (L.CELL_LSTM, 4), (L.CELL_GRU, 1)):
                for sm in (0, L.ATTN_SOFTMAX):
                    d = C.byref(_desc(cell | sm, layers, prec, 1, shape))
                    s = lib.recnet_sample_workspace_bytes(d, 64)
                    assert s > 0
                    if not (prec == L.PREC_BF16 and cell == L.CELL_LSTM and layers == 1):
                        assert s >= lib.recnet_greedy_workspace_bytes(d), (shape, prec, cell, layers, sm)


def test_oracle_noise_is_the_philox_word_of_the_element():
    seed, offset, B, V = 0x1234_5678_9ABC, 7, 3, 11
    for t in (0, 5):
        g = SM.gumbel(seed, offset, t, B, V)
        for row in range(B):
            for v in range(V):
                idx = (t * B + row) * V + v
                words = philox4x32_10(np.array([idx >> 2], dtype=np.uint64), (offset << 8) | 5, seed)
                w = int(words[idx & 3][0])
                u = ((w >> 8) + 0.5) / 2 ** 24
                assert float(g[row, v]) == -np.log(-np.log(u))
    assert torch.isfinite(g).all()


def test_oracle_sampler_at_zero_noise_and_tiny_temperature_is_greedy():
    V, EMB, E, H, A, B, Tn, cap = 13, 8, 16, 8, 8, 9, 5, 12
    for model_name, NL in (("LSTM", 1), ("LSTM", 2), ("GRU", 1)):
        P = O.init_decoder_params(V, EMB, E, H, A, n_layers=NL, model_name=model_name, seed=3, dtype=torch.float64)
        P["out.weight"] = P["out.weight"] * 6
        P["out.bias"][2] += 1.0
        feats = torch.randn(B, Tn, E, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
        ref = O.greedy_search(P, feats, model_name=model_name, n_layers=NL, caption_max_len=cap)
        got = SM.sample(P, feats, max_steps=cap + 1, tau=1e-6, model_name=model_name, n_layers=NL, zero_noise=True)
        fin = 0
        for b in range(B):
            n = int(got["lengths"][b])
            assert torch.equal(got["ids"][:n, b], ref[:n, b]), (model_name, NL, b)
            assert (got["ids"][n:, b] == 0).all()
            fin += n <= cap
        assert fin > 0                                                  # some row finished: the <EOS> rule was exercised
        assert float(got["logp"].abs().max()) < 1e-6                    # tau -> 0: the arg-max carries all the mass


@pytest.mark.parametrize("model_name,n_layers", [("GRU", 2), ("LSTM", L.MAX_LAYERS + 1)])
def test_sample_refuses_a_decoder_without_a_fused_driver(model_name, n_layers):
    dec = recnet_b200.Decoder(model_name, n_layers, 16, 8, 1, 8, 8, 11, 0.5, 0.5, 0.5, precision="fp32")
    assert not dec.uses_fused_sequence
    with pytest.raises(NotImplementedError, match=f"{n_layers}-layer {model_name}"):
        dec.sample(torch.zeros(2, 4, 16), 3, max_steps=5)


class _StubDecoder:
    """What forward_decoder_self_critical needs of a Decoder, with fixed samples: B0 = 2 videos, K = 2 samples each."""

    def __init__(self):
        self.ids = torch.tensor([[5, 2, 7, 3], [2, 0, 4, 2], [0, 0, 2, 0], [0, 0, 0, 0]])     # (max_steps = 4, N = 4)
        self.lengths = torch.tensor([2, 1, 3, 4], dtype=torch.int32)
        self.logp = -torch.rand(4, 4)
        self._rng = torch.tensor([11, 3])
        self.calls = []

    def sample(self, feats, K, *, max_steps, temperature, eos_id):
        self.calls.append(("sample", K, max_steps, temperature, eos_id))
        self._rng[1] += 1
        return self.ids.clone(), self.logp.clone(), self.lengths.clone(), torch.tensor([3], dtype=torch.int32)

    def greedy(self, feats, max_steps):
        self._rng[1] += 100                          # the replay must not see anything that happens to the buffer after sampling
        return torch.tensor([[4, 4], [2, 2]]), torch.tensor([2])

    def _meta(self):
        return {"H": 8}

    def _params(self):
        return (torch.zeros(1),)


def test_self_critical_weights_and_replay_inputs(monkeypatch):
    stub = _StubDecoder()
    seen = {}

    def apply(meta, feats, tokens_in, targets, ce_weight, rng, *params):
        seen.update(meta=meta, feats=feats, tokens_in=tokens_in, targets=targets, ce_weight=ce_weight, rng=rng.clone())
        return torch.tensor(0.5), torch.zeros(tokens_in.shape[0], 1, 4, 8), torch.tensor(1.0)

    monkeypatch.setattr(Fn.DecoderSequenceFn, "apply", apply)
    feats = torch.arange(2 * 3 * 1, dtype=torch.float32).view(2, 3, 1)
    rewards, baseline = torch.tensor([1.0, 4.0, 0.0, 2.0]), torch.tensor([1.5, 1.0])

    def reward_fn(sample_ids, greedy_ids):
        assert sample_ids.shape == (3, 4) and greedy_ids.shape == (2, 2)
        return rewards, baseline

    lam = torch.tensor(0.01)
    loss, hiddens, info = T.forward_decoder_self_critical({"model": stub, "lambda_reg": lam}, feats, reward_fn, n_samples=2,
                                                          temperature=0.7, max_steps=4)
    assert stub.calls == [("sample", 2, 4, 0.7, 2)]
    adv = torch.tensor([-0.5, 3.0, -1.5, 1.0])                          # row k * B0 + b against the baseline of video b
    assert torch.equal(info["advantage"], adv)
    mask = torch.tensor([[1, 1, 1, 1], [1, 0, 1, 1], [0, 0, 1, 1]], dtype=torch.float32)     # t < lengths, n = 3 steps
    assert torch.allclose(seen["ce_weight"], mask * adv / 4)
    assert torch.equal(seen["targets"], stub.ids[:3])
    assert torch.equal(seen["tokens_in"], torch.cat((torch.ones(1, 4, dtype=torch.long), stub.ids[:2])))
    assert torch.equal(seen["rng"], torch.tensor([11, 4]))               # the pair the sampler read
    assert torch.equal(seen["feats"], feats.repeat(2, 1, 1))
    assert seen["meta"]["lambda_reg"] is lam
    assert torch.equal(info["ids"], stub.ids[:3]) and hiddens.shape[0] == 3 and float(loss) == 0.5
