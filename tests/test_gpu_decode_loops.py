"""Kernel launches of one device decode call, read with recnet_launch_count: greedy, beam search (width 3) and sampling (eval and train
mode) of LSTM decoders with 1, 2 and 4 layers and of a single-layer GRU, in fp32 and bf16, and the same four calls of a softmax-attention
decoder.  A call launches a fixed set of kernels whatever tokens it decodes (a finished loop freezes on the device), so every count is
exact.  The bf16 single-layer LSTM greedy call runs on the projected-feature kernels, every other call on the general step path."""
import pytest
import torch

import recnet_b200
from recnet_b200 import _lib as L

pytestmark = pytest.mark.gpu

SHAPE = dict(B=8, T=5, E=32, H=16, A=16, EMB=16, V=23)
STEPS = 7
CONFIGS = [("LSTM", 1, False), ("LSTM", 2, False), ("LSTM", 4, False), ("GRU", 1, False), ("LSTM", 1, True)]

# launches per call: (precision, cell, n_layers, softmax) -> {greedy, beam, sample_eval, sample_train}
COUNTS = {
    ("fp32", "LSTM", 1, False): dict(greedy=65, beam=73, sample_eval=65, sample_train=65),
    ("fp32", "LSTM", 2, False): dict(greedy=81, beam=89, sample_eval=81, sample_train=81),
    ("fp32", "LSTM", 4, False): dict(greedy=113, beam=121, sample_eval=113, sample_train=113),
    ("fp32", "GRU", 1, False): dict(greedy=71, beam=79, sample_eval=71, sample_train=71),
    ("fp32", "LSTM", 1, True): dict(greedy=65, beam=73, sample_eval=65, sample_train=65),
    ("bf16", "LSTM", 1, False): dict(greedy=35, beam=73, sample_eval=65, sample_train=65),
    ("bf16", "LSTM", 2, False): dict(greedy=81, beam=89, sample_eval=81, sample_train=81),
    ("bf16", "LSTM", 4, False): dict(greedy=113, beam=121, sample_eval=113, sample_train=113),
    ("bf16", "GRU", 1, False): dict(greedy=71, beam=79, sample_eval=71, sample_train=71),
    ("bf16", "LSTM", 1, True): dict(greedy=65, beam=73, sample_eval=65, sample_train=65),
}


def launch_counts(precision, cell, n_layers, softmax):
    s = SHAPE
    torch.manual_seed(0)
    dec = recnet_b200.Decoder(cell, n_layers, s["E"], s["EMB"], 1.0, s["H"], s["A"], s["V"], 0.5, 0.5, 0.5, precision=precision,
                              attn_softmax=softmax).cuda()
    feats = torch.randn(s["B"], s["T"], s["E"], generator=torch.Generator().manual_seed(1)).cuda()
    calls = {"greedy": lambda: dec.eval().greedy(feats, STEPS), "beam": lambda: dec.eval().beam(feats, 3, STEPS),
             "sample_eval": lambda: dec.eval().sample(feats, max_steps=STEPS, seed=2),
             "sample_train": lambda: dec.train().sample(feats, max_steps=STEPS, seed=2)}
    lib, got = L.lib(), {}
    for mode, call in calls.items():
        n0 = lib.recnet_launch_count()
        call()
        got[mode] = lib.recnet_launch_count() - n0
    torch.cuda.synchronize()
    return got


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("cell,n_layers,softmax", CONFIGS)
def test_launches_per_decode_call(precision, cell, n_layers, softmax):
    assert launch_counts(precision, cell, n_layers, softmax) == COUNTS[precision, cell, n_layers, softmax]
