"""GPU checks of CIDEr-D on the device (CiderCorpus.score / recnet_cider_d) against the fp64 oracle of tests/cider_oracle.py, within
1e-4 * max(1, |oracle|):
  * a small-V corpus (dense n-gram collisions) with rows that are exact copies of references, repeated n-grams, 0-3-word captions,
    64-token rows without <EOS>, tokens after <EOS>, a -1 fill and ids near 65535; NaN for ids above 65535 and unknown videos;
  * time-major and batch-major layouts (contiguous and strided views) give the same bits, and two calls give the same bits;
  * 5 x 100 and 1024 rows on an MSVD-shaped corpus (1200 videos x 40 references, V 9000);
  * train.forward_decoder_self_critical with CiderCorpus.reward_fn: rewards and baseline equal the oracle's scores of the sampled and
    greedy ids, the loss is finite and one optimiser step runs."""
import random

import numpy as np
import pytest
import torch

from recnet_b200 import train as T
from recnet_b200.cider import CiderCorpus
from recnet_b200.data import synthetic_captions
from tests import cider_oracle as CO
from tests.test_cider_host import random_refs
from tests.test_gpu_parity import dev
from tests.test_gpu_sample import STEPS, _feats, _model, _params
from tests.test_gpu_stacked import MID

pytestmark = pytest.mark.gpu

BIG = (65535, 65534, 65533)


def _check(scores, ref, what):
    ref = torch.tensor(ref, dtype=torch.float64)
    err = ((scores.double().cpu() - ref).abs() / ref.abs().clamp(min=1.0)).max()
    print(f"[cider] {what}: {scores.numel()} rows, oracle mean {float(ref.mean()):.4f}, max scaled err {float(err):.2e}")
    assert float(err) < 1e-4, (what, float(err))


def _small_corpus():
    refs = random_refs(9, 6, V=10, seed=3, max_len=14)
    refs[4].append([7, 65535, 65534, 7, 65535, 65534, 2])          # ids near the top of the key range
    refs[5].append([65533, 8, 65535, 2, 0, 0])
    return refs


def _small_rows(refs, rnd):
    """(64, N) time-major candidate rows and their videos, covering the cases of the module docstring."""
    rows, vids = [], []

    def add(ids, v):
        rows.append((list(ids) + [0] * 64)[:64])
        vids.append(v)

    for v, rs in enumerate(refs):
        for r in rs:
            add(r, v)                                               # exact copies of references, tails included
        add([], v)
        add([rnd.randint(3, 9)], v)
        add([rnd.randint(3, 9) for _ in range(2)], v)
        add([rnd.randint(3, 9) for _ in range(3)] + [2] + [rnd.randint(3, 9) for _ in range(9)], v)   # tokens after <EOS>
        add([5, 6, 5, 6, 5, 6, 5, 6, 5], v)                          # repeated n-grams
        add([rnd.randint(3, 9) for _ in range(64)], v)              # 64 tokens, no <EOS>
        add([1, 4, 5, 6, 7] + [-1] * 59, v)                         # beam's -1 fill; <SOS> is a word
        add([rnd.choice((7,) + BIG) for _ in range(rnd.randint(4, 40))] + [2], v)
    return torch.tensor(rows, dtype=torch.int64).t().contiguous(), vids


def test_small_vocabulary_against_the_oracle():
    refs = _small_corpus()
    cc, o = CiderCorpus(refs, dev(), vocab_size=65536), CO.Corpus(refs)
    ids, vids = _small_rows(refs, random.Random(5))
    scores = cc.score(ids.to(dev()), vids)
    _check(scores, o.scores(ids.t().tolist(), vids), "small V")
    assert float(scores.max()) > 9.0                                 # some copies of a video's only references score near 10


def test_unkeyable_ids_and_unknown_videos_score_nan():
    refs = _small_corpus()
    cc = CiderCorpus(refs, dev(), vocab_size=65536)
    ids = torch.tensor([[3, 4, 65536, 2], [3, 4, 2, 65536], [3, 4, 5, 2], [3, 4, 5, 2]], dtype=torch.int64).t().contiguous()
    s = cc.score(ids.to(dev()), [0, 0, -1, len(refs)]).cpu()
    assert torch.isnan(s[0]) and not torch.isnan(s[1]) and torch.isnan(s[2]) and torch.isnan(s[3])


def test_layouts_and_repeated_calls_are_bit_identical():
    refs = _small_corpus()
    cc = CiderCorpus(refs, dev(), vocab_size=65536)
    ids, vids = _small_rows(refs, random.Random(6))
    ids = ids.to(dev())
    a = cc.score(ids, vids)
    assert torch.equal(a, cc.score(ids, vids))
    assert torch.equal(a, cc.score(ids.t().contiguous(), vids, layout="batch"))
    assert torch.equal(a, cc.score(ids.t(), vids, layout="batch"))                  # strided view, read in place
    wide = torch.zeros(64, 2 * ids.shape[1], dtype=torch.int64, device=dev())
    wide[:, ::2] = ids
    assert torch.equal(a, cc.score(wide[:, ::2], vids))                               # row stride 2


@pytest.fixture(scope="module")
def msvd():
    refs = synthetic_captions(1200, 40, 9000, seed=11)
    return refs, CiderCorpus(refs, dev()), CO.Corpus(refs)


def _msvd_rows(refs, n, seed):
    """Candidates of an MSVD-shaped batch: a third copies of references, a third references with words swapped, a third Zipf captions
    of other videos; time-major (31, n)."""
    rng = np.random.default_rng(seed)
    vids = rng.integers(0, len(refs), size=n)
    rows = np.zeros((n, 31), dtype=np.int64)
    for i, v in enumerate(vids):
        r = refs[v][rng.integers(0, len(refs[v]))].copy()
        if i % 3 == 1:
            r[: len(r) - 1][rng.random(len(r) - 1) < 0.3] = rng.integers(3, 9000)
        elif i % 3 == 2:
            w = refs[(v + 1) % len(refs)][0]
            r = w
        rows[i, : min(len(r), 31)] = r[:31]
    return torch.from_numpy(rows).t().contiguous(), vids.tolist()


@pytest.mark.parametrize("n", [500, 1024])
def test_msvd_shape_against_the_oracle(msvd, n):
    refs, cc, o = msvd
    ids, vids = _msvd_rows(refs, n, seed=n)
    s = cc.score(ids.to(dev()), vids)
    _check(s, o.scores(ids.t().tolist(), vids), f"MSVD shape, {n} rows")
    assert torch.equal(s, cc.score(ids.to(dev()), vids))


def test_self_critical_training_with_the_cider_reward():
    P = _params("LSTM", 1, eos_boost=0.0)       # <EOS> not lifted: greedy captions are not empty, so baselines are not all 0
    dec, model = _model("LSTM", 1, False, "fp32", True, P)
    B0 = MID["B"]
    # references drawn from the decoder's own greedy and sampled captions, mixed with random ones, so that the rewards spread
    feats = _feats().float().to(dev())
    g = model.greedy(feats, STEPS)[0].cpu()
    s = model.sample(feats, 2, max_steps=STEPS, seed=9)[0].cpu()
    rnd = random.Random(2)
    refs = [[[rnd.randint(3, MID["V"] - 1) for _ in range(rnd.randint(3, 12))] + [2] for _ in range(3)] for _ in range(2 * B0)]
    video_idx = list(range(2 * B0 - 1, B0 - 1, -1))                  # batch item b is corpus video 2 B0 - 1 - b
    for b, v in enumerate(video_idx):
        refs[v] += [g[:, b].tolist(), s[:, b].tolist()[:6] + [2]]
    cc, o = CiderCorpus(refs, dev(), vocab_size=MID["V"]), CO.Corpus(refs)
    K = 5
    torch.manual_seed(11)
    loss, _, info = T.forward_decoder_self_critical(dec, feats, cc.reward_fn(cc.index(video_idx)), n_samples=K, max_steps=STEPS)
    greedy = model.greedy(feats, STEPS)[0].cpu()
    ids = info["ids"].cpu()
    _check(info["rewards"], o.scores(ids.t().tolist(), [video_idx[r % B0] for r in range(K * B0)]), "SCST rewards")
    _check(info["baseline"], o.scores(greedy.t().tolist(), video_idx), "SCST baseline")
    assert float(info["baseline"].max()) > 0 and float(info["advantage"].abs().max()) > 0
    assert torch.isfinite(loss)
    before = [p.detach().clone() for p in model.parameters()]
    dec["optimizer"].zero_grad(set_to_none=True)
    loss.backward()
    dec["optimizer"].step()
    assert any(not torch.equal(a, p.detach()) for a, p in zip(before, model.parameters()))
