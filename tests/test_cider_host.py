"""CPU checks of CIDEr-D: the fp64 oracle (tests/cider_oracle.py) on hand-worked cases, the host build of recnet_b200.cider.CiderCorpus
against the oracle (document frequencies, ref_len, weights, norms, lengths, key order, the strip rule), its refusals, ``index`` with
'PAD', the row -> video assignment of ``reward_fn``, and the refusals of recnet_cider_d before any launch (null buffers, no GPU)."""
import ctypes as C
import math
import random

import numpy as np
import pytest
import torch

from recnet_b200 import _lib as L
from recnet_b200.cider import CiderCorpus
from tests import cider_oracle as CO

BAD_SHAPE, UNSUPPORTED = -1, -4
LN2 = math.log(2.0)


def random_refs(n_videos, n_refs, V, seed, max_len=12):
    """Small-V references (dense n-gram collisions), with <EOS>/<PAD> tails, tokens after <EOS>, -1 fills and empty references."""
    rnd = random.Random(seed)
    refs = []
    for _ in range(n_videos):
        rs = []
        for _ in range(rnd.randint(1, n_refs)):
            words = [rnd.randint(1, V - 1) for _ in range(rnd.randint(0, max_len))]
            words = [w if w != 2 else 3 for w in words]
            tail = rnd.choice([[], [2], [2, 0, 0], [2, 7, 8], [0, 5], [-1, -1]])
            rs.append(words + tail)
        refs.append(rs)
    return refs


# ---- the oracle on hand-worked cases ----------------------------------------------------------------------------------------------
def test_oracle_copy_of_the_only_reference_scores_ten():
    o = CO.Corpus([[[3, 4, 5, 6, 7, 2]], [[8, 9, 10, 11]]])
    assert abs(o.score([3, 4, 5, 6, 7, 2, 0], 0) - 10.0) < 1e-12
    assert abs(o.score([8, 9, 10, 11], 1) - 10.0) < 1e-12


def test_oracle_clips_a_repeated_ngram():
    o = CO.Corpus([[[5, 6]], [[7, 8]]])
    # hyp unigram 5 twice: w_h = 2 ln2, w_r = ln2 -> min(w_h, w_r) * w_r = ln2^2 over |h1| |r1| = 2 ln2 * sqrt(2) ln2; bigram (5, 5) absent
    assert abs(o.score([5, 5], 0) - 10.0 / 4 / (2 * math.sqrt(2))) < 1e-12


def test_oracle_length_penalty():
    o = CO.Corpus([[[3, 4, 5, 6, 7, 8, 9]], [[10]]])
    # every hyp n-gram is in the reference with weight ln2: val_n = sqrt(c_h / c_r); bigram lengths 3 and 6
    pen = math.exp(-(3 ** 2) / 72.0)
    want = 10.0 / 4 * pen * sum(math.sqrt(h / r) for h, r in zip((4, 3, 2, 1), (7, 6, 5, 4)))
    assert abs(o.score([3, 4, 5, 6], 0) - want) < 1e-12


def test_oracle_ngram_in_every_video_weighs_nothing():
    o = CO.Corpus([[[3, 4]], [[3, 5]]])
    vec, norm, _ = o.counts2vec(CO.precook((3, 4)))
    assert vec[0][(3,)] == 0.0 and vec[0][(4,)] == LN2 and vec[1][(3, 4)] == LN2
    assert o.score([3], 0) == 0.0
    assert abs(o.score([3, 4], 0) - 5.0) < 1e-12


def test_oracle_empty_candidate_and_single_video_corpus_score_zero():
    o = CO.Corpus([[[3, 4, 5]], [[6, 7]]])
    assert o.score([], 0) == 0.0 and o.score([2, 3, 4], 0) == 0.0 and o.score([0, 3], 1) == 0.0
    one = CO.Corpus([[[3, 4, 5, 6], [3, 4]]])
    assert one.ref_len == 0.0 and one.score([3, 4, 5, 6], 0) == 0.0


# ---- the host build against the oracle -------------------------------------------------------------------------------------------
def _decode(key):
    return tuple(g for g in ((int(key) >> s) & 0xFFFF for s in (48, 32, 16, 0)) if g)


@pytest.mark.parametrize("seed", [0, 1])
def test_build_matches_the_oracle(seed):
    refs = random_refs(7, 5, V=9, seed=seed)
    cc, o = CiderCorpus(refs, "cpu"), CO.Corpus(refs)
    assert cc.ref_len == o.ref_len
    assert {_decode(k): int(d) for k, d in zip(cc.df_keys, cc.df)} == {g: int(d) for g, d in o.df.items()}
    t = cc.tensors
    assert torch.equal(t["df_log"], torch.tensor([math.log(max(1.0, o.df[_decode(k)])) for k in cc.df_keys], dtype=torch.float32))
    r = 0
    for v, crefs in enumerate(o.crefs):
        assert list(range(int(t["video_refs"][v]), int(t["video_refs"][v + 1]))) == list(range(r, r + len(crefs)))
        for cnts in crefs:
            vec, norm, length = o.counts2vec(cnts)
            e0, e1 = int(t["ref_entries"][r]), int(t["ref_entries"][r + 1])
            got = {_decode(k): float(w) for k, w in zip(cc.entry_keys[e0:e1], t["entry_w"][e0:e1])}
            want = {g: w for n in range(4) for g, w in vec[n].items()}
            assert got.keys() == want.keys()
            for g in want:
                assert got[g] == float(np.float32(want[g])), g
            np.testing.assert_allclose(t["ref_norm"][r].double().numpy(), norm, rtol=1e-6, atol=0)
            np.testing.assert_allclose(cc.ref_norm[r], norm, rtol=1e-12, atol=0)
            assert int(t["ref_length"][r]) == length
            r += 1
    assert r == len(cc.ref_length)


def test_key_order_and_strip_rule():
    refs = [[[70, 5, 65535, 2, 9, 9], [5, 70, -1, 4], [1, 2], []], [[65535, 5, 0, 3]]]
    cc = CiderCorpus(refs, "cpu")
    # keys: id_j << (64 - 16 j); the order is implied by the zero padding
    assert int(cc.entry_keys[0]) == 5 << 48
    assert {_decode(k) for k in cc.df_keys} == {(70,), (5,), (65535,), (70, 5), (5, 65535), (70, 5, 65535), (5, 70), (1,),
                                               (65535, 5)}
    keys = [int(k) for k in cc.df_keys]
    assert keys == sorted(keys) and len(set(keys)) == len(keys)
    for r in range(len(cc.ref_length)):
        e = [int(k) for k in cc.entry_keys[cc.ref_entries[r]:cc.ref_entries[r + 1]]]
        assert e == sorted(e) and len(set(e)) == len(e)
    assert cc.ref_length.tolist() == [2, 1, 0, 0, 1]                # bigram counts of the stripped references
    assert cc.video_refs.tolist() == [0, 4, 5] and cc.ref_entries[3] == cc.ref_entries[4]   # the empty reference has no entries
    assert cc.tensors["entry_keys"].dtype == torch.int64 and int(cc.tensors["df_keys"][keys.index(65535 << 48)]) < 0


def test_build_refusals():
    with pytest.raises(ValueError, match="no videos"):
        CiderCorpus([], "cpu")
    with pytest.raises(ValueError, match="no references"):
        CiderCorpus({"a": [[3, 4]], "b": []}, "cpu")
    with pytest.raises(ValueError, match="65536"):
        CiderCorpus([[[3, 4]]], "cpu", vocab_size=65537)
    with pytest.raises(ValueError, match="65536"):
        CiderCorpus([[[3, 65536]]], "cpu")
    CiderCorpus([[[3, 65535]]], "cpu", vocab_size=65536)


def test_index_maps_clip_ids_and_pad():
    cc = CiderCorpus({"v0_1_2": [[3]], "v1_0_5": [[4]], "v2_3_4": [[5]]}, "cpu")
    assert cc.index(["v2_3_4", "v0_1_2", "PAD", "PAD"]).tolist() == [2, 0, 0, 0]
    assert cc.index(["v1_0_5"]).dtype == torch.int32
    with pytest.raises(ValueError):
        cc.index(["PAD", "v0_1_2"])
    with pytest.raises(KeyError):
        cc.index(["nope"])


def test_from_dataset_groups_captions_by_clip():
    from recnet_b200 import data as D

    class DS:
        vocab = D.Vocabulary(["a man runs.", "A dog runs", "a cat"], caption_max_len=30)
        pairs = [("c1", None, "a man runs."), ("c2", None, "a cat"), ("c1", None, "A dog runs, fast")]

    cc = CiderCorpus.from_dataset(DS(), "cpu")
    w = DS.vocab.word2idx
    o = CO.Corpus([[[w["a"], w["man"], w["runs"]], [w["a"], w["dog"], w["runs"]]], [[w["a"], w["cat"]]]])
    assert cc.vids == ["c1", "c2"] and cc.vocab_size == DS.vocab.n_vocabs and cc.ref_len == o.ref_len
    assert cc.video_refs.tolist() == [0, 2, 3] and cc.ref_length.tolist() == [2, 2, 1]


def test_reward_fn_assigns_sample_rows_to_videos():
    cc = CiderCorpus([[[3]], [[4]], [[5]]], "cpu")
    seen = []

    def stub(ids, video_idx, eos_id=2, layout="time"):
        seen.append((ids.shape, video_idx.tolist(), eos_id, layout))
        return torch.full((ids.shape[1],), float(len(seen)))

    cc.score = stub
    fn = cc.reward_fn(cc.index([2, 0]))
    rewards, baseline = fn(torch.zeros(7, 6, dtype=torch.long), torch.zeros(9, 2, dtype=torch.long))
    assert seen == [((7, 6), [2, 0, 2, 0, 2, 0], 2, "time"), ((9, 2), [2, 0], 2, "time")]
    assert rewards.tolist() == [1.0] * 6 and baseline.tolist() == [2.0] * 2
    with pytest.raises(RuntimeError):
        fn(torch.zeros(7, 5, dtype=torch.long), torch.zeros(9, 2, dtype=torch.long))


def test_score_needs_the_device():
    cc = CiderCorpus([[[3]]], "cpu")
    with pytest.raises(RuntimeError, match="device"):
        cc.score(torch.zeros(4, 2, dtype=torch.long), [0, 0])


# ---- ABI refusals before any launch ----------------------------------------------------------------------------------------------
def test_abi_refusals():
    lib = L.lib()
    call = lambda c, steps, rows: lib.recnet_cider_d(c, None, 1, 1, steps, rows, None, 2, None, None)
    ok = L.cider_corpus(n_videos=3, n_df=0, vocab=65536, ref_len=1.0)
    for steps, rows in ((0, 4), (65, 4), (-1, 4), (31, 0), (31, -3)):
        assert call(C.byref(ok), steps, rows) == BAD_SHAPE, (steps, rows)
    assert call(None, 31, 4) == BAD_SHAPE
    assert call(C.byref(L.cider_corpus(n_videos=0, vocab=10)), 31, 4) == BAD_SHAPE
    assert call(C.byref(L.cider_corpus(n_videos=3, vocab=65537)), 31, 4) == UNSUPPORTED
    assert call(C.byref(L.cider_corpus(n_videos=3, vocab=65537)), 64, 1) == UNSUPPORTED
