"""CIDEr-D on vocabulary ids, scored on the device: a validation metric and the self-critical reward.

The score is coco-caption's ``CiderD`` (n = 1..4, sigma = 6) with document frequencies taken from the corpus scored against
(coco-caption's "corpus" mode): for SCST the training split, for validation the validation split.  It works on vocabulary ids, so
punctuation stripping, lower-casing, truncation to ``caption_max_len`` and the dropping of unknown words are those of
``Vocabulary.encode``; it is therefore not the score coco-caption computes on raw text after the PTB tokenizer.

The caption of a row of ids is the ids before the first ``<EOS>``, ``<PAD>`` (0) or negative id (``Decoder.beam`` fills with -1, and
greedy decoding keeps emitting tokens after ``<EOS>``).  References are stripped by the same rule; every other id, ``<SOS>``
included, is a word.

``CiderCorpus`` builds the reference side once on the host in float64 (document frequencies, per-reference n-gram weights and
norms) and uploads it; ``score`` is one kernel launch (``recnet_cider_d``), one warp per candidate row."""
import ctypes as C
import math
from collections.abc import Mapping

import numpy as np
import torch

from . import _lib as L
from . import functional as Fn

MAX_VOCAB = 1 << 16            # ids are packed 16 bits apiece into a uint64 key per n-gram: sum_j a_j << (64 - 16 j)
N_ORDER = 4


def strip(ids, eos_id=2):
    """The caption of a sequence of ids: the ids before the first eos_id, <PAD> (0) or negative id, as a list of ints."""
    out = []
    for v in ids:
        v = int(v)
        if v == eos_id or v <= 0:
            break
        out.append(v)
    return out


class CiderCorpus:
    """The references of a corpus, ready for ``score``.

    ``refs`` maps clip ids to lists of reference id sequences (lists, tuples or 1-D tensors); a plain sequence of such lists is taken
    as clip ids 0, 1, ....  ``vocab_size`` defaults to the largest reference id + 1; it may not exceed 65536.  The build raises
    ``ValueError`` for an empty corpus, a video without references and a vocabulary over 65536 ids.  A reference may be empty (every
    word unknown): it still counts in its video's divisor.

    Host arrays (numpy, kept for inspection): ``df_keys`` (uint64, ascending) and ``df`` (video counts), ``video_refs`` /
    ``ref_entries`` (CSR offsets), ``entry_keys`` (uint64, ascending within a reference), ``entry_w`` (float64 weights
    count * (ref_len - log max(1, df))), ``ref_norm`` (float64 (n_refs, 4)), ``ref_length`` (bigram counts) and ``ref_len`` =
    log(number of videos).  Their fp32 copies live on ``device``."""

    def __init__(self, refs, device, vocab_size=None, eos_id=2):
        if isinstance(refs, Mapping):
            vids, refs = list(refs.keys()), list(refs.values())
        else:
            refs = list(refs)
            vids = list(range(len(refs)))
        if not refs:
            raise ValueError("CiderCorpus: the corpus has no videos")
        caps, video_of_ref = [], []
        for v, rs in enumerate(refs):
            rs = list(rs)
            if not rs:
                raise ValueError(f"CiderCorpus: video {vids[v]!r} has no references")
            for r in rs:
                caps.append(strip(r.tolist() if torch.is_tensor(r) else r, eos_id))
                video_of_ref.append(v)
        top = max((max(c) for c in caps if c), default=0)
        self.vocab_size = int(vocab_size) if vocab_size is not None else top + 1
        if self.vocab_size > MAX_VOCAB or top >= MAX_VOCAB:
            raise ValueError(f"CiderCorpus: a vocabulary of {max(self.vocab_size, top + 1)} ids; n-gram keys hold ids below {MAX_VOCAB}")
        self.vids = vids
        self._row = {vid: i for i, vid in enumerate(vids)}
        self.eos_id = int(eos_id)
        self._build_host(caps, np.asarray(video_of_ref, dtype=np.int64), len(refs))
        self.device = torch.device(device)
        self._upload()

    @classmethod
    def from_dataset(cls, dataset, device, eos_id=2):
        """The references of a ``data.CaptionFeatureDataset``: its captions grouped by clip id (in the dataset's clip order) and
        encoded with ``dataset.vocab.encode``."""
        refs = {}
        for vid, _, caption in dataset.pairs:
            refs.setdefault(vid, []).append(dataset.vocab.encode(caption))
        return cls(refs, device, vocab_size=dataset.vocab.n_vocabs, eos_id=eos_id)

    def index(self, vids):
        """Video rows of clip ids, as an int32 tensor on the corpus' device.  A 'PAD' clip id (``data.collate``'s padding of a short
        last batch) takes the row of the item before it, whose features it copies."""
        rows = []
        for vid in vids:
            if vid == "PAD":
                if not rows:
                    raise ValueError("CiderCorpus.index: a 'PAD' clip id with no item before it")
                rows.append(rows[-1])
            else:
                rows.append(self._row[vid])
        return torch.tensor(rows, dtype=torch.int32, device=self.device)

    # ---- host build (float64) ----
    def _build_host(self, caps, video_of_ref, n_videos):
        n_refs = len(caps)
        lens = np.array([len(c) for c in caps], dtype=np.int64)
        width = max(int(lens.max()), 1)
        ids = np.zeros((n_refs, width), dtype=np.uint64)
        for r, c in enumerate(caps):
            ids[r, : len(c)] = c
        ref_of, keys = [], []
        for n in range(N_ORDER):
            for i in range(width - n):
                valid = np.nonzero(lens >= i + n + 1)[0]
                if valid.size == 0:
                    break
                k = np.zeros(valid.size, dtype=np.uint64)
                for q in range(n + 1):
                    k |= ids[valid, i + q] << np.uint64(48 - 16 * q)
                ref_of.append(valid)
                keys.append(k)
        ref_of = np.concatenate(ref_of) if ref_of else np.zeros(0, dtype=np.int64)
        keys = np.concatenate(keys) if keys else np.zeros(0, dtype=np.uint64)
        # (reference, n-gram) pairs with their counts, sorted by reference then key
        o = np.lexsort((keys, ref_of))
        ref_of, keys = ref_of[o], keys[o]
        new = np.ones(keys.size, dtype=bool)
        new[1:] = (ref_of[1:] != ref_of[:-1]) | (keys[1:] != keys[:-1])
        starts = np.nonzero(new)[0]
        counts = np.diff(np.append(starts, keys.size))
        e_ref, e_key = ref_of[starts], keys[starts]
        # document frequency: videos whose references contain the n-gram
        e_vid = video_of_ref[e_ref]
        o = np.lexsort((e_vid, e_key))
        k2, v2 = e_key[o], e_vid[o]
        first = np.ones(k2.size, dtype=bool)
        first[1:] = (k2[1:] != k2[:-1]) | (v2[1:] != v2[:-1])
        k2 = k2[first]
        df_keys, df = np.unique(k2, return_counts=True)
        self.ref_len = math.log(float(n_videos))
        lg = np.log(np.maximum(1.0, df.astype(np.float64)))
        w = counts.astype(np.float64) * (self.ref_len - lg[np.searchsorted(df_keys, e_key)])
        order = N_ORDER - sum(((e_key >> np.uint64(s)) & np.uint64(0xFFFF) == 0).astype(np.int64) for s in (0, 16, 32))
        norm = np.zeros(n_refs * N_ORDER)
        np.add.at(norm, e_ref * N_ORDER + order - 1, w * w)
        self.df_keys, self.df, self.df_log = df_keys, df, lg
        self.video_refs = np.concatenate(([0], np.cumsum(np.bincount(video_of_ref, minlength=n_videos)))).astype(np.int32)
        self.ref_entries = np.concatenate(([0], np.cumsum(np.bincount(e_ref, minlength=n_refs)))).astype(np.int32)
        self.entry_keys, self.entry_w = e_key, w
        self.ref_norm = np.sqrt(norm).reshape(n_refs, N_ORDER)
        self.ref_length = np.maximum(lens - 1, 0).astype(np.int32)
        self.n_videos = n_videos

    def _upload(self):
        dev = self.device
        keys = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64)).to(dev)
        f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
        i32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev)
        self.tensors = {"df_keys": keys(self.df_keys), "df_log": f32(self.df_log), "video_refs": i32(self.video_refs),
                        "ref_entries": i32(self.ref_entries), "entry_keys": keys(self.entry_keys), "entry_w": f32(self.entry_w),
                        "ref_norm": f32(self.ref_norm), "ref_length": i32(self.ref_length)}
        self._desc = L.cider_corpus(n_videos=self.n_videos, n_df=int(self.df_keys.size), vocab=self.vocab_size, ref_len=self.ref_len,
                                    **{k: v.data_ptr() for k, v in self.tensors.items()})

    # ---- scoring ----
    def score(self, ids, video_idx, eos_id=2, layout="time"):
        """CIDEr-D of every row of ``ids`` (int64, on the corpus' device) against the references of video ``video_idx[row]``
        (rows as given by ``index``): a (rows,) float32 tensor on the device.  ``layout="time"``: ids is (steps, N), the layout of
        ``Decoder.sample`` / ``Decoder.greedy``; ``"batch"``: (N, steps), the layout of ``Decoder.beam``.  Strided views are read in
        place; steps <= 64.  A row whose caption holds an id above 65535 scores NaN.  The mean over rows is the corpus CIDEr-D."""
        if layout not in ("time", "batch"):
            raise ValueError(f"CiderCorpus.score: layout must be 'time' or 'batch', not {layout!r}")
        if self.device.type != "cuda" or not ids.is_cuda:
            raise RuntimeError("CiderCorpus.score runs on the device only: the corpus and ids must be CUDA tensors")
        if ids.dtype != torch.int64 or ids.dim() != 2:
            raise RuntimeError(f"CiderCorpus.score: ids must be a 2-D int64 tensor, got {ids.dtype} {tuple(ids.shape)}")
        steps, n = ids.shape if layout == "time" else ids.shape[::-1]
        ld_step, ld_row = ids.stride() if layout == "time" else ids.stride()[::-1]
        vidx = torch.as_tensor(video_idx, device=ids.device).to(torch.int32).contiguous()
        if vidx.shape != (n,):
            raise RuntimeError(f"CiderCorpus.score: {n} rows but video_idx has shape {tuple(vidx.shape)}")
        out = torch.empty(n, dtype=torch.float32, device=ids.device)
        L.check(L.lib().recnet_cider_d(C.byref(self._desc), ids.data_ptr(), ld_step, ld_row, steps, n, vidx.data_ptr(), int(eos_id),
                                       out.data_ptr(), Fn._stream()), "recnet_cider_d")
        return out

    def reward_fn(self, video_idx, eos_id=2):
        """The reward of ``train.forward_decoder_self_critical``: ``(sample_ids (n, K*B0), greedy_ids (L, B0)) -> (rewards (K*B0,),
        baseline (B0,))``, the CIDEr-D of every sample and of every greedy caption.  Sample row r belongs to video
        ``video_idx[r % B0]``, as ``Decoder.sample`` tiles its rows.  Two ``score`` calls, no host read."""
        video_idx = torch.as_tensor(video_idx, device=self.device).to(torch.int32)
        B0 = video_idx.shape[0]

        def reward(sample_ids, greedy_ids):
            N = sample_ids.shape[1]
            if N % B0 or greedy_ids.shape[1] != B0:
                raise RuntimeError(f"CiderCorpus.reward_fn: {N} sample rows and {greedy_ids.shape[1]} greedy rows for {B0} videos")
            return self.score(sample_ids, video_idx.repeat(N // B0), eos_id), self.score(greedy_ids, video_idx, eos_id)

        return reward
