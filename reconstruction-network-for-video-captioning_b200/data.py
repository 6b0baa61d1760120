"""Inputs of the hot path.

* ``synthetic_batch``: synthetic MSVD-shaped batches (SURVEY.md section 8d) -- what bench.py and the parity tests use.
* the real-data adapter below it (SURVEY.md section 8f item 4): the reference's vocabulary / caption / frame-sampling / collate
  pipeline (dataset/MSVD.py, dataset/transform.py) restated, so real features + captions can feed the same drivers.

Both produce tensors of exactly the shapes and value conventions the reference's loader does: feats (B, T, E) fp32;
targets (caption_max_len + 1, B) int64 = word ids, then <EOS>=2, then <PAD>=0 (no <SOS> inside targets,
dataset/MSVD.py:111-117); masks = targets > 0 (train.py:246)."""
import math
import re
import string

import numpy as np
import torch
import torch.utils.data

PAD, SOS, EOS = 0, 1, 2


def synthetic_batch(B, T, E, V, caption_max_len=30, seed=1234, full_length_first=True):
    g = torch.Generator().manual_seed(seed)
    feats = torch.randn(B, T, E, generator=g, dtype=torch.float32)
    lens = torch.randint(min(3, caption_max_len), caption_max_len + 1, (B,), generator=g)
    if full_length_first:
        lens[0] = caption_max_len          # => L = caption_max_len + 1 decoded steps every iteration (fixed work)
    targets = torch.zeros(caption_max_len + 1, B, dtype=torch.long)
    for b in range(B):
        n = int(lens[b])
        targets[:n, b] = torch.randint(3, V, (n,), generator=g)
        targets[n, b] = EOS
    return feats, targets, targets > PAD


def synthetic_captions(n_videos, n_refs, V, seed, min_len=3, max_len=30, zipf=1.0):
    """Seeded MSVD-shaped reference captions for CIDEr-D: ``n_refs`` per video, lengths uniform in [min_len, max_len], word ids 3..V-1
    drawn with Zipf weights 1 / rank^zipf (frequent words recur across videos, as in real captions), each ended by <EOS>.
    Returns refs[video][ref] = int64 numpy array."""
    rng = np.random.default_rng(seed)
    p = 1.0 / np.arange(1, V - 2, dtype=np.float64) ** zipf
    p /= p.sum()
    lens = rng.integers(min_len, max_len + 1, size=(n_videos, n_refs))
    words = rng.choice(np.arange(3, V, dtype=np.int64), size=int(lens.sum()), p=p)
    refs, k = [], 0
    for v in range(n_videos):
        rs = []
        for n in lens[v]:
            rs.append(np.append(words[k:k + n], EOS))
            k += n
        refs.append(rs)
    return refs


def shard_range(n_items: int, rank: int, world: int):
    """Contiguous shard [lo, hi) of n_items for `rank` of `world` (remainder spread over the first ranks)."""
    base, rem = divmod(n_items, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


# ------------------------------------------------------------------------------------------------------------------
# Real-data adapter (SURVEY.md section 8f, item 4): the reference's caption / frame pipeline restated so that real MSVD
# (or MSR-VTT) features + captions can replace the synthetic generator in front of the same hot path.  Host-side only:
# everything here produces the (B, T, E) float32 features and (caption_max_len + 1, B) int64 targets the sequence drivers take.
# ------------------------------------------------------------------------------------------------------------------
_PUNCT = re.compile('[%s]' % re.escape(string.punctuation))


def sentence_to_words(sentence, caption_max_len):
    """dataset/MSVD.py:31-37 (transform_sentence): drop non-ASCII characters (TrimExceptAscii), remove punctuation, lowercase,
    split on white space, truncate to caption_max_len words (dataset/transform.py:79-110)."""
    if isinstance(sentence, bytes):
        sentence = sentence.decode('ascii', 'ignore')
    sentence = sentence.encode('ascii', 'ignore').decode('ascii')
    return _PUNCT.sub('', sentence).lower().split()[:caption_max_len]


class Vocabulary:
    """dataset/MSVD.py:165-207 (MSVDVocab): word -> id in first-seen order after the initial tokens, words seen fewer than
    ``min_count`` times dropped (there is no <UNK>: unknown words are skipped when a caption is indexed)."""

    def __init__(self, captions, init_word2idx=None, min_count=1, caption_max_len=30):
        self.min_count, self.caption_max_len = min_count, caption_max_len
        self.word2idx = dict(init_word2idx if init_word2idx is not None else {'<PAD>': PAD, '<SOS>': SOS, '<EOS>': EOS})
        self.idx2word = {v: k for k, v in self.word2idx.items()}
        self.word_freq_dict = {}
        self.max_sentence_len = -1
        for caption in captions:
            words = sentence_to_words(caption, caption_max_len)
            self.max_sentence_len = max(self.max_sentence_len, len(words))
            for w in words:
                self.word_freq_dict[w] = self.word_freq_dict.get(w, 0) + 1
        self.n_vocabs_untrimmed = len(self.word_freq_dict)
        self.n_words_untrimmed = sum(self.word_freq_dict.values())
        keep = [w for w, f in self.word_freq_dict.items() if f >= min_count]          # dict order = first-seen order (MSVD.py:199)
        for idx, w in enumerate(keep, len(self.word2idx)):
            self.word2idx[w] = idx
            self.idx2word[idx] = w
        self.n_vocabs = len(self.word2idx)
        self.n_words = sum(self.word_freq_dict[w] for w in keep)

    @classmethod
    def from_csv(cls, caption_fpath, **kw):
        """MSVD.py:181-186: rows with Language == 'English' and a non-null Description."""
        return cls(_read_caption_table(caption_fpath)['Description'].values, **kw)

    def encode(self, caption):
        """transform_caption (MSVD.py:107-113): words -> known ids, + <EOS>, padded with <PAD> to max_sentence_len + 1."""
        ids = [self.word2idx[w] for w in sentence_to_words(caption, self.caption_max_len) if w in self.word2idx]
        ids.append(self.word2idx['<EOS>'])
        ids += [self.word2idx['<PAD>']] * (self.max_sentence_len + 1 - len(ids))
        return torch.tensor(ids, dtype=torch.long)

    def decode(self, ids):
        """ids -> sentence up to (not including) the first <EOS> / <PAD> (what eval.py prints)."""
        words = []
        for i in ids:
            i = int(i)
            if i in (self.word2idx['<EOS>'], self.word2idx['<PAD>']):
                break
            words.append(self.idx2word.get(i, ''))
        return ' '.join(w for w in words if w)


def _read_caption_table(caption_fpath):
    import pandas as pd
    df = pd.read_csv(caption_fpath)
    df = df[df['Language'] == 'English']
    return df[pd.notnull(df['Description'])]


def sample_frames(frames, n_sample, method="uniform", rng=None):
    """dataset/transform.py:9-62 + MSVD.py:100-104: pick ``n_sample`` of the n frame features (``uniform``: linspace indices;
    ``random``: a sorted random subset; ``uniform_jitter``: linspace + N(0, int(sqrt(n / n_sample / 4))) jitter, clipped, sorted),
    keep all of them when there are fewer, zero-pad to ``n_sample``; returns a float32 (n_sample, E) tensor.
    ``rng``: object with numpy.random's ``choice`` / ``normal`` (default: numpy.random, i.e. the reference's global generator)."""
    rng = np.random if rng is None else rng
    frames = np.asarray(frames)
    n = len(frames)
    if n >= n_sample:
        if method == "uniform":
            idx = [int(i) for i in np.linspace(0, n - 1, n_sample)]
        elif method == "random":
            idx = sorted(rng.choice(n, n_sample, replace=False))
        elif method == "uniform_jitter":
            std = int(math.sqrt(n / n_sample / 2 / 2))
            idx = [int(i) for i in np.linspace(0, n - 1, n_sample)]
            idx = [int(i + rng.normal(0, std)) for i in idx]
            idx = sorted(min(max(0, i), n - 1) for i in idx)
        else:
            raise NotImplementedError("Unknown frame sampling method: {}".format(method))          # MSVD.py:98
        frames = frames[idx]
    out = np.zeros((n_sample,) + frames.shape[1:], dtype=np.float32)
    out[: len(frames)] = frames
    return torch.from_numpy(out)


def load_features(video_fpath):
    """vid -> (n_frames, E) array from an HDF5 file (the reference's format, MSVD.py:229-234; needs h5py), an .npz archive or a dict."""
    if isinstance(video_fpath, dict):
        return video_fpath
    if str(video_fpath).endswith('.npz'):
        z = np.load(video_fpath)
        return {k: z[k] for k in z.files}
    try:
        import h5py
    except ImportError as ex:
        raise RuntimeError("reading {} needs h5py, which is not installed; convert the features to .npz".format(video_fpath)) from ex
    with h5py.File(video_fpath, 'r') as fin:
        return {vid: fin[vid][()] for vid in fin}


class CaptionFeatureDataset(torch.utils.data.Dataset):
    """dataset/MSVD.py:210-262 (MSVDDataset): one item per (clip, caption) pair -> (vid, feats (T, E) float32, targets (cap + 1,) int64).
    Clip ids are '<VideoID>_<Start>_<End>'; clips are visited in feature-file order, captions in CSV order."""

    def __init__(self, video_fpath, caption_fpath, vocab, n_frames, frame_sampling_method="uniform", rng=None):
        self.vocab, self.n_frames, self.method, self.rng = vocab, n_frames, frame_sampling_method, rng
        videos = load_features(video_fpath)
        df = _read_caption_table(caption_fpath)[['VideoID', 'Start', 'End', 'Description']]
        captions = {}
        for video_id, start, end, caption in df.values:
            captions.setdefault("{}_{}_{}".format(video_id, start, end), []).append(caption)
        self.pairs = [(vid, videos[vid], c) for vid in videos for c in captions.get(vid, [])]

    def __len__(self):
        return len(self.pairs)

    def __getitem__(self, i):
        vid, video, caption = self.pairs[i]
        return vid, sample_frames(video, self.n_frames, self.method, self.rng), self.vocab.encode(caption)


def collate(batch, batch_size=None):
    """MSVD.py:53-76: a short last batch is padded with copies of its last item (vid 'PAD'); features stay batch-major
    (B, T, E) float32, captions become time-major (cap + 1, B).  (The reference casts the captions to float here and back to long in
    train.py:248; they stay int64.)"""
    vids, videos, captions = (list(x) for x in zip(*batch))
    if batch_size is not None and len(vids) < batch_size:
        pad = batch_size - len(vids)
        vids += ["PAD"] * pad
        videos += [videos[-1].clone() for _ in range(pad)]
        captions += [captions[-1].clone() for _ in range(pad)]
    return vids, torch.stack(videos).float(), torch.stack(captions).transpose(0, 1).contiguous()


class PinnedBatchFeeder:
    """Double-buffered host -> device feed of (feats, targets) batches: batch i + 1 is copied from pinned host memory on a copy
    stream while step i computes (the pipeline bench.py's e2e leg times).  Iterating yields device tensors that stay valid until
    the next-but-one ``next()``."""

    def __init__(self, batches, device):
        self.it, self.device = iter(batches), torch.device(device)
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.slots = [None, None]
        self.ready = [torch.cuda.Event(), torch.cuda.Event()]
        self.k = 0
        self._issue(0)

    def _issue(self, k):
        try:
            _, feats, targets = next(self.it)
        except StopIteration:
            self.slots[k] = None
            return
        feats, targets = feats.pin_memory(), targets.pin_memory()
        self.copy_stream.wait_stream(torch.cuda.current_stream(self.device))          # the step that last read slot k has been issued
        with torch.cuda.stream(self.copy_stream):
            self.slots[k] = (feats.to(self.device, non_blocking=True), targets.to(self.device, non_blocking=True), feats, targets)
            self.ready[k].record(self.copy_stream)

    def __iter__(self):
        return self

    def __next__(self):
        k = self.k
        if self.slots[k] is None:
            raise StopIteration
        cur = torch.cuda.current_stream(self.device)
        cur.wait_event(self.ready[k])
        feats, targets = self.slots[k][0], self.slots[k][1]
        feats.record_stream(cur)                       # allocated on the copy stream, consumed on the compute stream
        targets.record_stream(cur)
        self.k = k ^ 1
        self._issue(self.k)
        return feats, targets
