"""fp64 CIDEr-D oracle on id captions: a plain-Python, dict-based restatement of coco-caption's CiderScorer / CiderD.compute_score
(n = 4, sigma = 6), with the document frequencies taken from the reference corpus ("corpus" mode).  It shares no code with
recnet_b200.cider: captions are tuples of ids, n-grams are tuples, vectors are dicts.

    corpus = Corpus(refs)                # refs[video] = list of id sequences
    corpus.score(candidate, video)       # CIDEr-D of one id sequence against the references of `video`
"""
import math
from collections import defaultdict

N, SIGMA = 4, 6.0


def caption(ids, eos_id=2):
    """Ids before the first eos_id, <PAD> (0) or negative id."""
    out = []
    for v in ids:
        v = int(v)
        if v == eos_id or v <= 0:
            break
        out.append(v)
    return tuple(out)


def precook(words, n=N):
    """CiderScorer's precook: n-gram -> count, for n = 1..4."""
    counts = defaultdict(int)
    for k in range(1, n + 1):
        for i in range(len(words) - k + 1):
            counts[tuple(words[i:i + k])] += 1
    return counts


class Corpus:
    def __init__(self, refs, eos_id=2):
        self.eos_id = eos_id
        self.crefs = [[precook(caption(r, eos_id)) for r in rs] for rs in refs]
        self.df = defaultdict(float)
        for rs in self.crefs:
            for g in set(g for r in rs for g in r):
                self.df[g] += 1
        self.ref_len = math.log(float(len(self.crefs)))

    def counts2vec(self, cnts):
        """CiderScorer.counts2vec: per-order weight dicts, their L2 norms, and the 'length' (the bigram count)."""
        vec = [defaultdict(float) for _ in range(N)]
        norm = [0.0] * N
        length = 0
        for g, tf in cnts.items():
            n = len(g) - 1
            df = math.log(max(1.0, self.df[g]))
            vec[n][g] = float(tf) * (self.ref_len - df)
            norm[n] += vec[n][g] ** 2
            if n == 1:
                length += tf
        return vec, [math.sqrt(x) for x in norm], length

    @staticmethod
    def sim(vec_h, vec_r, norm_h, norm_r, len_h, len_r):
        delta = float(len_h - len_r)
        val = [0.0] * N
        for n in range(N):
            for g in vec_h[n]:
                val[n] += min(vec_h[n][g], vec_r[n].get(g, 0.0)) * vec_r[n].get(g, 0.0)
            if norm_h[n] != 0 and norm_r[n] != 0:
                val[n] /= norm_h[n] * norm_r[n]
            val[n] *= math.exp(-(delta ** 2) / (2 * SIGMA ** 2))
        return val

    def score(self, ids, video):
        vec, norm, length = self.counts2vec(precook(caption(ids, self.eos_id)))
        total = [0.0] * N
        for r in self.crefs[video]:
            vr, nr, lr = self.counts2vec(r)
            for n, v in enumerate(self.sim(vec, vr, norm, nr, length, lr)):
                total[n] += v
        return 10.0 * (sum(total) / N) / len(self.crefs[video])

    def scores(self, rows, videos):
        return [self.score(r, v) for r, v in zip(rows, videos)]
