"""CPU restatement of coco-caption's CIDEr-D scorer (pycocoevalcap/cider/cider_scorer.py, used through
``Cider(n=4, sigma=6.0).compute_score(gts, res)``), document frequencies from the evaluated corpus.  It is the checker
of ``icei_b200.cider`` and shares no code with it.

Sentences are lists of tokens (any hashable values; the scorer splits strings on whitespace first).  The functions
follow the scorer line by line, in its order and in float64 (``np.log``, ``np.sqrt``, ``np.e ** x``, ``np.mean``), so
for string tokens the results are the scorer's bit for bit.  One difference: when no reference of the corpus has a
single token, the scorer fails in its sanity check (``max()`` of no document frequencies); here the check is skipped and
the formula gives 0 for every image.

Pinned by hand-derived cases in tests/test_cider.py, and compared there with the live package when it is importable."""
import math
from collections import defaultdict

import numpy as np


def precook(words, n=4):
    """n-gram counts of a sentence, orders 1..n: order outer, position inner (dict order = first occurrence)."""
    counts = defaultdict(int)
    for k in range(1, n + 1):
        for i in range(len(words) - k + 1):
            ngram = tuple(words[i:i + k])
            counts[ngram] += 1
    return counts


class CiderScorer:
    """CiderScorer of cider_scorer.py for one corpus: ``hypotheses[i]`` is scored against ``list_of_references[i]``."""

    def __init__(self, list_of_references, hypotheses, n=4, sigma=6.0):
        self.n = n
        self.sigma = sigma
        self.crefs = [[precook(ref, n) for ref in refs] for refs in list_of_references]
        self.ctest = [precook(test, n) for test in hypotheses]
        self.document_frequency = defaultdict(float)
        self.ref_len = None
        self.per_order = []          # the summed sim() vector of each image, before its mean

    def compute_doc_freq(self):
        for refs in self.crefs:
            # the references of one image form one set: an image adds at most 1 to an n-gram's count
            for ngram in set([ngram for ref in refs for (ngram, count) in ref.items()]):
                self.document_frequency[ngram] += 1

    def counts2vec(self, cnts):
        vec = [defaultdict(float) for _ in range(self.n)]
        length = 0
        norm = [0.0 for _ in range(self.n)]
        for (ngram, term_freq) in cnts.items():
            # an n-gram in no reference has df 0 -> max(1.0, 0) -> idf = ref_len
            df = np.log(max(1.0, self.document_frequency[ngram]))
            n = len(ngram) - 1
            vec[n][ngram] = float(term_freq) * (self.ref_len - df)
            norm[n] += pow(vec[n][ngram], 2)
            if n == 1:                # the scorer's length: the number of bigrams, not of tokens
                length += term_freq
        norm = [np.sqrt(n) for n in norm]
        return vec, norm, length

    def sim(self, vec_hyp, vec_ref, norm_hyp, norm_ref, length_hyp, length_ref):
        delta = float(length_hyp - length_ref)
        val = np.array([0.0 for _ in range(self.n)])
        for n in range(self.n):
            for (ngram, count) in vec_hyp[n].items():
                # clipping: min of the two weights
                val[n] += min(vec_hyp[n][ngram], vec_ref[n][ngram]) * vec_ref[n][ngram]
            if (norm_hyp[n] != 0) and (norm_ref[n] != 0):
                val[n] /= (norm_hyp[n] * norm_ref[n])
            assert not math.isnan(val[n])
            # Gaussian length penalty
            val[n] *= np.e ** (-(delta ** 2) / (2 * self.sigma ** 2))
        return val

    def compute_cider(self):
        self.ref_len = np.log(float(len(self.crefs)))
        scores = []
        for test, refs in zip(self.ctest, self.crefs):
            vec, norm, length = self.counts2vec(test)
            score = np.array([0.0 for _ in range(self.n)])
            for ref in refs:
                vec_ref, norm_ref, length_ref = self.counts2vec(ref)
                score += self.sim(vec, vec_ref, norm, norm_ref, length, length_ref)
            self.per_order.append(score.copy())
            # mean over the n orders, divided by the number of references, times 10
            score_avg = np.mean(score)
            score_avg /= len(refs)
            score_avg *= 10.0
            scores.append(score_avg)
        return scores

    def compute_score(self):
        self.compute_doc_freq()
        assert not self.document_frequency or len(self.ctest) >= max(self.document_frequency.values())
        score = self.compute_cider()
        return np.mean(np.array(score)), np.array(score)


def corpus_cider(list_of_references, hypotheses, n=4, sigma=6.0):
    """(corpus score, per-image scores float64 [n_img]) = ``Cider(n, sigma).compute_score(gts, res)`` with
    ``gts[i] = list_of_references[i]`` and ``res[i] = [hypotheses[i]]``."""
    return CiderScorer(list_of_references, hypotheses, n, sigma).compute_score()


def per_order(list_of_references, hypotheses, n=4, sigma=6.0):
    """[n_img, n] float64: for each image, the sum over its references of the sim() vector (orders 1..n)."""
    scorer = CiderScorer(list_of_references, hypotheses, n, sigma)
    scorer.compute_score()
    return np.array(scorer.per_order).reshape(len(hypotheses), n)


def document_frequency(list_of_references, n=4):
    """{n-gram tuple: number of images whose references contain it}, orders 1..n (compute_doc_freq)."""
    scorer = CiderScorer(list_of_references, [], n)
    scorer.compute_doc_freq()
    return {g: int(c) for g, c in scorer.document_frequency.items()}
