"""CPU restatement of coco-caption's ROUGE-L scorer (pycocoevalcap/rouge/rouge.py, ``Rouge().compute_score(gts, res)``).
It is the checker of ``icei_b200.rouge`` and shares no code with it.

``my_lcs`` and ``Rouge`` follow the scorer line by line and work, as it does, on sentences given as strings split on a
single space, so its rule for empty sentences comes from ``"".split(" ") == [""]`` itself.  ``corpus_rouge`` and
``sample_scores`` join integer token ids into such strings.  The arithmetic is the scorer's (Python float64, beta =
1.2), so the per-image scores are its own, bit for bit.

Pinned by hand-derived cases in tests/test_rouge.py, and compared there with the live package when it is importable."""
import numpy as np


def my_lcs(string, sub):
    """Length of the longest common subsequence of two token lists: the scorer's dynamic-programming table."""
    if len(string) < len(sub):
        sub, string = string, sub
    lengths = [[0 for i in range(0, len(sub) + 1)] for j in range(0, len(string) + 1)]
    for j in range(1, len(sub) + 1):
        for i in range(1, len(string) + 1):
            if string[i - 1] == sub[j - 1]:
                lengths[i][j] = lengths[i - 1][j - 1] + 1
            else:
                lengths[i][j] = max(lengths[i - 1][j], lengths[i][j - 1])
    return lengths[len(string)][len(sub)]


class Rouge:
    """The scorer's Rouge class."""

    def __init__(self):
        self.beta = 1.2

    def calc_score(self, candidate, refs):
        """ROUGE-L of ``candidate`` (a list holding one sentence string) against ``refs`` (sentence strings)."""
        assert len(candidate) == 1
        assert len(refs) > 0
        prec = []
        rec = []
        token_c = candidate[0].split(" ")
        for reference in refs:
            token_r = reference.split(" ")
            lcs = my_lcs(token_r, token_c)
            prec.append(lcs / float(len(token_c)))
            rec.append(lcs / float(len(token_r)))
        prec_max = max(prec)
        rec_max = max(rec)
        # precision and recall may come from different references
        if prec_max != 0 and rec_max != 0:
            score = ((1 + self.beta ** 2) * prec_max * rec_max) / float(rec_max + self.beta ** 2 * prec_max)
        else:
            score = 0.0
        return score

    def compute_score(self, gts, res):
        """(mean score, per-image scores) over the image ids of ``gts``, in its order."""
        assert gts.keys() == res.keys()
        imgIds = gts.keys()
        score = []
        for id in imgIds:
            hypo = res[id]
            ref = gts[id]
            score.append(self.calc_score(hypo, ref))
            assert type(hypo) is list
            assert len(hypo) == 1
            assert type(ref) is list
            assert len(ref) > 0
        average_score = np.mean(np.array(score))
        return average_score, np.array(score)


def words(ids):
    """Integer token ids as the scorer's input: one string, ids joined by single spaces."""
    return " ".join(map(str, ids))


def corpus_rouge(list_of_references, hypotheses):
    """(corpus score, per-image scores float64 [n_img]) = ``Rouge().compute_score(gts, res)`` with
    ``gts[i] = list_of_references[i]`` and ``res[i] = [hypotheses[i]]``, ids joined as words."""
    gts = {i: [words(r) for r in refs] for i, refs in enumerate(list_of_references)}
    res = {i: [words(h)] for i, h in enumerate(hypotheses)}
    return Rouge().compute_score(gts, res)


def sample_scores(corpus_references, image_ids, hypotheses):
    """float64 [R]: the ROUGE-L of ``hypotheses[r]`` against ``corpus_references[image_ids[r]]`` (``calc_score``), as
    self-critical training scores the samples of a minibatch against the training corpus."""
    scorer = Rouge()
    return np.array([scorer.calc_score([words(h)], [words(r) for r in corpus_references[i]])
                     for h, i in zip(hypotheses, image_ids)], dtype=np.float64)
