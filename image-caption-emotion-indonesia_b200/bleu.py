"""Corpus BLEU on the GPU: a drop-in for ``nltk.translate.bleu_score.corpus_bleu`` on integer token ids, the metric the
reference selects its checkpoints by (stylenet/train_multitask.py:341, evaluator.py:103).

The n-gram statistics of every hypothesis come from one kernel (K10, ``sn_bleu_counts``: clipped matches and
denominators for n = 1..4, hypothesis length, closest reference length, all int32).  The host packs the corpus with
numpy, makes one host-to-device copy, and reads back one column sum of 10 int64 totals; nltk's final formula is then
evaluated on those integers in float64, in nltk's order.  Integer statistics are exact, so the scores are those of
nltk's pure-Python loop, bit for bit."""
import array
import math
import sys
from itertools import chain

import numpy as np
import torch

from . import ops

MAX_ORDER = 4


def _weight_sets(weights):
    """nltk's rule: ``weights`` is one tuple of weights, or a list of such tuples when its first item is indexable."""
    if len(weights) == 0:
        raise ValueError("weights is empty")
    try:
        weights[0][0]
    except TypeError:
        weights = [weights]
    for w in weights:
        if not 1 <= len(w) <= MAX_ORDER:
            raise ValueError("BLEU weights need 1..%d entries (n-gram orders); got %r" % (MAX_ORDER, tuple(w)))
    return weights


def _tokens(flat):
    """int32 array of the token ids in ``flat`` (a list); TypeError for non-integers, ValueError outside int32.
    array.array converts a list of Python ints in C with exactly these checks (typecode "i" is 32-bit on every
    platform CUDA supports); it is about three times faster than np.array on such a list."""
    try:
        return np.frombuffer(array.array("i", flat), np.int32)
    except OverflowError:
        raise ValueError("token ids must fit in int32") from None
    except TypeError as e:
        raise TypeError("BLEU tokens must be integer ids: %s" % e) from None


def _pack(list_of_references, hypotheses):
    """CSR form of the corpus in ONE int64 host buffer: hyp_off [n+1] | ref_off [R+1] | ref_group [n+1] | tokens
    (int32 pairs: hypotheses, then references).  Returns (buffer, section sizes, max_sentence_len, max_group_tokens)."""
    n = len(hypotheses)
    n_refs = np.fromiter(map(len, list_of_references), np.int64, n)
    if n_refs.size and n_refs.min() == 0:
        raise ValueError("hypothesis %d has no references" % int(np.argmin(n_refs)))
    refs = list(chain.from_iterable(list_of_references))
    hyp_len = np.fromiter(map(len, hypotheses), np.int64, n)
    ref_len = np.fromiter(map(len, refs), np.int64, len(refs))
    flat = []
    for s in chain(hypotheses, refs):      # list.extend per sentence: half the cost of an element-wise chain
        flat.extend(s)
    tok = _tokens(flat)
    R, T = len(refs), tok.size
    buf = np.zeros(2 * n + R + 3 + (T + 1) // 2, np.int64)
    hyp_off, ref_off, ref_group = buf[:n + 1], buf[n + 1:n + R + 2], buf[n + R + 2:2 * n + R + 3]
    np.cumsum(hyp_len, out=hyp_off[1:])
    np.cumsum(ref_len, out=ref_off[1:])
    np.cumsum(n_refs, out=ref_group[1:])
    buf[2 * n + R + 3:].view(np.int32)[:T] = tok
    max_len = int(max(hyp_len.max(initial=0), ref_len.max(initial=0)))
    group = hyp_len + ref_off[ref_group[1:]] - ref_off[ref_group[:-1]]
    return buf, (n, R, int(hyp_off[-1]), int(ref_off[-1])), max_len, int(group.max(initial=0))


def _stats(list_of_references, hypotheses):
    """Per-hypothesis statistics [n, 10] int32 on the current CUDA device (columns: include/sn100.h, K10)."""
    buf, (n, R, Th, Tr), max_len, max_group = _pack(list_of_references, hypotheses)
    dev = torch.from_numpy(buf).to(torch.device("cuda", torch.cuda.current_device()))
    k = 2 * n + R + 3
    tok = dev[k:].view(torch.int32)
    return ops.bleu_counts(tok[:Th], dev[:n + 1], tok[Th:Th + Tr], dev[n + 1:n + R + 2], dev[n + R + 2:k],
                           max_len, max_group)


def _score(tot, weight):
    """nltk's corpus_bleu tail on the integer totals: brevity penalty, method0 smoothing, weighted log-mean."""
    num, den, c, r = tot[0:MAX_ORDER], tot[MAX_ORDER:2 * MAX_ORDER], tot[8], tot[9]
    bp = 1 if c > r else (0 if c == 0 else math.exp(1 - r / c))
    p = [num[i] / den[i] if num[i] != 0 else sys.float_info.min for i in range(len(weight))]
    return bp * math.exp(math.fsum(w * math.log(x) for w, x in zip(weight, p)))


def corpus_bleu(list_of_references, hypotheses, weights=(0.25, 0.25, 0.25, 0.25)):
    """Corpus BLEU of ``hypotheses`` (lists of integer token ids) against ``list_of_references`` (one list of
    references per hypothesis), computed on the current CUDA device.

    The same result as ``nltk.translate.bleu_score.corpus_bleu(list_of_references, hypotheses, weights)`` with its
    defaults: no smoothing (``method0``: a zero n-gram precision counts as ``sys.float_info.min``) and
    ``auto_reweigh=False``.  ``smoothing_function`` and ``auto_reweigh`` are not accepted.  Orders 1..len(weights) are
    used, at most 4.  ``weights`` may also be a list of weight tuples: the scores of all of them then come from one
    kernel run and are returned as a list (as in nltk, a list holding one tuple returns a plain score).

    Raises AssertionError when the two lists differ in length (as nltk), ValueError for a hypothesis without references
    (nltk: ``min()`` of an empty sequence), for more than 4 weights, for an empty ``weights`` and for token ids outside
    int32, TypeError for tokens that are not integers, and ``SnError`` for a sentence longer than 256 tokens.  An empty
    corpus scores 0; so does a corpus without a single unigram match."""
    assert len(list_of_references) == len(hypotheses), (
        "The number of hypotheses and their reference(s) should be the same ")
    weights = _weight_sets(weights)
    zero = 0 if len(weights) == 1 else [0] * len(weights)
    if len(hypotheses) == 0:
        return zero
    tot = _stats(list_of_references, hypotheses).sum(0, dtype=torch.int64).tolist()
    if tot[0] == 0:
        return zero
    scores = [_score(tot, w) for w in weights]
    return scores[0] if len(weights) == 1 else scores
