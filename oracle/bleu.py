"""CPU restatement of nltk's corpus BLEU (nltk/translate/bleu_score.py), the model-selection metric of the reference
(stylenet/train_multitask.py:341, evaluator.py:103).  It is the checker of ``icei_b200.bleu`` and shares no code with it.

Tokens may be any hashable values.  Only the default smoothing (``SmoothingFunction().method0``) and
``auto_reweigh=False`` are restated -- the reference calls ``corpus_bleu`` with neither argument.  Like nltk, the corpus
sums the UN-normalised numerators and denominators of every sentence (nltk builds ``Fraction(..., _normalize=False)``);
``modified_precision`` therefore returns the pair (numerator, denominator) instead of a Fraction.

Pinned by the known answers in nltk's docstrings (tests/test_bleu.py)."""
import math
import sys
from collections import Counter


def ngrams(sequence, n):
    """nltk.util.ngrams: the n-grams of a sequence, in order."""
    sequence = list(sequence)
    return [tuple(sequence[i:i + n]) for i in range(len(sequence) - n + 1)]


def modified_precision(references, hypothesis, n):
    """nltk.translate.bleu_score.modified_precision -> (numerator, denominator), un-normalised."""
    counts = Counter(ngrams(hypothesis, n)) if len(hypothesis) >= n else Counter()
    max_counts = {}
    for reference in references:
        reference_counts = Counter(ngrams(reference, n)) if len(reference) >= n else Counter()
        for ngram in counts:
            max_counts[ngram] = max(max_counts.get(ngram, 0), reference_counts[ngram])
    clipped_counts = {ngram: min(count, max_counts[ngram]) for ngram, count in counts.items()}
    numerator = sum(clipped_counts.values())
    denominator = max(1, sum(counts.values()))
    return numerator, denominator


def closest_ref_length(references, hyp_len):
    """nltk.translate.bleu_score.closest_ref_length: ties go to the shorter reference."""
    ref_lens = (len(reference) for reference in references)
    return min(ref_lens, key=lambda ref_len: (abs(ref_len - hyp_len), ref_len))


def brevity_penalty(closest_ref_len, hyp_len):
    """nltk.translate.bleu_score.brevity_penalty."""
    if hyp_len > closest_ref_len:
        return 1
    elif hyp_len == 0:
        return 0
    else:
        return math.exp(1 - closest_ref_len / hyp_len)


def corpus_bleu(list_of_references, hypotheses, weights=(0.25, 0.25, 0.25, 0.25)):
    """nltk.translate.bleu_score.corpus_bleu with smoothing method0 and auto_reweigh=False.  ``weights`` may be a list
    of weight tuples: then one score per tuple (a list, unless it holds one tuple)."""
    p_numerators = Counter()
    p_denominators = Counter()
    hyp_lengths, ref_lengths = 0, 0
    assert len(list_of_references) == len(hypotheses), (
        "The number of hypotheses and their reference(s) should be the same ")
    try:
        weights[0][0]
    except TypeError:
        weights = [weights]
    max_weight_length = max(len(weight) for weight in weights)
    for references, hypothesis in zip(list_of_references, hypotheses):
        for i in range(1, max_weight_length + 1):
            numerator, denominator = modified_precision(references, hypothesis, i)
            p_numerators[i] += numerator
            p_denominators[i] += denominator
        hyp_len = len(hypothesis)
        hyp_lengths += hyp_len
        ref_lengths += closest_ref_length(references, hyp_len)
    bp = brevity_penalty(ref_lengths, hyp_lengths)
    if p_numerators[1] == 0:
        return 0 if len(weights) == 1 else [0] * len(weights)
    # method0: a zero precision becomes sys.float_info.min, so that its log stands for "0" in the geometric mean
    p_n = [p_numerators[i] / p_denominators[i] if p_numerators[i] != 0 else sys.float_info.min
           for i in range(1, max_weight_length + 1)]
    bleu_scores = []
    for weight in weights:
        s = (w_i * math.log(p_i) for w_i, p_i in zip(weight, p_n) if p_i > 0)
        bleu_scores.append(bp * math.exp(math.fsum(s)))
    return bleu_scores[0] if len(weights) == 1 else bleu_scores


def sentence_bleu(references, hypothesis, weights=(0.25, 0.25, 0.25, 0.25)):
    """nltk.translate.bleu_score.sentence_bleu: corpus_bleu of a one-sentence corpus."""
    return corpus_bleu([references], [hypothesis], weights)


def sentence_stats(references, hypothesis):
    """The ten integers sn_bleu_counts writes for one hypothesis (layout: include/sn100.h, K10)."""
    mp = [modified_precision(references, hypothesis, n) for n in range(1, 5)]
    return ([m[0] for m in mp] + [m[1] for m in mp] + [len(hypothesis)]
            + [closest_ref_length(references, len(hypothesis)) if references else 0])
