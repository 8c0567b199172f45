"""ROUGE-L on the GPU: coco-caption's ``Rouge().compute_score(gts, res)`` (pycocoevalcap/rouge/rouge.py) on integer
token ids, beta = 1.2.

One kernel (K13, csrc/sn_rouge.cu) computes every image's score: exact longest-common-subsequence lengths against each
reference (bit-parallel, one warp per image), then the scorer's F-measure in float64, one correctly rounded operation
at a time in the scorer's order.  The scores are therefore the scorer's bit for bit, including its rule for empty
sentences (``"".split(" ")`` is ``[""]``: one token, shared only with another empty sentence).  The host packs the
corpus with ``bleu._pack`` (one host-to-device copy) and reads the per-image scores back once; the corpus score is
their ``np.mean``, as in the scorer.

``corpus_rouge`` scores one hypothesis set.  ``RougeL`` keeps the references on the device, for scoring several
hypothesis sets against them, and sampled captions for self-critical training (``score_samples``, as
``cider.CiderD``'s)."""
import numpy as np
import torch

from . import ops
from ._lib import SnError
from .bleu import _pack, _tokens
from .cider import _check_samples

BETA2 = 1.2 ** 2           # the scorer's self.beta ** 2, computed once here and handed to the kernel as a double
MAX_LEN = 256              # tokens per sentence (SN_BLEU_MAX_LEN, include/sn100.h): the hypothesis bit vector


def _upload(list_of_references, hypotheses):
    """Checks and packs the corpus and copies it to the device once.  Returns the device views (hyp_tok, hyp_off,
    ref_tok, ref_off, ref_group) and max_sentence_len.  A sentence longer than MAX_LEN raises SnError before the
    copy."""
    buf, (n_img, R, Th, Tr), max_len, _ = _pack(list_of_references, hypotheses)
    if max_len > MAX_LEN:
        raise SnError("ROUGE-L: a sentence has %d tokens; the limit is %d" % (max_len, MAX_LEN))
    k = 2 * n_img + R + 3
    dev = torch.from_numpy(buf).to(torch.device("cuda", torch.cuda.current_device()))
    tok = dev[k:].view(torch.int32)
    return (tok[:Th], dev[:n_img + 1], tok[Th:Th + Tr], dev[n_img + 1:n_img + R + 2], dev[n_img + R + 2:k]), max_len


def corpus_rouge(list_of_references, hypotheses):
    """ROUGE-L of ``hypotheses`` (lists of integer token ids, one per image) against ``list_of_references`` (one list
    of references per image), computed on the current CUDA device.  Returns (corpus score, per-image scores as numpy
    float64 [n_img]): ``Rouge().compute_score(gts, res)`` of coco-caption with ``gts[i]`` = the references and
    ``res[i]`` = [hypothesis] of image i, ids joined as words.

    Raises ValueError for an empty corpus, lists of different lengths, an image without references and token ids
    outside int32, TypeError for ids that are not integers, and ``SnError`` for a sentence longer than 256 tokens, all
    before any device work.  Empty hypotheses and references are valid, and so are negative ids."""
    if len(list_of_references) != len(hypotheses):
        raise ValueError("%d reference lists for %d hypotheses" % (len(list_of_references), len(hypotheses)))
    if len(hypotheses) == 0:
        raise ValueError("ROUGE-L of an empty corpus")
    (hyp_tok, hyp_off, ref_tok, ref_off, ref_group), max_len = _upload(list_of_references, hypotheses)
    scores = ops.rouge_l(hyp_tok, hyp_off, ref_tok, ref_off, ref_group, max_len, BETA2).cpu().numpy()
    return float(np.mean(scores)), scores


class RougeL:
    """The references of a corpus, on the current CUDA device.  ``RougeL(refs).compute_score(hyps)`` equals
    ``corpus_rouge(refs, hyps)`` bit for bit; the references are packed and copied once, when the object is made.
    Raises as ``corpus_rouge``."""

    def __init__(self, list_of_references):
        self.n_img = len(list_of_references)
        if self.n_img == 0:
            raise ValueError("ROUGE-L of an empty corpus")
        views, self._ref_max_len = _upload(list_of_references, [[]] * self.n_img)
        _, _, self._ref_tok, self._ref_off, self._ref_group = views

    def compute_score(self, hypotheses):
        """(corpus score, per-image scores numpy float64 [n_img]) of ``hypotheses``, one per image, in order.  Raises
        as ``corpus_rouge``, before any device work."""
        if len(hypotheses) != self.n_img:
            raise ValueError("%d hypotheses for %d reference lists" % (len(hypotheses), self.n_img))
        hyp_len = np.fromiter(map(len, hypotheses), np.int64, self.n_img)
        max_len = max(self._ref_max_len, int(hyp_len.max()))
        if max_len > MAX_LEN:
            raise SnError("ROUGE-L: a sentence has %d tokens; the limit is %d" % (max_len, MAX_LEN))
        flat = []
        for h in hypotheses:
            flat.extend(h)
        tok = _tokens(flat)
        buf = np.zeros(self.n_img + 1 + (tok.size + 1) // 2, np.int64)       # hyp_off | tokens, one copy
        np.cumsum(hyp_len, out=buf[1:self.n_img + 1])
        buf[self.n_img + 1:].view(np.int32)[:tok.size] = tok
        dev = torch.from_numpy(buf).to(self._ref_off.device)
        scores = ops.rouge_l(dev[self.n_img + 1:].view(torch.int32)[:tok.size], dev[:self.n_img + 1], self._ref_tok,
                             self._ref_off, self._ref_group, max_len, BETA2).cpu().numpy()
        return float(np.mean(scores)), scores

    def score_samples(self, seqs, lengths, image_ids, start_token, end_token):
        """ROUGE-L of sampled captions against this corpus, for self-critical training (``scst.scst_step`` takes a
        ``RougeL`` in place of a ``cider.CiderD``): device float64 [R].  Row r's hypothesis is ``seqs[r, 1:lengths[r]]``
        (column 0 holds ``start_token``) without a final ``end_token`` -- the layout of ``sample_captions`` -- and its
        references are those of image ``image_ids[r]`` of the corpus this object was built from.  ``seqs`` (int64
        [R, ld]) and ``lengths`` (int64 [R]) stay on the device; ``image_ids`` is a host sequence of R corpus positions.
        With ``image_ids = range(n_img)`` the scores equal those of ``compute_score`` on the same hypotheses bit for
        bit.  Raises ValueError, before any device work, for a ``seqs`` that is not 2-D, mismatched lengths and an image
        id out of range, and ``SnError`` for rows wider than 257 columns (256 tokens after <start>)."""
        R, ld, ids = _check_samples(seqs, lengths, image_ids, self.n_img)
        dev = self._ref_off.device
        if R == 0:
            return torch.empty(0, dtype=torch.float64, device=dev)
        seqs = seqs.to(device=dev, dtype=torch.int64).contiguous()
        lengths = lengths.to(device=dev, dtype=torch.int64).contiguous()
        return ops.rouge_l_rows(seqs, lengths, torch.from_numpy(ids).to(dev), end_token, self.n_img, self._ref_tok,
                                self._ref_off, self._ref_group, max(self._ref_max_len, ld - 1), BETA2)
