"""CIDEr-D on the GPU: coco-caption's ``Cider(n=4, sigma=6.0).compute_score(gts, res)``
(pycocoevalcap/cider/cider_scorer.py) on integer token ids, with document frequencies from the evaluated corpus.

Two kernels (K11, csrc/sn_cider.cu): ``sn_cider_df`` counts, for every n-gram of the references, the images whose
references contain it, into a table on the device keyed on the full n-gram; ``sn_cider_scores`` then computes every
image's score in float64 (tf-idf vectors, norms, clipped products, the Gaussian length penalty).  The host packs the
corpus with ``bleu._pack`` (one host-to-device copy) and reads the per-image scores back once; the corpus score is
their ``np.mean``, as in the scorer.  Results match the scorer to rounding: the device ``log`` / ``pow`` are not
glibc's, and sums run in a different (but fixed) order, so a score is identical from run to run.

``corpus_cider`` scores one hypothesis set.  ``CiderD`` keeps the references and their document-frequency table on the
device, for scoring several hypothesis sets (every style, every epoch) against the same references."""
import math
import numbers

import numpy as np
import torch

from . import ops
from ._lib import SnError
from .bleu import _pack, _tokens

MAX_ORDER = 4
_DF_ERRORS = ((1, "the document-frequency table is full"), (2, "a token id is negative"),
              (4, "a sentence is longer than declared"))


def _check_params(n, sigma):
    if isinstance(n, bool) or not isinstance(n, numbers.Integral) or not 1 <= n <= MAX_ORDER:
        raise ValueError("CIDEr-D n must be an integer in 1..%d; got %r" % (MAX_ORDER, n))
    if not isinstance(sigma, numbers.Real) or not math.isfinite(sigma) or not sigma > 0:
        raise ValueError("CIDEr-D sigma must be finite and > 0; got %r" % (sigma,))


def _check_ids(tok):
    if tok.size and int(tok.min()) < 0:
        raise ValueError("CIDEr-D token ids must be non-negative")


def _capacity(ref_off, n):
    """Table slots for the references with offsets ``ref_off``: the power of two >= 2 x their number of n-grams of
    orders 1..n, so that the table is at most half full."""
    ref_len = np.diff(ref_off)
    grams = sum(int(np.maximum(ref_len - k, 0).sum()) for k in range(n))
    return 1 << max(1, (2 * grams - 1).bit_length())


def _check_df(err):
    if err:
        raise SnError("sn_cider_df: " + "; ".join(msg for bit, msg in _DF_ERRORS if err & bit))


def _check_samples(seqs, lengths, image_ids, n_img):
    """The argument checks of ``score_samples`` (ValueError, no device work): returns (R, ld, image ids int64 [R])."""
    if not isinstance(seqs, torch.Tensor) or seqs.dim() != 2:
        raise ValueError("seqs must be a 2-D tensor [R, max_len]; got %s" % (
            tuple(seqs.shape) if isinstance(seqs, torch.Tensor) else type(seqs).__name__,))
    R, ld = seqs.shape
    if not isinstance(lengths, torch.Tensor) or tuple(lengths.shape) != (R,):
        raise ValueError("lengths must be a tensor of shape [%d]" % R)
    ids = np.asarray(image_ids)
    if ids.shape != (R,):
        raise ValueError("%d image ids for %d rows" % (ids.size, R))
    if R and (not np.issubdtype(ids.dtype, np.integer) or int(ids.min()) < 0 or int(ids.max()) >= n_img):
        raise ValueError("image ids must be integers in 0..%d" % (n_img - 1))
    return R, ld, ids.astype(np.int64)


def _upload(list_of_references, hypotheses):
    """Checks and packs the corpus and copies it to the device once.  Returns the device views (hyp_tok, hyp_off,
    ref_tok, ref_off, ref_group), max_sentence_len, max_group_tokens, and the host copies of ref_off and ref_group."""
    buf, (n_img, R, Th, Tr), max_len, max_group = _pack(list_of_references, hypotheses)
    k = 2 * n_img + R + 3
    _check_ids(buf[k:].view(np.int32)[:Th + Tr])
    dev = torch.from_numpy(buf).to(torch.device("cuda", torch.cuda.current_device()))
    tok = dev[k:].view(torch.int32)
    views = (tok[:Th], dev[:n_img + 1], tok[Th:Th + Tr], dev[n_img + 1:n_img + R + 2], dev[n_img + R + 2:k])
    return views, max_len, max_group, buf[n_img + 1:n_img + R + 2], buf[n_img + R + 2:k]


def corpus_cider(list_of_references, hypotheses, n=4, sigma=6.0):
    """CIDEr-D of ``hypotheses`` (lists of integer token ids, one per image) against ``list_of_references`` (one list
    of references per image), computed on the current CUDA device.  Returns (corpus score, per-image scores as numpy
    float64 [n_img]): ``Cider(n, sigma).compute_score(gts, res)`` of coco-caption with ``gts[i]`` = the references and
    ``res[i]`` = [hypothesis] of image i, ids joined as words; document frequencies come from these references.

    Raises ValueError for an empty corpus, lists of different lengths, an image without references, ``n`` outside 1..4,
    a ``sigma`` that is not finite or not > 0, and token ids that are negative or outside int32, TypeError for ids that
    are not integers (all before any device work), and ``SnError`` for a sentence longer than 256 tokens or an image
    whose tokens do not fit in shared memory.  Empty hypotheses and references are valid."""
    _check_params(n, sigma)
    if len(list_of_references) != len(hypotheses):
        raise ValueError("%d reference lists for %d hypotheses" % (len(list_of_references), len(hypotheses)))
    if len(hypotheses) == 0:
        raise ValueError("CIDEr-D of an empty corpus")
    views, max_len, max_group, ref_off_h, _ = _upload(list_of_references, hypotheses)
    hyp_tok, hyp_off, ref_tok, ref_off, ref_group = views
    n_img = len(hypotheses)
    # the scores and the table's error word come back in one copy
    res = torch.empty(n_img + 1, dtype=torch.float64, device=hyp_off.device)
    err = res[n_img:].view(torch.int32)[:1]
    keys, counts = ops.cider_df(ref_tok, ref_off, ref_group, n, max_len, max_group, _capacity(ref_off_h, n), err)
    ops.cider_scores(hyp_tok, hyp_off, ref_tok, ref_off, ref_group, n, sigma, max_len, max_group, keys, counts,
                     out=res[:n_img])
    host = res.cpu().numpy()
    _check_df(int(host[n_img:].view(np.int32)[0]))
    scores = host[:n_img]
    return float(np.mean(scores)), scores


class CiderD:
    """The references of a corpus and their document-frequency table, on the current CUDA device.
    ``CiderD(refs, n, sigma).compute_score(hyps)`` equals ``corpus_cider(refs, hyps, n, sigma)`` bit for bit; the
    references are packed, copied and counted once, when the object is made.  Raises as ``corpus_cider``."""

    def __init__(self, list_of_references, n=4, sigma=6.0):
        _check_params(n, sigma)
        self.n, self.sigma = n, sigma
        self.n_img = len(list_of_references)
        if self.n_img == 0:
            raise ValueError("CIDEr-D of an empty corpus")
        views, self._ref_max_len, _, ref_off_h, ref_group_h = _upload(list_of_references, [[]] * self.n_img)
        _, _, self._ref_tok, self._ref_off, self._ref_group = views
        self._ref_tokens = np.diff(ref_off_h[ref_group_h])          # per image
        err = torch.empty(1, dtype=torch.int32, device=self._ref_off.device)
        self._keys, self._counts = ops.cider_df(self._ref_tok, self._ref_off, self._ref_group, n,
                                                self._ref_max_len, int(self._ref_tokens.max()),
                                                _capacity(ref_off_h, n), err)
        _check_df(int(err.item()))

    def compute_score(self, hypotheses):
        """(corpus score, per-image scores numpy float64 [n_img]) of ``hypotheses``, one per image, in order."""
        if len(hypotheses) != self.n_img:
            raise ValueError("%d hypotheses for %d reference lists" % (len(hypotheses), self.n_img))
        hyp_len = np.fromiter(map(len, hypotheses), np.int64, self.n_img)
        flat = []
        for h in hypotheses:
            flat.extend(h)
        tok = _tokens(flat)
        _check_ids(tok)
        buf = np.zeros(self.n_img + 1 + (tok.size + 1) // 2, np.int64)
        np.cumsum(hyp_len, out=buf[1:self.n_img + 1])
        buf[self.n_img + 1:].view(np.int32)[:tok.size] = tok
        dev = torch.from_numpy(buf).to(self._ref_off.device)
        max_len = max(self._ref_max_len, int(hyp_len.max()))
        max_group = int((hyp_len + self._ref_tokens).max())
        scores, _ = ops.cider_scores(dev[self.n_img + 1:].view(torch.int32)[:tok.size], dev[:self.n_img + 1],
                                     self._ref_tok, self._ref_off, self._ref_group, self.n, self.sigma, max_len,
                                     max_group, self._keys, self._counts)
        scores = scores.cpu().numpy()
        return float(np.mean(scores)), scores

    def score_samples(self, seqs, lengths, image_ids, start_token, end_token):
        """CIDEr-D of sampled captions against this corpus, for self-critical training (scst.py): device float64 [R].
        Row r's hypothesis is ``seqs[r, 1:lengths[r]]`` (column 0 holds ``start_token``) without a final
        ``end_token`` -- the layout of ``sample_captions`` -- and its references are those of image ``image_ids[r]``
        of the corpus this object was built from; idf uses that corpus' document frequencies and log(its image count),
        not the number of rows.  ``seqs`` (int64 [R, ld]) and ``lengths`` (int64 [R]) stay on the device; ``image_ids``
        is a host sequence of R corpus positions.  With ``image_ids = range(n_img)`` the scores equal those of
        ``compute_score`` on the same hypotheses bit for bit.  Raises ValueError, before any device work, for a
        ``seqs`` that is not 2-D, mismatched lengths and an image id out of range."""
        R, ld, ids = _check_samples(seqs, lengths, image_ids, self.n_img)
        dev = self._ref_off.device
        if R == 0:
            return torch.empty(0, dtype=torch.float64, device=dev)
        seqs = seqs.to(device=dev, dtype=torch.int64).contiguous()
        lengths = lengths.to(device=dev, dtype=torch.int64).contiguous()
        # shared-memory bounds from host-known sizes: the row width and the references of the images used
        max_len = max(self._ref_max_len, ld - 1)
        max_group = ld - 1 + int(self._ref_tokens[ids].max())
        return ops.cider_scores_rows(seqs, lengths, torch.from_numpy(ids).to(dev), end_token, self.n_img, self._ref_tok,
                                     self._ref_off, self._ref_group, self.n, self.sigma, max_len, max_group, self._keys,
                                     self._counts)
