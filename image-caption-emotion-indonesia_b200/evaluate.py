"""Batched evaluation (SURVEY.md section 8 f2): the two loops that follow the decoder in the reference,
  * ``validate``  = val_factual / val_emotion of stylenet/train_multitask.py:272-361 (teacher_forcing_ratio = 0 forward,
    token loss, top-5 accuracy, per-caption arg-max ids for BLEU), and
  * ``generate``  = the per-image ``sample()`` loop of stylenet/evaluator.py:63-101 (``styles=``: every image in every
    style, one mixed-style beam search per batch),
with everything id-level done on the device: the loss / top-5 / arg-max come out of the fused softmax kernel instead of
five passes over the [N, V] logits on the host, and beam search runs for a whole batch of images at once
(``sample_batch``).  Corpus BLEU over the ids (``bleu.corpus_bleu``, nltk's semantics) and CIDEr-D
(``cider.corpus_cider``) and ROUGE-L (``rouge.corpus_rouge``, both coco-caption's semantics) run on the device too:
``validate(..., bleu_weights=..., cider=True, rouge=True)`` adds them to the result, and ``generate``'s captions go to
``bleu.corpus_bleu`` / ``cider.CiderD`` / ``rouge.RougeL`` once <start> / <end> are stripped.  Ids -> words stays
with the caller."""
import torch

from .bleu import corpus_bleu
from .cider import corpus_cider
from .rouge import corpus_rouge
from .packing import get_plan


def _strip(ids, start, end):
    return [w for w in ids if w != start and w != end]


@torch.no_grad()
def validate(decoder, batches, start_token, end_token, encoder=None, mode=None, attention=None, bleu_weights=None,
             cider=False, rouge=False):
    """``batches`` yields (images_or_features, captions [B,T] int64, lengths, all_captions | None) like the reference's
    data loader (sorted by length, data_loader.py:116-145).  Returns dict(loss, top5 (percent), hypotheses,
    references, n_tokens) with the reference's definitions: loss = token-mean cross entropy averaged over batches
    weighted by tokens (AverageMeter, utils.py:93-110), top5 = accuracy(scores, targets, 5) (utils.py:127-140),
    hypotheses = per-caption arg-max ids cut to the caption length with <start>/<end> removed.
    ``bleu_weights`` (a weight tuple or a list of them): the dict also holds "bleu" =
    ``bleu.corpus_bleu(references, hypotheses, bleu_weights)`` (train_multitask.py:341); every batch then needs its
    all_captions, else ValueError.  ``cider=True``: the dict also holds "cider" = the corpus CIDEr-D
    ``cider.corpus_cider(references, hypotheses)[0]``, with the same need for all_captions.  ``rouge=True``: the dict
    also holds "rouge_l" = the corpus ROUGE-L ``rouge.corpus_rouge(references, hypotheses)[0]``, with the same need."""
    was_training = decoder.training
    decoder.eval()
    if encoder is not None:
        encoder.eval()
    att = hasattr(decoder, "attention") if attention is None else attention
    kw = {} if mode is None else {"mode": mode}
    tot_loss = tot_hit = 0.0
    tot_tok = 0
    hyps, refs = [], []
    for images, captions, lengths, all_caps in batches:
        if all_caps is None and (bleu_weights is not None or cider or rouge):
            decoder.train(was_training)
            raise ValueError("validate(bleu_weights=... / cider=True / rouge=True) needs the references (all_captions) "
                             "of every batch")
        feats = encoder(images) if encoder is not None else images
        lengths = [int(l) for l in lengths]
        if att:
            l1 = [l - 1 for l in lengths]
            loss, st = decoder.forward_loss(captions[:, :-1], l1, feats, full_captions=captions,
                                            teacher_forcing_ratio=0.0, backward=False, **kw)
            plan = get_plan(l1)
        else:
            loss, st = decoder.forward_loss(captions, lengths, feats, teacher_forcing_ratio=0.0, backward=False, **kw)
            plan = get_plan(lengths)
        n = plan.N
        tot_loss += float(loss.item()) * n
        tot_hit += float(st["top5hit"].sum().item())
        tot_tok += n
        am = st["argmax"].cpu().tolist()
        for b, L in enumerate(plan.lengths):
            hyps.append(_strip([am[plan.off[t] + b] for t in range(L)], start_token, end_token))
        if all_caps is not None:
            for caps in all_caps:
                refs.append([_strip([int(w) for w in c], start_token, end_token) for c in caps])
    decoder.train(was_training)
    res = {"loss": tot_loss / max(tot_tok, 1), "top5": 100.0 * tot_hit / max(tot_tok, 1), "hypotheses": hyps,
           "references": refs, "n_tokens": tot_tok}
    if bleu_weights is not None:
        res["bleu"] = corpus_bleu(refs, hyps, bleu_weights)
    if cider:
        res["cider"] = corpus_cider(refs, hyps)[0]
    if rouge:
        res["rouge_l"] = corpus_rouge(refs, hyps)[0]
    return res


@torch.no_grad()
def generate(decoder, feature_batches, start_token, end_token, k=5, mode=None, encoder=None, styles=None, **sample_kw):
    """Beam-search captions for every image: ``feature_batches`` yields feature tensors ([n, E] / [n, S, S, D]) or, with
    ``encoder``, image batches.  Returns a list of id lists (one per image, as ``sample()`` would return them).
    ``styles`` (style decoders, e.g. ``STYLES``): caption every image in every listed style with ONE mixed-style
    ``sample_batch`` per feature batch; returns {style: [id lists]}, each entry equal to ``generate(..., mode=style)``."""
    decoder.eval()
    kw = dict(sample_kw)
    if styles is not None:
        styles = list(styles)
        if mode is not None:
            raise ValueError("generate() takes mode or styles, not both")
        if not styles:
            raise ValueError("empty styles")
        if len(set(styles)) != len(styles):
            raise ValueError("duplicate style in %r" % (styles,))
        out = {s: [] for s in styles}
        for x in feature_batches:
            feats = encoder(x) if encoder is not None else x
            n = feats.shape[0]
            # image-major, style-minor: image i in style s is row i * len(styles) + s
            rep = feats.repeat_interleave(len(styles), 0)
            ids = decoder.sample_batch(rep, start_token, end_token, k=k, mode=styles * n, **kw)
            for j, t in enumerate(ids):
                out[styles[j % len(styles)]].append(t[0].tolist())
        return out
    if mode is not None:
        kw["mode"] = mode
    out = []
    for x in feature_batches:
        feats = encoder(x) if encoder is not None else x
        for ids in decoder.sample_batch(feats, start_token, end_token, k=k, **kw):
            out.append(ids[0].tolist())
    return out
