"""CPU restatement of self-critical training on CIDEr-D (``icei_b200.scst``, K12 ``sn_sample_step``) in numpy / torch
float64.  It is the checker of the GPU path and shares no code with it:

- ``hash_u32`` / ``gumbel``: the counter-based noise of include/sn100.h (sn_sample_step), from the C expressions;
- ``draw``: the Gumbel-max (or arg-max) choice of one step over given logits;
- ``teacher_forced_logits``: the logits the sampler sees for a given sequence, built on the reference's
  ``forward_step`` (step 0 feeds the image, step t the token of step t - 1);
- ``weighted_loss``: sum_r w_r NLL_r / denom through the port's autograd;
- ``sample_scores``: CIDEr-D of samples against a corpus' references with that corpus' document frequencies (an
  external df table), built on oracle/cider.py's ``CiderScorer``;
- ``reference_step``: one SCST step given the GPU's samples (the sampling itself is random, the rest is checked).
"""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import cider as cider_oracle
from oracle.port import pack_targets

M64 = (1 << 64) - 1
SEED_MUL = 0x9E3779B97F4A7C15


def hash_u32(seed, row, col):
    """sn_common.cuh hash_u32 on Python ints (uint64 arithmetic made explicit)."""
    x = (seed ^ ((row << 32) | col)) & M64
    x ^= x >> 33
    x = (x * 0xff51afd7ed558ccd) & M64
    x ^= x >> 33
    x = (x * 0xc4ceb9fe1a85ec53) & M64
    x ^= x >> 33
    return x & 0xFFFFFFFF


def hash_u32_np(seed, row, cols):
    """hash_u32 over a numpy array of columns (uint64, wrapping)."""
    with np.errstate(over="ignore"):
        x = np.uint64(seed) ^ ((np.uint64(row) << np.uint64(32)) | cols.astype(np.uint64))
        x ^= x >> np.uint64(33)
        x *= np.uint64(0xff51afd7ed558ccd)
        x ^= x >> np.uint64(33)
        x *= np.uint64(0xc4ceb9fe1a85ec53)
        x ^= x >> np.uint64(33)
    return (x & np.uint64(0xFFFFFFFF)).astype(np.uint64)


def step_seed(seed, step):
    """seed_t = seed * 0x9E3779B97F4A7C15 + step (uint64, wrapping)."""
    return (seed * SEED_MUL + step) & M64


def gumbel(seed, step, row, V):
    """float64 [V]: g_v = -log(-log(u)), u = ((hash_u32(seed_t, row, v) >> 8) + 0.5) / 2^24."""
    h = hash_u32_np(step_seed(seed, step), row, np.arange(V, dtype=np.uint64))
    u = ((h >> np.uint64(8)).astype(np.float64) + 0.5) / 16777216.0
    return -np.log(-np.log(u))


def perturbed(logits, seed, step, row, temperature):
    """float64 [V]: logit_v / temperature + g_v (the float32 logits widened first, as the kernel does)."""
    x = np.asarray(logits, dtype=np.float32).astype(np.float64)
    return x / float(temperature) + gumbel(seed, step, row, x.shape[0])


def draw(logits, seed, step, row, temperature=1.0, greedy=False):
    """The token of one draw: the first index of the maximum (np.argmax keeps the lowest index)."""
    if greedy:
        return int(np.argmax(np.asarray(logits, dtype=np.float32)))
    return int(np.argmax(perturbed(logits, seed, step, row, temperature)))


def teacher_forced_logits(step_fn, embed, out, feature, seq, length):
    """float64 [length - 1, V]: the logits the sampler sees on sequence ``seq`` (``[<start>, w1, ...]``) -- step 0 feeds
    ``feature`` (output discarded), step t >= 1 feeds ``embed(seq[t - 1])``, row t - 1 holds step t's logits.
    ``step_fn(x, (h, c)) -> (h, (h, c))``, ``embed`` / ``out``: the decoder's embedding and output projection."""
    x = feature.double().view(1, -1)
    H = out.weight.shape[1]
    state = (x.new_zeros(1, H), x.new_zeros(1, H))
    h, state = step_fn(x, state)
    rows = []
    for t in range(1, int(length)):
        x = embed(torch.tensor([int(seq[t - 1])])).double()
        h, state = step_fn(x, state)
        rows.append(out(h)[0])
    return torch.stack(rows).detach()


def weighted_loss(outputs, targets, weights, denom):
    """sum_r w_r * NLL_r / denom over packed rows (the loss of ``forward_loss(..., token_weights=w, n_global=denom)``)."""
    nll = F.cross_entropy(outputs, targets, reduction="none")
    return (weights.to(nll.dtype) * nll).sum() / float(denom)


def advantages(rewards, n, baseline, greedy_rewards=None):
    r = np.asarray(rewards, dtype=np.float64).reshape(-1, n)
    if baseline == "mean":
        base = (r.sum(1, keepdims=True) - r) / (n - 1)
    else:
        base = np.broadcast_to(np.asarray(greedy_rewards, dtype=np.float64).reshape(-1, 1), r.shape)
    return (r - base).reshape(-1), base.reshape(-1)


def sample_scores(corpus_references, image_ids, hypotheses, n=4, sigma=6.0):
    """float64 [R]: the CIDEr-D of ``hypotheses[r]`` against ``corpus_references[image_ids[r]]``, with the document
    frequencies and ``ref_len = log(len(corpus_references))`` of the whole corpus (an external df table, as
    self-critical training scores samples of a minibatch against the training corpus).  The scorer's own steps
    (``compute_doc_freq``, ``counts2vec``, ``sim`` and the mean of ``compute_cider``) in its order, so when
    ``image_ids`` is ``range(len(corpus_references))`` this is ``oracle.cider.corpus_cider``'s per-image vector."""
    scorer = cider_oracle.CiderScorer(corpus_references, [], n, sigma)
    scorer.compute_doc_freq()
    scorer.ref_len = np.log(float(len(scorer.crefs)))
    scores = []
    for hyp, i in zip(hypotheses, image_ids):
        vec, norm, length = scorer.counts2vec(cider_oracle.precook(hyp, n))
        score = np.array([0.0 for _ in range(n)])
        for ref in scorer.crefs[i]:
            vec_ref, norm_ref, length_ref = scorer.counts2vec(ref)
            score += scorer.sim(vec, vec_ref, norm, norm_ref, length, length_ref)
        score_avg = np.mean(score)
        score_avg /= len(scorer.crefs[i])
        score_avg *= 10.0
        scores.append(score_avg)
    return np.array(scores, dtype=np.float64)


def _hyp(seq, length, end_token):
    h = [int(t) for t in seq[1:int(length)]]
    if h and h[-1] == end_token:
        h = h[:-1]
    return h


def reference_step(forward, params, optimizer, corpus_refs, features, image_ids, seqs, lengths, n, baseline,
                   end_token, greedy_seqs=None, greedy_lengths=None, grad_clip=0.5):
    """One SCST step on the CPU given the sampled ``seqs`` / ``lengths`` (and the greedy captions for
    baseline="greedy"): rewards (``sample_scores``), advantages, the stable length sort, token weights
    (0 on the image step), the weighted loss through ``forward(captions, lengths, features)`` (teacher-forced, no
    dropout), clip_gradient and ``optimizer.step()``.  Returns (loss, mean reward, mean baseline)."""
    seqs = torch.as_tensor(seqs).cpu()
    lens = [int(l) for l in torch.as_tensor(lengths).cpu().tolist()]
    ids = [int(i) for i in image_ids for _ in range(n)]
    rewards = sample_scores(corpus_refs, ids, [_hyp(s, l, end_token) for s, l in zip(seqs, lens)])
    g = None
    if baseline == "greedy":
        g = sample_scores(corpus_refs, list(image_ids),
                          [_hyp(s, l, end_token) for s, l in zip(torch.as_tensor(greedy_seqs).cpu(),
                                                                 torch.as_tensor(greedy_lengths).tolist())])
    adv, base = advantages(rewards, n, baseline, g)
    order = sorted(range(len(lens)), key=lambda r: -lens[r])
    lens_s = [lens[r] for r in order]
    cap = seqs[order]
    feats = features.detach().cpu()[[r // n for r in order]]
    weights = []
    B = len(lens_s)
    for t in range(lens_s[0]):
        for b in range(B):
            if lens_s[b] > t:
                weights.append(adv[order[b]] if t >= 1 else 0.0)
    weights = torch.tensor(weights, dtype=torch.float64)
    for p in params:
        p.grad = None
    out = forward(cap, lens_s, feats)
    loss = weighted_loss(out, pack_targets(cap, lens_s), weights, sum(lens_s) - B)
    loss.backward()
    for p in params:
        if p.grad is not None:
            p.grad.data.clamp_(-grad_clip, grad_clip)
    optimizer.step()
    return float(loss), float(np.mean(rewards)), float(np.mean(base))
