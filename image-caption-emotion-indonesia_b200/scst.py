"""Self-critical sequence training on CIDEr-D (Rennie et al. 2017; the "new self-critical" baseline of Luo 2020): the
fine-tuning phase that follows cross-entropy training of a captioner.  One step samples captions (K12), scores them
against the training references on the device (K11, ``CiderD.score_samples``), and trains on the sampled captions with
the reward-weighted caption loss (K5 ``token_weights``) and the optimizer.  The only host round trip is one copy of the
sample lengths, for the length sort that packing needs."""
import numpy as np
import torch

from .packing import get_plan

BASELINES = ("mean", "greedy")


def sort_by_length(lengths):
    """Stable order of the rows by length, descending (the ``pack_padded_sequence`` contract)."""
    lengths = [int(l) for l in lengths]
    return sorted(range(len(lengths)), key=lambda r: -lengths[r])


def advantages(rewards, n, baseline, greedy_rewards=None):
    """Per-sample advantage, image-major rows (row i * n + j = sample j of image i).
    "mean": the reward minus the mean reward of the image's other n - 1 samples; "greedy": the reward minus the reward
    of the image's greedy caption (``greedy_rewards`` [n_img]).  Returns (advantage [R], baseline [R]), in the
    dtype of ``rewards`` (on its device)."""
    r = rewards.view(-1, n)
    if baseline == "mean":
        base = (r.sum(1, keepdim=True) - r) / (n - 1)
    else:
        base = greedy_rewards.view(-1, 1).expand_as(r)
    return (r - base).reshape(-1), base.reshape(-1)


def token_weights(adv_sorted, plan):
    """float32 [N] in packed row order for samples sorted by length: row (b, t) gets adv_sorted[b] for t >= 1 and 0 for
    t = 0, the image step whose target is <start>."""
    d = plan.dev(adv_sorted.device) if adv_sorted.is_cuda else {
        "row_b": torch.from_numpy(plan.row_b_np), "row_t": torch.from_numpy(plan.row_t_np)}
    w = adv_sorted.to(torch.float32).index_select(0, d["row_b"].long())
    return torch.where(d["row_t"] > 0, w, torch.zeros_like(w))


def scst_step(decoder, optimizer, cider, features, image_ids, start_token, end_token, mode="factual", n=5,
              baseline="mean", temperature=1.0, seed=0):
    """One self-critical training step on CIDEr-D for the images ``features [n_img, E]``.

    1. ``n`` captions per image from ``decoder.sample_captions`` (seed ``seed``, dropout off, no gradient).
    2. ``baseline="greedy"`` (Rennie): the greedy caption of each image, from the same sampler.
    3. Rewards: ``cider.score_samples`` against the references of training images ``image_ids`` (host sequence of
       n_img positions in the corpus ``cider`` was built from; the loader has to yield each image's index).
    4. Advantages on the device (``advantages``): "mean" (Luo, needs n >= 2) or "greedy".
    5. One device-to-host copy of the lengths; rows stable-sorted by length, descending; samples, features and
       advantages permuted on the device.
    6. Token weights (``token_weights``): the sample's advantage on every step but the image step.
    7. ``decoder.forward_loss(seqs, lengths, features, teacher_forcing_ratio=1.0, token_weights=w,
       n_global=sum(L_b - 1))`` after ``optimizer.zero_grad()``: loss = -sum_b adv_b log p(sample_b) / #drawn tokens.
    8. ``optimizer.step()``.

    The sampler has no dropout, while the loss forward applies the decoder's dropout as the caller set it (``train()``
    / ``eval()``).  ``features`` are constants: no feature gradient is computed.  Vary ``seed`` from step to step (e.g.
    the iteration number) to draw fresh samples.  Returns device scalars (loss, mean sample reward, mean baseline).
    Raises ValueError for an unknown baseline, "mean" with n < 2 and ``image_ids`` of the wrong length, and as
    ``sample_captions`` for its arguments, all before any device work."""
    if baseline not in BASELINES:
        raise ValueError("baseline must be one of %s; got %r" % (BASELINES, baseline))
    if baseline == "mean" and not (isinstance(n, int) and n >= 2):
        raise ValueError('baseline "mean" needs n >= 2 samples per image; got n = %r' % (n,))
    feats = features.detach().reshape(features.shape[0], -1)
    n_img = feats.shape[0]
    ids = np.asarray(image_ids)
    if ids.shape != (n_img,):
        raise ValueError("%d image ids for %d images" % (ids.size, n_img))
    with torch.no_grad():
        seqs, lengths, _ = decoder.sample_captions(feats, start_token, end_token, n=n, temperature=temperature,
                                                   seed=seed, mode=mode)
        rewards = cider.score_samples(seqs, lengths, np.repeat(ids, n), start_token, end_token)
        greedy_rewards = None
        if baseline == "greedy":
            gseqs, glens, _ = decoder.sample_captions(feats, start_token, end_token, n=1, seed=seed, mode=mode,
                                                      greedy=True)
            greedy_rewards = cider.score_samples(gseqs, glens, ids, start_token, end_token)
        adv, base = advantages(rewards, n, baseline, greedy_rewards)
        lens_h = lengths.cpu().tolist()                            # the step's one device-to-host copy
        order = sort_by_length(lens_h)
        lens_sorted = [lens_h[r] for r in order]
        idx = torch.tensor(order, dtype=torch.int64).to(seqs.device, non_blocking=True)
        seqs_p = seqs.index_select(0, idx)
        feats_p = feats.index_select(0, torch.div(idx, n, rounding_mode="floor"))
        plan = get_plan(lens_sorted)
        w = token_weights(adv.index_select(0, idx), plan)
    optimizer.zero_grad()
    loss, _ = decoder.forward_loss(seqs_p, lens_sorted, feats_p, teacher_forcing_ratio=1.0, mode=mode,
                                   token_weights=w, n_global=sum(lens_sorted) - len(lens_sorted))
    optimizer.step()
    return loss, rewards.mean(), base.mean()
