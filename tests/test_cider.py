"""CIDEr-D (K11 ``sn_cider_df`` / ``sn_cider_scores`` + ``icei_b200.cider``): the CPU oracle pinned to hand-derived
answers and, when importable, to coco-caption's scorer; the argument checks that fail before any device call; on the
GPU, per-image, per-order and corpus scores against the oracle, the document-frequency table read back exactly, run-to-run
determinism, the limits, and ``evaluate.validate(..., cider=True)``."""
import math
import random

import numpy as np
import pytest

from oracle import cider as oc


def close(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape
    assert np.all(np.abs(got - want) <= 1e-12 * np.maximum(1.0, np.abs(want))), (got, want)


# ---- the oracle ------------------------------------------------------------------------------------------------------
def test_oracle_one_image_corpus_scores_zero():
    # ref_len = log 1 = 0 and every reference n-gram has df 1: every weight is 0
    mean, scores = oc.corpus_cider([[[1, 2, 3, 4, 5], [1, 2, 9]]], [[1, 2, 3, 4, 5]])
    assert mean == 0.0 and scores.tolist() == [0.0]


def test_oracle_perfect_match_scores_ten_and_seven_and_a_half():
    # 2 images, no shared n-gram: every weight of image 0 is log 2 and its cosines are 1
    mean, scores = oc.corpus_cider([[[1, 2, 3, 4, 5]], [[7, 8]]], [[1, 2, 3, 4, 5], [7]])
    assert scores[0] == pytest.approx(10.0, rel=1e-15, abs=0)
    assert mean == np.mean(scores)
    # 3 tokens: the 4-gram order is empty, so the mean over 4 orders is 3/4
    _, scores = oc.corpus_cider([[[1, 2, 3]], [[7, 8]]], [[1, 2, 3], [7]])
    assert scores[0] == pytest.approx(7.5, rel=1e-15, abs=0)


def test_oracle_length_is_the_bigram_count():
    sc = oc.CiderScorer([[[1]], [[2]]], [[1], [2]])
    sc.compute_doc_freq()
    sc.ref_len = np.log(2.0)
    assert sc.counts2vec(oc.precook([7]))[2] == 0                # one token: no bigram
    assert sc.counts2vec(oc.precook([7, 8, 9]))[2] == 2
    assert sc.counts2vec(oc.precook([], 4))[2] == 0
    sc1 = oc.CiderScorer([[[1]]], [[1]], n=1)
    sc1.ref_len = 0.0
    assert sc1.counts2vec(oc.precook([7, 8, 9], 1))[2] == 0      # n = 1 counts no bigrams at all
    # one-token hypothesis = its one-token reference: unigram cosine 1, delta 0 -> 10 * 1 / 4
    _, scores = oc.corpus_cider([[[7]], [[1, 2]]], [[7], [1]])
    assert scores[0] == pytest.approx(2.5, rel=1e-15, abs=0)
    # bigram counts 1 and 3 (delta 2): the unigram cosine 2 / sqrt(2 * 4) times e^(-4 / 72)
    _, scores = oc.corpus_cider([[[5, 6, 7, 8]], [[1]]], [[5, 6], [1]], n=1)
    assert scores[0] == pytest.approx(10 * 2 / math.sqrt(8), rel=1e-14)   # n = 1: no penalty at all
    _, scores = oc.corpus_cider([[[5, 6, 7, 8]], [[1]]], [[5, 6], [1]], n=2)
    want = 10 * (2 / math.sqrt(8) + 1 / math.sqrt(3)) * math.exp(-4 / 72) / 2
    assert scores[0] == pytest.approx(want, rel=1e-14)
    # sigma scales the penalty
    _, scores = oc.corpus_cider([[[5, 6, 7, 8]], [[1]]], [[5, 6], [1]], n=2, sigma=2.5)
    assert scores[0] == pytest.approx(want * math.exp(4 / 72 - 4 / 12.5), rel=1e-14)


def test_oracle_clipping():
    # "3 3 3 3" against "3 9": unigram min(4w, w) * w = w^2 over norms 4w and w sqrt 2; bigram (3, 3) is not in the
    # reference; bigram counts 3 and 1
    _, scores = oc.corpus_cider([[[3, 9]], [[7, 8]]], [[3, 3, 3, 3], [7]])
    assert scores[0] == pytest.approx(10 * (1 / (4 * math.sqrt(2))) * math.exp(-4 / 72) / 4, rel=1e-14)


def test_oracle_absent_ngram_has_idf_log_n():
    sc = oc.CiderScorer([[[1]], [[7, 8]], [[5]]], [[1, 2], [7], [5]])
    sc.compute_doc_freq()
    sc.ref_len = np.log(3.0)
    vec, norm, _ = sc.counts2vec(oc.precook([2, 2]))
    assert vec[0][(2,)] == 2 * math.log(3.0) and vec[1][(2, 2)] == math.log(3.0)
    # hypothesis "1 2" against "1": the unigram "2" counts in the hypothesis norm -> cosine 1 / sqrt 2
    _, scores = oc.corpus_cider([[[1]], [[7, 8]], [[5]]], [[1, 2], [7], [5]])
    assert scores[0] == pytest.approx(10 * (1 / math.sqrt(2)) * math.exp(-1 / 72) / 4, rel=1e-14)


def test_oracle_document_frequency_counts_an_image_once():
    df = oc.document_frequency([[[1, 2], [2, 1, 2]], [[1]], [[]]], 2)
    assert df == {(1,): 2, (2,): 1, (1, 2): 1, (2, 1): 1}


def test_oracle_empty_sentences():
    mean, scores = oc.corpus_cider([[[1, 2]], [[]], [[3], []]], [[], [1, 2], [3]])
    assert scores[0] == 0.0 and scores[1] == 0.0          # empty hypothesis; reference vectors of norm 0
    assert scores[2] > 0.0                                 # the empty reference adds 0 but counts in the average
    assert mean == np.mean(scores)
    assert oc.corpus_cider([[[]], [[]]], [[1], []])[1].tolist() == [0.0, 0.0]


def _random_corpus(rng, n, vocab, max_len, max_refs, ids=None):
    """Hypotheses and 1..max_refs references cut from a shared "scene" per image, with substitutions, some empty."""
    refs, hyps = [], []
    for _ in range(n):
        scene = [rng.randrange(vocab) for _ in range(max_len)]

        def sent():
            L = rng.randint(0, max_len)
            s0 = rng.randint(0, max_len - L)
            return [w if rng.random() > 0.2 else rng.randrange(vocab) for w in scene[s0:s0 + L]]
        refs.append([sent() for _ in range(rng.randint(1, max_refs))])
        hyps.append(sent())
    if ids is not None:
        refs = [[[ids[w] for w in r] for r in rs] for rs in refs]
        hyps = [[ids[w] for w in h] for h in hyps]
    return refs, hyps


def test_oracle_matches_live_pycocoevalcap():
    cider_mod = pytest.importorskip("pycocoevalcap.cider.cider")
    rng = random.Random(5)
    for vocab, n, sigma in ((4, 4, 6.0), (30, 4, 6.0), (30, 2, 3.0)):
        refs, hyps = _random_corpus(rng, 200, vocab, 20, 5)
        gts = {i: [" ".join(map(str, r)) for r in rs] for i, rs in enumerate(refs)}
        res = {i: [" ".join(map(str, h))] for i, h in enumerate(hyps)}
        mean, scores = cider_mod.Cider(n=n, sigma=sigma).compute_score(gts, res)
        want_mean, want = oc.corpus_cider(refs, hyps, n, sigma)
        assert np.array_equal(np.asarray(scores), want) and mean == want_mean


# ---- argument checks (all before any device call) ---------------------------------------------------------------------
def test_argument_errors_before_device_work():
    from icei_b200.cider import CiderD, corpus_cider
    good_r, good_h = [[[1, 2]]], [[1, 2]]
    for refs, hyps in (([], []), ([[[1, 2]]], [[1, 2], [3]]), ([[[1, 2]], []], [[1, 2], [3]]),
                       ([[[1, 2]]], [[1, -1]]), ([[[-5]]], [[1]]), ([[[1, 2]]], [[1, 2 ** 31]]),
                       ([[[1, 2 ** 63]]], [[1]])):
        with pytest.raises(ValueError):
            corpus_cider(refs, hyps)
    for bad in ([[1.0, 2]], [["a"]], [[1, None]]):
        with pytest.raises(TypeError):
            corpus_cider(good_r, bad)
        with pytest.raises(TypeError):
            corpus_cider([bad], good_h)
    for n in (0, 5, -1, 2.0, True, "4"):
        with pytest.raises(ValueError):
            corpus_cider(good_r, good_h, n=n)
        with pytest.raises(ValueError):
            CiderD(good_r, n=n)
    for sigma in (0.0, -1.0, float("inf"), float("nan"), "6"):
        with pytest.raises(ValueError):
            corpus_cider(good_r, good_h, sigma=sigma)
        with pytest.raises(ValueError):
            CiderD(good_r, sigma=sigma)
    for refs in ([], [[[1]], []], [[[1, -2]]], [[[2 ** 31]]]):
        with pytest.raises(ValueError):
            CiderD(refs)
    with pytest.raises(TypeError):
        CiderD([[[0.5]]])


def test_table_capacity_rule():
    from icei_b200.cider import _capacity
    off = np.array([0, 5, 5, 6, 20])                       # references of 5, 0, 1 and 14 tokens
    grams = {1: 20, 2: 4 + 13, 3: 3 + 12, 4: 2 + 11}
    total = 0
    for n in (1, 2, 3, 4):
        total += grams[n]
        cap = _capacity(off, n)
        assert cap & (cap - 1) == 0 and cap >= 2 * total and cap < 4 * total
    assert _capacity(np.array([0, 0]), 4) == 2


# ---- on the GPU ------------------------------------------------------------------------------------------------------
def _run(refs, hyps, n=4, sigma=6.0, capacity=None):
    """The two kernels on one corpus: (scores, per_order, keys, counts, err) on the host."""
    import torch
    from icei_b200 import cider, ops
    (hyp_tok, hyp_off, ref_tok, ref_off, ref_group), max_len, max_group, ref_off_h, _ = cider._upload(refs, hyps)
    err = torch.full((1,), -1, dtype=torch.int32, device=hyp_off.device)
    keys, counts = ops.cider_df(ref_tok, ref_off, ref_group, n, max_len, max_group,
                                capacity or cider._capacity(ref_off_h, n), err)
    scores, per_order = ops.cider_scores(hyp_tok, hyp_off, ref_tok, ref_off, ref_group, n, sigma, max_len, max_group,
                                         keys, counts)
    return (scores.cpu().numpy(), per_order.cpu().numpy(), keys.cpu().numpy(), counts.cpu().numpy(),
            int(err.item()))


def _table(keys, counts):
    """{n-gram: count} of the occupied slots; every occupied slot holds a distinct key and a positive count."""
    out = {}
    for row, c in zip(keys.tolist(), counts.tolist()):
        if row[0] < 0:
            assert row == [-1, -1, -1, -1] and c == 0
            continue
        k = sum(1 for w in row if w >= 0)
        assert all(w >= 0 for w in row[:k]) and all(w == -1 for w in row[k:])
        g = tuple(row[:k])
        assert g not in out and c > 0
        out[g] = c
    return out


def _check_against_oracle(refs, hyps, n=4, sigma=6.0):
    from icei_b200.cider import CiderD, corpus_cider
    scores, per_order, keys, counts, err = _run(refs, hyps, n, sigma)
    want_mean, want = oc.corpus_cider(refs, hyps, n, sigma)
    assert err == 0
    close(scores, want)
    close(per_order[:, :n], oc.per_order(refs, hyps, n, sigma))
    assert not per_order[:, n:].any()
    assert _table(keys, counts) == oc.document_frequency(refs, n)
    mean, got = corpus_cider(refs, hyps, n, sigma)
    assert isinstance(mean, float) and got.dtype == np.float64
    close(got, want)
    close(mean, want_mean)
    assert mean == np.mean(got)
    mean_d, got_d = CiderD(refs, n, sigma).compute_score(hyps)
    assert np.array_equal(got_d, got) and mean_d == mean
    return got


EDGE = {
    "one_image": ([[[1, 2, 3, 4, 5], [1, 2, 9]]], [[1, 2, 3, 4, 5]]),
    "perfect_5": ([[[1, 2, 3, 4, 5]], [[7, 8]]], [[1, 2, 3, 4, 5], [7]]),
    "perfect_3": ([[[1, 2, 3]], [[7, 8]]], [[1, 2, 3], [7]]),
    "one_token": ([[[7]], [[1, 2]]], [[7], [1]]),
    "length_penalty": ([[[5, 6, 7, 8]], [[1]]], [[5, 6], [1]]),
    "clipping": ([[[3, 9]], [[7, 8]]], [[3, 3, 3, 3], [7]]),
    "absent_ngram": ([[[1]], [[7, 8]], [[5]]], [[1, 2], [7], [5]]),
    "empty_sentences": ([[[1, 2]], [[]], [[3], []]], [[], [1, 2], [3]]),
    "all_refs_empty": ([[[]], [[]]], [[1], []]),
    "repeats": ([[[4, 4, 4, 4, 4, 4], [4, 4, 5, 4, 4]], [[4]]], [[4, 4, 4, 4, 4], [4, 4]]),
    "big_ids": ([[[0, 2 ** 31 - 1, 2 ** 31 - 1, 0]], [[2 ** 31 - 1, 5]]], [[0, 2 ** 31 - 1, 0], [2 ** 31 - 1]]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(EDGE))
def test_edge_cases_match_oracle(case):
    refs, hyps = EDGE[case]
    got = _check_against_oracle(refs, hyps)
    if case == "perfect_5":
        assert got[0] == pytest.approx(10.0, rel=1e-12)
    if case == "perfect_3":
        assert got[0] == pytest.approx(7.5, rel=1e-12)
    if case == "one_image":
        assert got.tolist() == [0.0]
    for n in (1, 2, 3):
        _check_against_oracle(refs, hyps, n)


@pytest.mark.gpu
@pytest.mark.parametrize("n,sigma", [(1, 6.0), (2, 6.0), (3, 6.0), (4, 6.0), (4, 2.5), (2, 0.75)])
def test_random_ragged_corpora_match_oracle(n, sigma):
    rng = random.Random(100 * n + int(4 * sigma))
    # small vocabularies so that every order matches, mapped to ids spread over the whole int32 range
    ids = [2 ** 31 - 1 - 7919 * v for v in range(9)] + [0]
    refs, hyps = _random_corpus(rng, 700, 10, 24, 7, ids)
    assert any(len(h) == 0 for h in hyps) and any(len(r) == 0 for rs in refs for r in rs)
    got = _check_against_oracle(refs, hyps, n, sigma)
    assert (got > 0).mean() > 0.5
    refs, hyps = _random_corpus(rng, 300, 200, 20, 5)
    _check_against_oracle(refs, hyps, n, sigma)


@pytest.mark.gpu
def test_document_frequency_table_under_heavy_probing():
    """A table with barely more slots than distinct n-grams: long probe chains, the same counts and scores."""
    from icei_b200._lib import SnError
    from icei_b200.cider import _check_df
    rng = random.Random(7)
    refs, hyps = _random_corpus(rng, 480, 40, 16, 5)
    want_df = oc.document_frequency(refs, 4)
    distinct = len(want_df)
    tight = 1 << (distinct - 1).bit_length()               # the smallest power of two that holds them all
    assert distinct > 0.95 * tight
    scores_ref, per_ref, _, _, err = _run(refs, hyps)
    assert err == 0
    scores, per_order, keys, counts, err = _run(refs, hyps, capacity=tight)
    assert err == 0
    assert _table(keys, counts) == want_df
    assert np.array_equal(scores, scores_ref) and np.array_equal(per_order, per_ref)
    # too small: the kernel reports it and the host raises
    *_, err = _run(refs, hyps, capacity=tight // 2)
    assert err & 1
    with pytest.raises(SnError, match="full"):
        _check_df(err)
    _check_df(0)


@pytest.mark.gpu
def test_runs_are_bitwise_identical_and_ciderd_reuse_equals_corpus_cider():
    from icei_b200.cider import CiderD, corpus_cider
    rng = random.Random(21)
    refs, hyps = _random_corpus(rng, 3000, 50, 20, 5)
    hyps2 = [h[::-1] for h in hyps]
    m1, s1 = corpus_cider(refs, hyps)
    m2, s2 = corpus_cider(refs, hyps)
    assert m1 == m2 and np.array_equal(s1, s2)
    scorer = CiderD(refs)
    for h, (m, s) in ((hyps, (m1, s1)), (hyps2, corpus_cider(refs, hyps2)), (hyps, (m1, s1))):
        md, sd = scorer.compute_score(h)
        assert md == m and np.array_equal(sd, s)
    p1 = _run(refs, hyps)[1]
    assert np.array_equal(p1, _run(refs, hyps)[1])
    with pytest.raises(ValueError):
        scorer.compute_score(hyps[:-1])
    with pytest.raises(ValueError):
        scorer.compute_score(hyps[:-1] + [[-3]])


@pytest.mark.gpu
def test_large_image_group_uses_opt_in_shared_memory():
    """100 references of up to 200 tokens: 80 KB of ids for one CTA (above the 48 KB default)."""
    rng = random.Random(3)
    refs = [[[rng.randrange(5) for _ in range(rng.randint(150, 200))] for _ in range(100)], [[1, 2, 3]]]
    hyps = [[rng.randrange(5) for _ in range(150)], [1, 2, 3]]
    _check_against_oracle(refs, hyps)


@pytest.mark.gpu
def test_limits_are_rejected_before_launch():
    from icei_b200._lib import SnError
    from icei_b200.cider import CiderD, corpus_cider
    with pytest.raises(SnError, match="256"):
        corpus_cider([[[1, 2]]], [[1] * 257])
    with pytest.raises(SnError, match="256"):
        corpus_cider([[[1, 2], [3] * 257]], [[1, 2]])
    with pytest.raises(SnError, match="256"):
        CiderD([[[1, 2]]]).compute_score([[1] * 257])
    corpus_cider([[[1, 2]]], [[1] * 256])
    with pytest.raises(SnError, match="shared memory"):
        corpus_cider([[[1] * 256] * 250], [[1, 2]])                  # 64 000 ids for one image
    with pytest.raises(SnError, match="shared memory"):
        CiderD([[[1] * 256] * 250])


# ---- evaluate.validate(..., cider=True) --------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["factored", "nic", "factored_att"])
def test_validate_cider(kind):
    import torch
    import icei_b200 as sn
    from icei_b200.evaluate import validate
    from oracle import port
    V, E, H, F, A, D = 331, 28, 32, 40, 24, 48
    torch.manual_seed(0)
    if kind == "factored":
        dec, kw, att = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0), {"mode": "happy"}, False
    elif kind == "nic":
        dec, kw, att = sn.DecoderRNN(E, H, V, 1, dropout=0.0), {}, False
    else:
        dec, kw, att = sn.DecoderFactoredLSTMAtt(A, E, H, F, V, 1, feature_size=D, dropout=0.0), {"mode": "sad"}, True
    port.sharpen_for_decode(dec, scale=20.0, end_bias=-5.0)      # captions of real words, not <end> everywhere
    dec = dec.cuda().eval()
    data = []
    for seed, B in ((1, 7), (2, 12)):
        cap, lens, feats = port.synthetic_batch(B, 9, V, E=None if att else E, feat_shape=(3, 3, D) if att else None,
                                                ragged=True, seed=seed)
        data.append((feats.cuda(), cap.cuda(), lens, [[c[:l].tolist()] for c, l in zip(cap, lens)]))
    hyps = validate(dec, data, 1, 2, **kw)["hypotheses"]
    # references sharing n-grams with the arg-max hypotheses: a copy with one id replaced, a prefix, the caption
    rng = random.Random(0)
    batches, i = [], 0
    for feats, cap, lens, caps in data:
        all_caps = []
        for c in caps:
            h = hyps[i]
            i += 1
            sub = list(h)
            if sub:
                sub[rng.randrange(len(sub))] = rng.randrange(3, V)
            all_caps.append([[1] + sub + [2], [1] + h[: len(h) // 2] + [2], c[0]])
        batches.append((feats, cap, lens, all_caps))
    plain = validate(dec, batches, 1, 2, **kw)
    assert "cider" not in plain
    res = validate(dec, batches, 1, 2, cider=True, **kw)
    assert set(res) == set(plain) | {"cider"}
    assert all(res[k] == plain[k] for k in plain)
    want, _ = oc.corpus_cider(res["references"], res["hypotheses"])
    close(res["cider"], want)
    assert want > 0.0
    both = validate(dec, batches, 1, 2, cider=True, bleu_weights=(0.25,) * 4, **kw)
    assert both["cider"] == res["cider"] and "bleu" in both
    with pytest.raises(ValueError):
        validate(dec, batches[:1] + [batches[1][:3] + (None,)], 1, 2, cider=True, **kw)
