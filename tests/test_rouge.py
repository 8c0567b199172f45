"""ROUGE-L (K13 ``sn_rouge_l`` / ``sn_rouge_l_rows`` + ``icei_b200.rouge``): the CPU oracle pinned to hand-derived
answers, to a brute-force LCS and, when importable, to coco-caption's scorer; the argument checks that fail before any
device call; on the GPU, per-image scores bitwise equal to the oracle's (edge cases, ragged corpora across the word
boundaries of the bit vector, dense and sparse vocabularies, 1 to 40 references), run-to-run identity, ``RougeL`` reuse,
the rows form, ``scst_step`` with a ROUGE-L reward, the limits, and ``evaluate.validate(..., rouge=True)``."""
import itertools
import random

import numpy as np
import pytest
import torch

from oracle import rouge as orouge

START, END = 1, 2


# ---- the oracle ------------------------------------------------------------------------------------------------------
def test_oracle_hand_derived_values():
    def score(refs, hyp):
        mean, scores = orouge.corpus_rouge([refs], [hyp])
        assert mean == scores[0] and scores.dtype == np.float64
        return scores[0]
    assert score([[1, 3, 5, 4]], [1, 2, 3, 4]) == 0.75                          # LCS 3 of 4 and 4: p = r = 3/4
    assert score([[1, 2, 3, 4]], [1, 2]) == 0.6288659793814433                  # p = 1, r = 1/2
    assert score([[], [5, 6]], [5]) == 0.6288659793814433                       # the empty reference adds LCS 0
    assert score([[1, 2, 3, 9, 9, 9], [1]], [1, 2, 3]) == 1.0                   # p from one reference, r from the other
    assert score([[1, 2], [7]], []) == 0.0                                      # empty hypothesis, non-empty refs
    assert score([[1, 2], []], []) == 1.0                                       # "" matches only ""
    assert score([[]], [4, 5]) == 0.0
    assert score([[9, 9]], [1, 2]) == 0.0                                       # no common token
    assert score([[-3, 7]], [-3, 7]) == 1.0                                     # ids are only compared
    assert orouge.my_lcs("".split(" "), "".split(" ")) == 1
    mean, scores = orouge.corpus_rouge([[[1, 3, 5, 4]], [[1, 2, 3, 4]]], [[1, 2, 3, 4], [1, 2]])
    assert scores.tolist() == [0.75, 0.6288659793814433] and mean == np.mean(scores)


def _brute_lcs(a, b):
    if len(a) > len(b):
        a, b = b, a
    for k in range(len(a), 0, -1):
        for sub in itertools.combinations(a, k):
            it = iter(b)
            if all(any(x == y for y in it) for x in sub):                      # sub is a subsequence of b
                return k
    return 0


def test_oracle_lcs_matches_brute_force():
    rng = random.Random(11)
    for _ in range(1500):
        vocab = rng.choice((2, 3, 6))
        a = [rng.randrange(vocab) for _ in range(rng.randint(0, 8))]
        b = [rng.randrange(vocab) for _ in range(rng.randint(0, 8))]
        assert orouge.my_lcs(a, b) == _brute_lcs(a, b) == orouge.my_lcs(b, a), (a, b)


def _corpus(rng, n, vocab, lengths, n_refs, ids=None):
    """Per image a "scene" of vocabulary ids; the hypothesis and 1..n_refs references are spans of it of a length drawn
    from ``lengths`` (tokens past the scene are fresh ids), with 20 % of the ids replaced.  ``ids`` maps the vocabulary
    to other integers."""
    refs, hyps = [], []
    longest = max(lengths)
    for _ in range(n):
        scene = [rng.randrange(vocab) for _ in range(longest + 8)]

        def sent():
            L = rng.choice(lengths)
            s0 = rng.randint(0, len(scene) - L)
            return [w if rng.random() > 0.2 else rng.randrange(vocab) for w in scene[s0:s0 + L]]
        refs.append([sent() for _ in range(rng.randint(1, n_refs))])
        hyps.append(sent())
    if ids is not None:
        refs = [[[ids[w] for w in r] for r in rs] for rs in refs]
        hyps = [[ids[w] for w in h] for h in hyps]
    return refs, hyps


def test_oracle_matches_live_pycocoevalcap():
    rouge_mod = pytest.importorskip("pycocoevalcap.rouge.rouge")
    rng = random.Random(5)
    for vocab in (2, 4, 30):
        refs, hyps = _corpus(rng, 200, vocab, list(range(0, 21)), 5)
        gts = {i: [" ".join(map(str, r)) for r in rs] for i, rs in enumerate(refs)}
        res = {i: [" ".join(map(str, h))] for i, h in enumerate(hyps)}
        mean, scores = rouge_mod.Rouge().compute_score(gts, res)
        want_mean, want = orouge.corpus_rouge(refs, hyps)
        assert np.array_equal(np.asarray(scores), want) and mean == want_mean


# ---- argument checks (all before any device call) ---------------------------------------------------------------------
def test_argument_errors_before_device_work():
    import icei_b200 as sn
    from icei_b200.rouge import RougeL, corpus_rouge
    good_r, good_h = [[[1, 2]]], [[1, 2]]
    for refs, hyps in (([], []), ([[[1, 2]]], [[1, 2], [3]]), ([[[1, 2]], []], [[1, 2], [3]]),
                       ([[[1, 2]]], [[1, 2 ** 31]]), ([[[1, -2 ** 31 - 1]]], [[1]]), ([[[1, 2 ** 63]]], [[1]])):
        with pytest.raises(ValueError):
            corpus_rouge(refs, hyps)
    for bad in ([[1.0, 2]], [["a"]], [[1, None]]):
        with pytest.raises(TypeError):
            corpus_rouge(good_r, bad)
        with pytest.raises(TypeError):
            corpus_rouge([bad], good_h)
    for refs in ([], [[[1]], []], [[[2 ** 31]]]):
        with pytest.raises(ValueError):
            RougeL(refs)
    with pytest.raises(TypeError):
        RougeL([[[0.5]]])
    from icei_b200._lib import SnError
    with pytest.raises(SnError, match="256"):
        corpus_rouge([[[1, 2]]], [[1] * 257])
    with pytest.raises(SnError, match="256"):
        corpus_rouge([[[1, 2], [3] * 257]], [[1, 2]])
    with pytest.raises(SnError, match="256"):
        RougeL([[[1, 2], [3] * 257]])
    scorer = object.__new__(sn.rouge.RougeL)          # the checks run before the object's device state is touched
    scorer.n_img, scorer._ref_max_len = 4, 2
    with pytest.raises(ValueError):
        scorer.compute_score([[1]] * 3)
    with pytest.raises(TypeError):
        scorer.compute_score([[1], [2], [3], [4.5]])
    with pytest.raises(ValueError):
        scorer.compute_score([[1], [2], [3], [2 ** 40]])
    with pytest.raises(SnError, match="256"):
        scorer.compute_score([[1], [2], [3], [4] * 257])
    seqs = torch.zeros(3, 5, dtype=torch.int64)
    lens = torch.full((3,), 3, dtype=torch.int64)
    for args in ((seqs[0], lens, [0, 1, 2]), (seqs, lens[:2], [0, 1, 2]), (seqs, lens, [0, 1]), (seqs, lens, [0, 4, 1]),
                 (seqs, lens, [0, -1, 1]), (seqs, lens, [0.0, 1.0, 2.0])):
        with pytest.raises(ValueError):
            scorer.score_samples(*args, START, END)


# ---- on the GPU ------------------------------------------------------------------------------------------------------
def _check_against_oracle(refs, hyps):
    """corpus_rouge and RougeL.compute_score bitwise equal to the oracle, per image and for the corpus."""
    from icei_b200.rouge import RougeL, corpus_rouge
    want_mean, want = orouge.corpus_rouge(refs, hyps)
    mean, got = corpus_rouge(refs, hyps)
    assert isinstance(mean, float) and got.dtype == np.float64
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, [(int(i), got[i], want[i], hyps[i], refs[i]) for i in bad[:3]]
    assert mean == want_mean
    mean_r, got_r = RougeL(refs).compute_score(hyps)
    assert np.array_equal(got_r, got) and mean_r == mean
    return got


EDGE = {
    "lcs_3_of_4": ([[[1, 3, 5, 4]]], [[1, 2, 3, 4]], [0.75]),
    "prefix": ([[[1, 2, 3, 4]]], [[1, 2]], [0.6288659793814433]),
    "empty_ref_and_match": ([[[], [5, 6]]], [[5]], [0.6288659793814433]),
    "p_and_r_from_two_refs": ([[[1, 2, 3, 9, 9, 9], [1]]], [[1, 2, 3]], [1.0]),
    "empty_hyp": ([[[1, 2], [7]], [[1, 2], []], [[]], [[3]]], [[], [], [], [3]], [0.0, 1.0, 1.0, 1.0]),
    "empty_ref_only": ([[[]], [[]]], [[4, 5], [4]], [0.0, 0.0]),
    "no_common_token": ([[[9, 9]]], [[1, 2]], [0.0]),
    "repeats": ([[[4, 4, 4, 4, 4, 4], [4, 4, 5, 4, 4]], [[4]]], [[4, 4, 4, 4, 4], [4, 4]], None),
    "negative_and_big_ids": ([[[-2 ** 31, 2 ** 31 - 1, -1, 0]], [[0, -1]]], [[-2 ** 31, -1, 0, 2 ** 31 - 1], [-1]], None),
    "one_token": ([[[7]], [[7, 8]]], [[7], [8]], [1.0, None]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(EDGE))
def test_edge_cases_match_oracle(case):
    refs, hyps, pinned = EDGE[case]
    got = _check_against_oracle(refs, hyps)
    for g, p in zip(got.tolist(), pinned or []):
        assert p is None or g == p


BOUNDARY = [0, 1, 2, 31, 32, 33, 63, 64, 65]


@pytest.mark.gpu
@pytest.mark.parametrize("vocab", [2, 10000])
def test_random_ragged_corpora_match_oracle(vocab):
    rng = random.Random(vocab)
    # ids spread over the whole int32 range, negatives included, and 0: the kernel's filler for hypothesis positions
    # past the end, so references full of 0 exercise the bits beyond the hypothesis
    ids = [2 ** 31 - 1 - 7919 * v for v in range(vocab // 2)] + [-2 ** 31 + 104729 * v for v in range(vocab - vocab // 2)]
    ids[0] = 0
    # lengths on both sides of each 32-bit word boundary up to three words, and random ones
    refs, hyps = _corpus(rng, 400, vocab, BOUNDARY + list(range(3, 60)), 6, ids)
    assert any(len(h) == 0 for h in hyps) and any(len(r) == 0 for rs in refs for r in rs)
    got = _check_against_oracle(refs, hyps)
    assert (got > 0).mean() > 0.5 and (got < 1).mean() > 0.5
    # the longest sentences: 1..3 references of 96..256 tokens
    refs, hyps = _corpus(rng, 24, vocab, [95, 96, 97, 127, 128, 129, 191, 192, 193, 224, 255, 256], 3, ids)
    _check_against_oracle(refs, hyps)
    # up to 40 references per image
    refs, hyps = _corpus(rng, 60, vocab, BOUNDARY + list(range(3, 25)), 40, ids)
    assert max(len(rs) for rs in refs) >= 35
    _check_against_oracle(refs, hyps)


@pytest.mark.gpu
def test_runs_are_bitwise_identical_and_rougel_reuse_equals_corpus_rouge():
    from icei_b200.rouge import RougeL, corpus_rouge
    rng = random.Random(21)
    refs, hyps = _corpus(rng, 3000, 50, list(range(0, 21)), 5)
    hyps2 = [h[::-1] for h in hyps]
    m1, s1 = corpus_rouge(refs, hyps)
    m2, s2 = corpus_rouge(refs, hyps)
    assert m1 == m2 and np.array_equal(s1, s2)
    scorer = RougeL(refs)
    for h, (m, s) in ((hyps, (m1, s1)), (hyps2, corpus_rouge(refs, hyps2)), (hyps, (m1, s1))):
        md, sd = scorer.compute_score(h)
        assert md == m and np.array_equal(sd, s)
    want_mean, want = orouge.corpus_rouge(refs, hyps2)
    assert np.array_equal(scorer.compute_score(hyps2)[1], want)


@pytest.mark.gpu
def test_oversized_image_gets_nan():
    """The kernel's own guard: an image whose sentences exceed the declared maximum scores NaN, the others do not."""
    from icei_b200 import ops, rouge
    refs, hyps = [[[1, 2]], [[1, 2, 3, 4]], [[5]]], [[1, 2], [1], [5, 6, 7]]
    views, max_len = rouge._upload(refs, hyps)
    assert max_len == 4
    got = ops.rouge_l(*views, 2, rouge.BETA2).cpu().numpy()
    assert got[0] == 1.0 and np.isnan(got[1]) and np.isnan(got[2])


def _rows(rng, R, ld, V):
    """seqs [R, ld] as sample_captions writes them (<start> in column 0), lengths, and the hypotheses they hold: rows
    of only <start>, rows ending in <end>, rows cut by the length limit."""
    seqs = torch.zeros(R, ld, dtype=torch.int64)
    lens = torch.zeros(R, dtype=torch.int64)
    hyps = []
    for r in range(R):
        L = 1 if r % 7 == 0 else rng.randint(1, ld)
        body = [rng.randrange(3, V) for _ in range(L - 1)]
        if L >= 2 and rng.random() < 0.7:
            body[-1] = END
        seqs[r, 0] = START
        seqs[r, 1:L] = torch.tensor(body, dtype=torch.int64)
        seqs[r, L:] = rng.randrange(3, V)                       # what lies past the length is never read
        lens[r] = L
        hyps.append(body[:-1] if body and body[-1] == END else body)
    return seqs, lens, hyps


@pytest.mark.gpu
def test_rows_form_vs_compute_score_and_oracle():
    import icei_b200 as sn
    rng = random.Random(1)
    V, n_img = 12, 16
    refs, _ = _corpus(rng, n_img, V - 3, BOUNDARY[:4] + list(range(3, 12)), 4, ids=list(range(3, V)))
    scorer = sn.rouge.RougeL(refs)
    for ld in (11, 40, 257):
        seqs, lens, hyps = _rows(rng, 48, ld, V)
        # identity ids: bitwise equal to compute_score on the same hypotheses
        got = scorer.score_samples(seqs[:n_img].cuda(), lens[:n_img].cuda(), list(range(n_img)), START, END)
        _, want = scorer.compute_score(hyps[:n_img])
        assert got.dtype == torch.float64 and got.is_cuda and np.array_equal(got.cpu().numpy(), want)
        # repeated, shuffled ids
        ids = [rng.randrange(n_img) for _ in range(48)]
        got = scorer.score_samples(seqs.cuda(), lens.cuda(), np.array(ids), START, END).cpu().numpy()
        assert np.array_equal(got, orouge.sample_scores(refs, ids, hyps))
    assert scorer.score_samples(seqs[:0], lens[:0], [], START, END).numel() == 0


@pytest.mark.gpu
def test_scst_step_with_rougel_reward():
    """scst_step takes a RougeL as its scorer: the mean reward it returns is the oracle's mean ROUGE-L of the samples
    drawn with the same seed (per-sample rewards bitwise; the mean within rounding of a different summation order)."""
    import icei_b200 as sn
    from oracle import port
    V, E, H, F, max_len = 40, 24, 32, 24, 7
    torch.manual_seed(2)
    ref = port.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0, max_seq_length=max_len)
    port.lively_weights(ref, out_gain=3.0, end_bias=1.0)
    dec = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0, max_seq_length=max_len)
    dec.load_state_dict(ref.state_dict())
    dec = dec.cuda().train()
    rng = random.Random(3)
    refs = [[[rng.randrange(3, V) for _ in range(rng.randint(2, 8))] for _ in range(rng.randint(1, 4))]
            for _ in range(10)]
    ids = [7, 2, 2, 9, 0, 4]
    feats = torch.randn(len(ids), E, generator=torch.Generator().manual_seed(5)).cuda()
    scorer = sn.rouge.RougeL(refs)
    opt = sn.FusedClampAdam(dec, lr=1e-3, grad_clip=0.5)
    n, seed = 4, 17
    for baseline in ("mean", "greedy"):
        with torch.no_grad():
            seqs, lens, _ = dec.sample_captions(feats, START, END, n=n, seed=seed, mode="happy")
        hyps = []
        for s, L in zip(seqs.cpu().tolist(), lens.cpu().tolist()):
            h = s[1:L]
            hyps.append(h[:-1] if h and h[-1] == END else h)
        want = orouge.sample_scores(refs, np.repeat(ids, n), hyps)
        assert np.array_equal(scorer.score_samples(seqs, lens, np.repeat(ids, n), START, END).cpu().numpy(), want)
        before = [p.detach().clone() for p in dec.parameters()]
        loss, rmean, bmean = sn.scst.scst_step(dec, opt, scorer, feats, ids, START, END, mode="happy", n=n,
                                               baseline=baseline, seed=seed)
        assert abs(float(rmean) - float(np.mean(want))) <= 1e-15 * max(1.0, float(np.mean(want)))
        assert 0.0 < float(rmean) < 1.0 and np.isfinite(float(loss)) and np.isfinite(float(bmean))
        assert any(not torch.equal(a, b) for a, b in zip(before, dec.parameters()))


@pytest.mark.gpu
def test_limits_are_rejected_before_launch():
    from icei_b200._lib import SnError
    from icei_b200.rouge import RougeL
    # the host-side checks of the same limit are in test_argument_errors_before_device_work
    scorer = RougeL([[[1, 2]]])
    with pytest.raises(SnError, match="256"):
        scorer.compute_score([[1] * 257])
    seqs = torch.full((1, 258), 1, dtype=torch.int64, device="cuda")
    with pytest.raises(SnError, match="256"):
        scorer.score_samples(seqs, torch.full((1,), 258, dtype=torch.int64, device="cuda"), [0], START, END)
    _check_against_oracle([[[1] * 256, [2] * 256]], [[1, 2] * 128])
    _check_against_oracle([[[1, 2]]], [[1] * 256])


# ---- evaluate.validate(..., rouge=True) --------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["factored", "nic", "factored_att"])
def test_validate_rouge(kind):
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
    # references sharing subsequences with the arg-max hypotheses: a copy with one id replaced, a prefix, the caption
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
    assert "rouge_l" not in plain
    res = validate(dec, batches, 1, 2, rouge=True, **kw)
    assert set(res) == set(plain) | {"rouge_l"}
    assert all(res[k] == plain[k] for k in plain)
    want, _ = orouge.corpus_rouge(res["references"], res["hypotheses"])
    assert res["rouge_l"] == want and 0.0 < want <= 1.0
    both = validate(dec, batches, 1, 2, rouge=True, cider=True, bleu_weights=(0.25,) * 4, **kw)
    assert both["rouge_l"] == res["rouge_l"] and "bleu" in both and "cider" in both
    with pytest.raises(ValueError):
        validate(dec, batches[:1] + [batches[1][:3] + (None,)], 1, 2, rouge=True, **kw)
