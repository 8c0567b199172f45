"""Corpus BLEU (K10 ``sn_bleu_counts`` + ``icei_b200.bleu``): the CPU oracle pinned to nltk's documented answers and to
hand-derived edge cases; the argument checks that fail before any device call; on the GPU, the kernel's per-hypothesis
integers and the final scores against the oracle, exactly, and ``evaluate.validate(..., bleu_weights=...)``."""
import math
import random
import sys
import warnings

import pytest

from oracle import bleu as ob

W4 = [(1.0,), (0.5, 0.5), (1 / 3, 1 / 3, 1 / 3), (0.25, 0.25, 0.25, 0.25)]

# nltk/translate/bleu_score.py docstring examples (sentence_bleu / corpus_bleu)
HYP1 = ("It is a guide to action which ensures that the military always obeys the commands of the party").split()
REF1A = "It is a guide to action that ensures that the military will forever heed Party commands".split()
REF1B = ("It is the guiding principle which guarantees the military forces always being under the command of the "
         "Party").split()
REF1C = "It is the practical guide for the army always to heed the directions of the party".split()
HYP2 = "he read the book because he was interested in world history".split()
REF2A = "he was interested in world history because he read the book".split()


# ---- the oracle ------------------------------------------------------------------------------------------------------
def test_oracle_reproduces_nltk_sentence_bleu_docstring():
    assert ob.sentence_bleu([REF1A, REF1B, REF1C], HYP1) == 0.5045666840058485


def test_oracle_reproduces_nltk_corpus_bleu_docstring():
    assert ob.corpus_bleu([[REF1A, REF1B, REF1C], [REF2A]], [HYP1, HYP2]) == 0.5920778868801042


def test_oracle_clipping():
    # nltk's modified_precision docstring: "the" 7 times against refs holding it at most twice -> 2/7
    ref1 = "the cat is on the mat".split()
    ref2 = "there is a cat on the mat".split()
    assert ob.modified_precision([ref1, ref2], ["the"] * 7, 1) == (2, 7)
    # "the the the the" vs "the cat": unigram 1/4, bigram "the the" 0/3
    assert ob.modified_precision([[3, 9]], [3, 3, 3, 3], 1) == (1, 4)
    assert ob.modified_precision([[3, 9]], [3, 3, 3, 3], 2) == (0, 3)
    assert ob.modified_precision([[3, 3, 9], [3, 9, 3, 3, 3]], [3, 3, 3, 3], 1) == (4, 4)
    assert ob.modified_precision([[3, 3, 9], [3, 9, 3, 3, 3]], [3, 3, 3, 3], 2) == (2, 3)


def test_oracle_short_hypothesis_denominator_adds_one():
    # a hypothesis shorter than n contributes 1 to the order-n denominator (max(1, .)), 0 to the numerator
    assert [ob.modified_precision([[7, 8]], [7, 8], n) for n in (1, 2, 3, 4)] == [(2, 2), (1, 1), (0, 1), (0, 1)]
    assert ob.corpus_bleu([[[7, 8]]], [[7, 8]], (0.5, 0.5)) == 1.0
    # orders 3 and 4 have no match: their precision is sys.float_info.min (method0)
    want = math.exp(0.25 * 2 * math.log(sys.float_info.min))
    assert ob.corpus_bleu([[[7, 8]]], [[7, 8]]) == pytest.approx(want, rel=1e-12)


def test_oracle_empty_hypothesis():
    assert ob.brevity_penalty(3, 0) == 0
    assert ob.corpus_bleu([[[1, 2, 3]]], [[]]) == 0
    assert ob.sentence_stats([[5, 6]], []) == [0, 0, 0, 0, 1, 1, 1, 1, 0, 2]
    # next to a perfect 4-token hypothesis: c = 4, r = 2 + 4, p_n = 4/5, 3/4, 2/3, 1/2
    got = ob.corpus_bleu([[[5, 6]], [[1, 2, 3, 4]]], [[], [1, 2, 3, 4]])
    assert got == pytest.approx(math.exp(1 - 6 / 4) * 0.2 ** 0.25, rel=1e-14)


def test_oracle_no_unigram_match_is_zero():
    assert ob.corpus_bleu([[[4, 5, 6]]], [[1, 2, 3]]) == 0
    assert ob.corpus_bleu([[[4, 5, 6]]], [[1, 2, 3]], W4) == [0, 0, 0, 0]


def test_oracle_closest_ref_length_tie_goes_to_the_shorter():
    assert ob.closest_ref_length([[1] * 4, [1] * 6], 5) == 4
    assert ob.closest_ref_length([[1] * 6, [1] * 4], 5) == 4
    assert ob.closest_ref_length([[1] * 6, [1] * 3], 5) == 6


def test_oracle_weights_length_1_to_4_and_lists():
    refs, hyps = [[[1, 2, 3, 4, 6]]], [[1, 2, 3, 4, 5]]     # p_n = 4/5, 3/4, 2/3, 1/2; c = r = 5 -> bp = 1
    want = [0.8, math.sqrt(0.6), 0.4 ** (1 / 3), 0.2 ** 0.25]
    got = [ob.corpus_bleu(refs, hyps, w) for w in W4]
    assert got == pytest.approx(want, rel=1e-14)
    assert ob.corpus_bleu(refs, hyps, W4) == got
    assert ob.corpus_bleu(refs, hyps, [W4[3]]) == got[3]         # a one-tuple list returns the score itself (nltk)


def _random_corpus(rng, n, vocab, max_len, max_refs, cap_len=None):
    """Hypotheses and references cut from a shared "scene" per item, with substitutions, so every order matches."""
    refs, hyps = [], []
    for _ in range(n):
        scene = [rng.randrange(vocab) for _ in range(max_len)]

        def sent():
            L = rng.randint(0, max_len)
            s0 = rng.randint(0, max_len - L)
            return [w if rng.random() > 0.2 else rng.randrange(vocab) for w in scene[s0:s0 + L]]
        refs.append([sent() for _ in range(rng.randint(1, max_refs))])
        hyps.append(sent())
    if cap_len:
        for i in range(0, n, max(1, n // 8)):
            hyps[i] = [rng.randrange(vocab) for _ in range(cap_len)]
            refs[i][0] = hyps[i][: cap_len // 2] + [rng.randrange(vocab) for _ in range(cap_len - cap_len // 2)]
    return refs, hyps


def test_oracle_matches_live_nltk():
    nltk_bleu = pytest.importorskip("nltk.translate.bleu_score")
    rng = random.Random(5)
    for vocab in (4, 30):
        refs, hyps = _random_corpus(rng, 300, vocab, 20, 5)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            for w in W4:
                assert ob.corpus_bleu(refs, hyps, w) == nltk_bleu.corpus_bleu(refs, hyps, w)
            assert ob.sentence_bleu(refs[0], hyps[0]) == nltk_bleu.sentence_bleu(refs[0], hyps[0])


# ---- argument checks of bleu.corpus_bleu (all before any device call) -------------------------------------------------
def test_corpus_bleu_argument_errors():
    from icei_b200.bleu import corpus_bleu
    with pytest.raises(AssertionError):
        corpus_bleu([[[1, 2]]], [[1, 2], [3]])
    with pytest.raises(ValueError):
        corpus_bleu([[[1, 2]], []], [[1, 2], [3]])                 # second hypothesis has no reference
    with pytest.raises(TypeError):
        corpus_bleu([[[1, 2]]], [[1.0, 2]])
    with pytest.raises(TypeError):
        corpus_bleu([[["a", "b"]]], [["a"]])
    with pytest.raises(TypeError):
        corpus_bleu([[[1, None]]], [[1]])
    for bad in (2 ** 31, -2 ** 31 - 1, 2 ** 63, 2 ** 70):
        with pytest.raises(ValueError):
            corpus_bleu([[[1, 2]]], [[1, bad]])
    with pytest.raises(ValueError):
        corpus_bleu([[[1, 2]]], [[1, 2]], (0.2,) * 5)
    with pytest.raises(ValueError):
        corpus_bleu([[[1, 2]]], [[1, 2]], [(0.5, 0.5), (0.2,) * 5])
    with pytest.raises(ValueError):
        corpus_bleu([[[1, 2]]], [[1, 2]], ())
    with pytest.raises(TypeError):
        corpus_bleu([[[1, 2]]], [[1, 2]], smoothing_function=None)


def test_corpus_bleu_empty_corpus_is_zero():
    from icei_b200.bleu import corpus_bleu
    assert corpus_bleu([], []) == 0
    assert corpus_bleu([], [], W4) == [0, 0, 0, 0]


def test_pack_layout():
    from icei_b200.bleu import _pack
    buf, (n, R, Th, Tr), max_len, max_group = _pack([[[5, 6], [7]], [[8, 9, 10]]], [[1, 2, 3], []])
    assert (n, R, Th, Tr) == (2, 3, 3, 6)
    assert buf[:3].tolist() == [0, 3, 3]                      # hyp_off
    assert buf[3:7].tolist() == [0, 2, 3, 6]                  # ref_off
    assert buf[7:10].tolist() == [0, 2, 3]                    # ref_group
    assert buf[10:].view("int32")[:9].tolist() == [1, 2, 3, 5, 6, 7, 8, 9, 10]
    assert (max_len, max_group) == (3, 6)


# ---- on the GPU: the kernel and the scores against the oracle ----------------------------------------------------------
EDGE = {
    "empty_hyp": ([[[5, 6]], [[1, 2, 3, 4]]], [[], [1, 2, 3, 4]]),
    "all_empty": ([[[1, 2, 3]]], [[]]),
    "short_hyp": ([[[7, 8]]], [[7, 8]]),
    "no_unigram": ([[[4, 5, 6]]], [[1, 2, 3]]),
    "clipping": ([[[3, 9]], [[3, 3, 9], [3, 9, 3, 3, 3]]], [[3, 3, 3, 3], [3, 3, 3, 3]]),
    "tie": ([[[1] * 4, [2] * 6], [[2] * 6, [1] * 4]], [[1] * 5, [1, 1, 2, 2, 1]]),
    "weights": ([[[1, 2, 3, 4, 6]]], [[1, 2, 3, 4, 5]]),
    "negative_ids": ([[[-2 ** 31, 2 ** 31 - 1, 0]]], [[-2 ** 31, 2 ** 31 - 1, 1]]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(EDGE))
def test_edge_cases_equal_oracle(case):
    from icei_b200.bleu import _stats, corpus_bleu
    refs, hyps = EDGE[case]
    st = _stats(refs, hyps).cpu().tolist()
    assert st == [ob.sentence_stats(r, h) for r, h in zip(refs, hyps)]
    for w in W4:
        assert corpus_bleu(refs, hyps, w) == ob.corpus_bleu(refs, hyps, w)
    assert corpus_bleu(refs, hyps, W4) == ob.corpus_bleu(refs, hyps, W4)
    assert corpus_bleu(refs, hyps, [W4[2]]) == ob.corpus_bleu(refs, hyps, [W4[2]])


@pytest.mark.gpu
def test_stats_and_scores_equal_oracle_on_random_corpus():
    from icei_b200.bleu import _stats, corpus_bleu
    rng = random.Random(11)
    refs, hyps = _random_corpus(rng, 2100, 6, 45, 7, cap_len=256)
    assert max(len(h) for h in hyps) == 256 and min(len(h) for h in hyps) == 0
    st = _stats(refs, hyps).cpu().tolist()
    want = [ob.sentence_stats(r, h) for r, h in zip(refs, hyps)]
    assert st == want
    assert all(sum(row[n] for row in st) > 0 for n in range(4))        # every order has matches
    for w in W4:
        assert corpus_bleu(refs, hyps, w) == ob.corpus_bleu(refs, hyps, w)
    assert corpus_bleu(refs, hyps, W4) == ob.corpus_bleu(refs, hyps, W4)
    assert _stats(refs, hyps).cpu().tolist() == st                    # run to run


@pytest.mark.gpu
def test_large_reference_group_uses_opt_in_shared_memory():
    """100 references of up to 200 tokens: 80 KB of tokens for one CTA (above the 48 KB default)."""
    from icei_b200.bleu import _stats, corpus_bleu
    rng = random.Random(3)
    refs = [[[rng.randrange(5) for _ in range(200)] for _ in range(100)], [[1, 2, 3]]]
    hyps = [[rng.randrange(5) for _ in range(150)], [1, 2, 3]]
    assert _stats(refs, hyps).cpu().tolist() == [ob.sentence_stats(r, h) for r, h in zip(refs, hyps)]
    assert corpus_bleu(refs, hyps, W4) == ob.corpus_bleu(refs, hyps, W4)


@pytest.mark.gpu
def test_limits_are_rejected_before_launch():
    from icei_b200._lib import SnError
    from icei_b200.bleu import corpus_bleu
    with pytest.raises(SnError, match="256"):
        corpus_bleu([[[1, 2]]], [[1] * 257])
    with pytest.raises(SnError, match="256"):
        corpus_bleu([[[1, 2], [3] * 257]], [[1, 2]])
    corpus_bleu([[[1, 2]]], [[1] * 256])
    with pytest.raises(SnError, match="shared memory"):
        corpus_bleu([[[1] * 256] * 250], [[1, 2]])                   # 64 000 tokens for one hypothesis


# ---- evaluate.validate(..., bleu_weights=...) --------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["factored", "nic", "factored_att"])
def test_validate_bleu(kind):
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
    res = validate(dec, batches, 1, 2, bleu_weights=W4, **kw)
    assert set(res) == set(plain) | {"bleu"}
    assert all(res[k] == plain[k] for k in plain)
    want = ob.corpus_bleu(res["references"], res["hypotheses"], W4)
    assert res["bleu"] == want and want[0] > 0.3 and want[3] > 1e-3
    assert validate(dec, batches, 1, 2, bleu_weights=W4[3], **kw)["bleu"] == want[3]
    with pytest.raises(ValueError):
        validate(dec, batches[:1] + [batches[1][:3] + (None,)], 1, 2, bleu_weights=W4[3], **kw)
