"""Self-critical training (icei_b200.scst, K12 sampling, weighted K5, per-sample K11) -- host logic and the CPU oracle:
the noise hash pinned to the C expression, the external-df CIDEr-D oracle, argument errors (raised before any device
work) and the length sort / token-weight layout on host-built plans."""
import numpy as np
import pytest
import torch

from oracle import cider as cider_oracle
from oracle import scst as scst_oracle


# (seed, step, row, col, hash_u32(seed_t, row, col), hash_u32(seed_t, 0, 0)) with seed_t = seed * 0x9E3779B97F4A7C15 +
# step, evaluated by a C program compiled from the expressions of sn_common.cuh / include/sn100.h
HASH_PINS = [(0, 1, 5, 9999, 2946844260, 885181228),
             (7, 2, 5, 9999, 655532466, 3513806905),
             (123456789, 41, 5, 9999, 3980739137, 3206005920)]


@pytest.mark.parametrize("seed,step,row,col,h,h00", HASH_PINS)
def test_hash_restatement_pinned(seed, step, row, col, h, h00):
    st = scst_oracle.step_seed(seed, step)
    assert scst_oracle.hash_u32(st, row, col) == h
    assert scst_oracle.hash_u32(st, 0, 0) == h00
    assert int(scst_oracle.hash_u32_np(st, row, np.array([col]))[0]) == h


def test_gumbel_and_draw():
    g = scst_oracle.gumbel(3, 2, 1, 64)
    u = ((scst_oracle.hash_u32_np(scst_oracle.step_seed(3, 2), 1, np.arange(64)) >> np.uint64(8)).astype(np.float64)
         + 0.5) / 2 ** 24
    assert np.array_equal(g, -np.log(-np.log(u)))
    logits = np.zeros(64, np.float32)
    assert scst_oracle.draw(logits, 3, 2, 1) == int(np.argmax(g))
    logits[17] = 1.0
    logits[40] = 1.0
    assert scst_oracle.draw(logits, 3, 2, 1, greedy=True) == 17          # ties -> the lowest index


def _corpus(seed, n_img, V=12):
    rng = np.random.default_rng(seed)
    return [[list(rng.integers(0, V, rng.integers(1, 9))) for _ in range(rng.integers(1, 4))] for _ in range(n_img)]


def test_external_df_equals_corpus_cider_on_its_own_corpus():
    refs = _corpus(0, 9)
    rng = np.random.default_rng(1)
    hyps = [list(rng.integers(0, 12, rng.integers(0, 9))) for _ in range(9)]
    _, per = cider_oracle.corpus_cider(refs, hyps)
    got = scst_oracle.sample_scores(refs, list(range(9)), hyps)
    assert np.array_equal(got, per)
    # repeated ids: each row scored against its image with the corpus' df and log N
    ids = [3, 3, 0, 8]
    rows = scst_oracle.sample_scores(refs, ids, [hyps[3], hyps[3], hyps[0], hyps[8]])
    assert np.array_equal(rows, per[ids])


def _cpu_decoder():
    import icei_b200 as sn
    return sn.DecoderFactoredLSTM(8, 16, 8, 20, 1, dropout=0.0, max_seq_length=6)


@pytest.mark.parametrize("kw", [dict(n=0), dict(n=1.5), dict(temperature=0.0), dict(temperature=float("nan")),
                                dict(temperature=float("inf")), dict(temperature=-1.0), dict(seed=-1),
                                dict(mode=["factual", "happy"]), dict(mode="neutral")])
def test_sample_captions_argument_errors(kw):
    dec = _cpu_decoder()
    with pytest.raises(ValueError):
        dec.sample_captions(torch.zeros(2, 8), 1, 2, **kw)


def test_scst_step_argument_errors():
    import icei_b200 as sn
    dec = _cpu_decoder()
    feats = torch.zeros(3, 8)
    for kw in (dict(baseline="max"), dict(baseline="mean", n=1), dict(image_ids=[0, 1])):
        args = dict(image_ids=[0, 1, 2])
        args.update(kw)
        ids = args.pop("image_ids")
        with pytest.raises(ValueError):
            sn.scst.scst_step(dec, None, None, feats, ids, 1, 2, **args)


def test_score_samples_argument_errors():
    import icei_b200 as sn
    cd = object.__new__(sn.cider.CiderD)          # the checks run before the object's device state is touched
    cd.n_img = 4
    seqs = torch.zeros(3, 5, dtype=torch.int64)
    lens = torch.full((3,), 3, dtype=torch.int64)
    with pytest.raises(ValueError):
        cd.score_samples(seqs[0], lens, [0, 1, 2], 1, 2)                  # not 2-D
    with pytest.raises(ValueError):
        cd.score_samples(seqs, lens[:2], [0, 1, 2], 1, 2)                 # lengths of another size
    with pytest.raises(ValueError):
        cd.score_samples(seqs, lens, [0, 1], 1, 2)                        # image ids of another size
    with pytest.raises(ValueError):
        cd.score_samples(seqs, lens, [0, 4, 1], 1, 2)                     # out of range
    with pytest.raises(ValueError):
        cd.score_samples(seqs, lens, [0, -1, 1], 1, 2)


def test_sort_and_token_weight_layout():
    import icei_b200 as sn
    lens = [3, 5, 2, 5, 4, 3]
    order = sn.scst.sort_by_length(lens)
    assert order == [1, 3, 4, 0, 5, 2]                                    # descending, stable
    lens_s = [lens[r] for r in order]
    plan = sn.PackPlan(lens_s)
    adv = torch.tensor([0.5, -1.0, 2.0, 0.0, 3.0, -0.25], dtype=torch.float64)
    w = sn.scst.token_weights(adv, plan)
    assert w.dtype == torch.float32 and w.shape == (plan.N,)
    want = []
    for t in range(lens_s[0]):                                            # packed rows: time-major
        for b in range(len(lens_s)):
            if lens_s[b] > t:
                want.append(0.0 if t == 0 else float(adv[b]))
    assert torch.equal(w, torch.tensor(want, dtype=torch.float32))


def test_advantages():
    import icei_b200 as sn
    r = torch.tensor([1.0, 2.0, 3.0, 0.0, 0.0, 6.0], dtype=torch.float64)
    adv, base = sn.scst.advantages(r, 3, "mean")
    assert torch.allclose(base, torch.tensor([2.5, 2.0, 1.5, 3.0, 3.0, 0.0], dtype=torch.float64))
    assert torch.allclose(adv, r - base)
    adv, base = sn.scst.advantages(r, 3, "greedy", torch.tensor([1.0, 4.0], dtype=torch.float64))
    assert torch.equal(base, torch.tensor([1.0, 1, 1, 4, 4, 4], dtype=torch.float64))
    a2, b2 = scst_oracle.advantages(r.numpy(), 3, "greedy", [1.0, 4.0])
    assert np.array_equal(adv.numpy(), a2) and np.array_equal(base.numpy(), b2)
