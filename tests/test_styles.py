"""Several styles in one beam search (``sample_batch(..., mode=[...])``), host side: argument checks, the stable grouping
by style and the way results return to input order.  No GPU needed: bad input is rejected before any device work."""
import pytest
import torch


def _styles():
    from icei_b200 import STYLES
    return STYLES


def test_group_styles_is_stable_and_in_style_order():
    from icei_b200.decode import group_styles
    STYLES = _styles()
    modes = ["sad", "factual", "sad", "angry", "factual"]
    groups, order = group_styles(modes, 5, STYLES)
    assert groups.styles == ("factual", "sad", "angry")
    assert groups.counts == (2, 2, 1)
    assert order == [1, 4, 0, 2, 3]                  # within a style, input order is kept
    assert [modes[i] for i in order] == ["factual", "factual", "sad", "sad", "angry"]
    g1, o1 = group_styles(tuple(STYLES), 4, STYLES)
    assert g1.styles == tuple(STYLES) and g1.counts == (1, 1, 1, 1) and o1 == [0, 1, 2, 3]
    g2, o2 = group_styles(["happy"] * 3, 3, STYLES)
    assert g2.styles == ("happy",) and g2.counts == (3,) and o2 == [0, 1, 2]
    # the groups are the session key: equal requests give equal, hashable keys
    assert hash(groups) == hash(group_styles(list(modes), 5, STYLES)[0])


def test_ungroup_returns_input_order():
    from icei_b200.decode import group_styles, ungroup
    modes = ["angry", "happy", "angry", "factual", "happy", "sad"]
    groups, order = group_styles(modes, len(modes), _styles())
    grouped = ["%s#%d" % (modes[i], i) for i in order]      # what a grouped beam search returns, image by image
    assert ungroup(grouped, order) == ["%s#%d" % (m, i) for i, m in enumerate(modes)]


@pytest.mark.parametrize("modes,n_img", [
    ([], 0),                                   # empty list
    (["factual", "sad"], 3),                   # wrong length
    (["factual", "sad", "cheerful"], 3),       # unknown style
    (["factual", None], 2),                    # not a style name
    ("factual,sad", 2),                        # a string is one style, not a list
])
def test_group_styles_rejects_bad_lists(modes, n_img):
    from icei_b200.decode import group_styles
    with pytest.raises(ValueError):
        group_styles(modes, n_img, _styles())


def test_sample_batch_rejects_bad_style_lists_before_device_work():
    """The decoders stay on the CPU: a ValueError (not a device error) shows the check runs first."""
    import icei_b200 as sn
    from icei_b200.decoders_att import DecoderFactoredLSTMAtt
    dec = sn.DecoderFactoredLSTM(8, 16, 12, 30, 1, dropout=0.0, max_seq_length=5)
    stack = sn.DecoderFactoredLSTMStack(8, 16, 12, 30, 2, dropout=0.0, max_seq_length=5)
    feats = torch.randn(3, 8)
    for d in (dec, stack):
        for bad in ([], ["factual", "sad"], ["factual", "sad", "glad"]):
            with pytest.raises(ValueError):
                d.sample_batch(feats, 1, 2, k=2, mode=bad)
        with pytest.raises(ValueError):                      # sample() takes one style
            d.sample(feats[:1], 1, 2, k=2, mode=["factual"])
    att = DecoderFactoredLSTMAtt(16, 8, 16, 12, 30, 1, feature_size=8, dropout=0.0, max_seq_length=5)
    fmap = torch.randn(3, 2, 2, 8)
    for bad in ([], ["factual"] * 2, ["factual", "sad", "glad"]):
        with pytest.raises(ValueError):
            att.sample_batch(fmap, 1, 2, k=2, mode=bad)


def test_generate_styles_argument_checks():
    import icei_b200 as sn
    from icei_b200 import evaluate
    dec = sn.DecoderFactoredLSTM(8, 16, 12, 30, 1, dropout=0.0, max_seq_length=5)
    batches = [torch.randn(2, 8)]
    with pytest.raises(ValueError):
        evaluate.generate(dec, batches, 1, 2, styles=())
    with pytest.raises(ValueError):
        evaluate.generate(dec, batches, 1, 2, mode="sad", styles=("sad",))
    with pytest.raises(ValueError):
        evaluate.generate(dec, batches, 1, 2, styles=("sad", "glad"))
    with pytest.raises(ValueError):
        evaluate.generate(dec, batches, 1, 2, styles=("sad", "sad"))
