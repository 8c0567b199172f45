"""Checkpoint interchange (SURVEY.md section 8 f3), CPU: reference whole-object checkpoints (stylenet/utils.py:63-90) ->
drop-in modules and back.  The live-reference cases are skipped unless SN_REFERENCE_ROOT names a checkout of the original."""
import os
import sys

import pytest
import torch

import icei_b200 as sn
from icei_b200 import checkpoint as ck
from oracle import reference_loader as rl


def _make(kind):
    if kind == "factored":
        return sn.DecoderFactoredLSTM(12, 16, 20, 53, 1, dropout=0.3, max_seq_length=17)
    if kind == "factored_att":
        return sn.DecoderFactoredLSTMAtt(24, 12, 16, 20, 53, 1, feature_size=40, dropout=0.3, max_seq_length=17)
    if kind == "nic":
        return sn.DecoderRNN(12, 16, 53, 1, dropout=0.3, max_seq_length=17)
    if kind == "nic_att":
        return sn.DecoderRNNAtt(24, 12, 16, 53, 1, feature_size=40, dropout=0.3, max_seq_length=17)
    return sn.DecoderFactoredLSTMStack(12, 16, 20, 53, 3, dropout=0.3, max_seq_length=17)


@pytest.mark.parametrize("kind", ["factored", "factored_att", "nic", "nic_att", "stack"])
def test_decoder_rebuilt_from_state_dict_alone(kind):
    torch.manual_seed(0)
    src = _make(kind)
    dec = ck.decoder_from_state_dict(src.state_dict(), dropout=0.3, max_seq_length=17)
    assert type(dec) is type(src)
    for a in ("hidden_size", "vocab_size", "max_seq_length"):
        assert getattr(dec, a) == getattr(src, a)
    for (n, p), (n2, q) in zip(src.state_dict().items(), dec.state_dict().items()):
        assert n == n2 and torch.equal(p, q)
    with pytest.raises(ValueError):
        ck.decoder_from_state_dict({"foo.weight": torch.zeros(2, 2)})


def test_save_checkpoint_writes_reference_layout_and_load_model_reads_it(tmp_path):
    torch.manual_seed(0)
    dec = _make("factored")
    opt, lang = sn.FusedClampAdam(dec, lr=2e-4), sn.FusedClampAdam(dec, lr=5e-4)
    opt._state(); opt.m.uniform_(-1, 1); opt.steps_dev.fill_(2)
    f = ck.save_checkpoint(str(tmp_path), "flickr", "factual", 3, {"factual": 0, "emotion": 1}, None, dec, opt, lang,
                           {"factual": 0.03, "emotion": 0.0}, True)
    assert os.path.basename(f) == "factual_checkpoint_flickr.pth.tar"
    assert os.path.exists(str(tmp_path / "factual_BEST_checkpoint_flickr.pth.tar"))
    state = torch.load(f, weights_only=False)
    assert set(state) == {"epoch", "epochs_since_improvement", "bleu-4", "encoder", "decoder", "optimizer", "lang_optimizer"}
    assert state["epoch"] == 3 and state["optimizer"].param_groups[0]["lr"] == 2e-4
    enc2, dec2 = ck.load_model(f)
    assert enc2 is None and not dec2.training
    assert all(torch.equal(p, q) for p, q in zip(dec.state_dict().values(), dec2.state_dict().values()))


needs_ref = pytest.mark.skipif(not rl.available(), reason="reference tree not present")


@needs_ref
@pytest.mark.parametrize("name,ctor", [
    ("stylenet", lambda m: m.DecoderFactoredLSTM(12, 16, 20, 53, 1, dropout=0.4, max_seq_length=21)),
    ("stylenet_att", lambda m: m.DecoderFactoredLSTMAtt(24, 12, 16, 20, 53, 1, feature_size=40, dropout=0.4, max_seq_length=21)),
    ("nic", lambda m: m.DecoderRNN(12, 16, 53, 1, dropout=0.4, max_seq_length=21)),
    ("nic_att", lambda m: m.DecoderRNNAtt(24, 12, 16, 53, 1, feature_size=40, dropout=0.4, max_seq_length=21)),
])
def test_reference_whole_object_checkpoint_converts_both_ways(tmp_path, name, ctor):
    """save_checkpoint of the UNMODIFIED reference (whole decoder + both Adam objects pickled) -> drop-in decoder and
    FusedClampAdam with identical weights / moments / step counts; export_state loads back into the reference."""
    mod = rl.load(name)
    sys.modules[mod.__name__] = mod                 # torch.load resolves pickled classes by module name
    utils = rl.load("stylenet_utils")
    torch.manual_seed(0)
    ref = ctor(mod)
    opt = torch.optim.Adam(ref.parameters(), lr=2e-4)
    lang = torch.optim.Adam(ref.parameters(), lr=5e-4)
    # two reference training steps so that the optimizers carry state (inactive styles keep none: grad is None)
    att = name.endswith("att")
    cap = torch.randint(4, 53, (5, 7)); cap[:, 0] = 1
    lens = [7, 6, 6, 4, 3]
    feats = torch.randn(5, 3, 3, 40) if att else torch.randn(5, 12)
    for o in (opt, lang):
        kw = {"mode": "happy"} if name.startswith("stylenet") else {}
        out = ref(cap[:, :-1], [l - 1 for l in lens], feats, teacher_forcing_ratio=1.0, **kw) if att else \
            ref(cap, lens, feats, teacher_forcing_ratio=1.0, **kw)
        out = out[0] if att else out
        o.zero_grad()
        out.logsumexp(1).mean().backward()
        utils.clip_gradient(o, 0.5)
        o.step()
    utils.save_checkpoint(str(tmp_path), "d", "factual", 1, {"factual": 0}, None, ref, opt, lang, {"factual": 0.1}, False)
    out = ck.convert_checkpoint(str(tmp_path / "factual_checkpoint_d.pth.tar"))
    dec = out["decoder"]
    assert type(dec).__name__ == type(ref).__name__ and dec.max_seq_length == 21 and dec.dropout.p == 0.4
    assert out["epoch"] == 1 and out["bleu-4"] == {"factual": 0.1}
    for (n, p), (n2, q) in zip(ref.state_dict().items(), dec.state_dict().items()):
        assert n == n2 and torch.equal(p, q)
    for mine, theirs in ((out["optimizer"], opt), (out["lang_optimizer"], lang)):
        a, b = mine.state_dict(), theirs.state_dict()
        assert sorted(a["state"]) == sorted(b["state"]) and a["param_groups"][0]["lr"] == b["param_groups"][0]["lr"]
        for i in b["state"]:
            assert float(a["state"][i]["step"]) == float(b["state"][i]["step"])
            assert torch.equal(a["state"][i]["exp_avg"], b["state"][i]["exp_avg"])
            assert torch.equal(a["state"][i]["exp_avg_sq"], b["state"][i]["exp_avg_sq"])
    # and back: plain tensors the reference classes load
    exp = ck.export_state(dec, out["optimizer"], out["lang_optimizer"])
    ref2 = ctor(mod)
    ref2.load_state_dict(exp["decoder"])
    opt2 = torch.optim.Adam(ref2.parameters(), lr=1.0)
    opt2.load_state_dict(exp["optimizer"])
    assert opt2.param_groups[0]["lr"] == 2e-4
    assert all(torch.equal(p, q) for p, q in zip(ref.state_dict().values(), ref2.state_dict().values()))
    # the drop-in's own pickle goes through load_model too
    ck.save_checkpoint(str(tmp_path), "mine", "factual", 2, {}, None, dec, out["optimizer"], out["lang_optimizer"], {}, False)
    _, dec3 = ck.load_model(str(tmp_path / "factual_checkpoint_mine.pth.tar"))
    assert all(torch.equal(p, q) for p, q in zip(ref.state_dict().values(), dec3.state_dict().values()))
