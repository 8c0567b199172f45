"""Pin the CPU oracle (oracle/port.py) against vectors produced by the unmodified reference
modules (tests/golden/*.npz, made by oracle/make_golden.py) and, when SN_REFERENCE_ROOT names a
checkout of the original project, against the live reference.  float64 throughout: tolerance 1e-10 relative."""
import random

import numpy as np
import pytest
import torch

from oracle import port, reference_loader as rl
from golden_util import CASES, build_port, load_golden, rel_l2, sd_from

TOL = 1e-10


def _fwd(dec, rec, tf, mode, att, grad_feats=False):
    cap = torch.from_numpy(rec["in.captions"])
    lens = [int(x) for x in rec["in.lengths"]]
    feats = torch.from_numpy(rec["in.features"]).clone().requires_grad_(grad_feats)
    kw = {} if mode is None else {"mode": mode}
    random.seed(1234)
    if att:
        l1 = [l - 1 for l in lens]
        out, alphas = dec(cap[:, :-1], l1, feats, teacher_forcing_ratio=tf, **kw)
        loss = port.caption_loss(out, port.pack_targets(cap[:, 1:], l1), alphas)
    else:
        out = dec(cap, lens, feats, teacher_forcing_ratio=tf, **kw)
        alphas = None
        loss = port.caption_loss(out, port.pack_targets(cap, lens))
    return out, alphas, loss, feats


@pytest.mark.parametrize("name", list(CASES))
def test_port_matches_golden_forward_backward(name):
    att, modes = CASES[name]
    rec = load_golden(name)
    torch.set_default_dtype(torch.float64)
    try:
        dec = build_port(name, rec)
        dec.train()
        for mode in modes:
            tag = "" if mode is None else "." + mode
            dec.zero_grad()
            out, alphas, loss, feats = _fwd(dec, rec, 1.0, mode, att, grad_feats=not att)
            loss.backward()
            assert rel_l2(out.detach(), rec["tf1.logits" + tag]) < TOL
            assert abs(loss.item() - float(rec["tf1.loss" + tag])) < TOL
            if att:
                assert rel_l2(alphas.detach(), rec["tf1.alphas" + tag]) < TOL
            else:
                assert rel_l2(feats.grad, rec["tf1.dfeatures" + tag]) < TOL
            pre = "tf1.grad%s." % tag
            names = {n for n, p in dec.named_parameters() if p.grad is not None}
            assert names == {k[len(pre):] for k in rec if k.startswith(pre)}
            for n, p in dec.named_parameters():
                if p.grad is not None:
                    g = rec[pre + n]
                    if n.endswith("full_att.bias"):   # true gradient is 0 (softmax shift invariance)
                        assert float(p.grad.abs().max()) < 1e-12 and float(np.abs(g).max()) < 1e-12
                    else:
                        assert rel_l2(p.grad, g) < 1e-9, n
            with torch.no_grad():
                out0, _, _, _ = _fwd(dec, rec, 0.0, mode, att)
            assert rel_l2(out0, rec["tf0.logits" + tag]) < TOL
            assert np.array_equal(out0.argmax(1).numpy(), rec["tf0.argmax" + tag])
            out5, _, _, _ = _fwd(dec, rec, 0.5, mode, att)
            assert rel_l2(out5.detach(), rec["tf05.logits" + tag]) < TOL
        if name == "factored":
            cap = torch.from_numpy(rec["in.captions"])
            l1 = [int(x) - 1 for x in rec["in.lengths"]]
            outl = dec(cap[:, :-1], l1, None, teacher_forcing_ratio=1.0, mode="sad")
            assert rel_l2(outl.detach(), rec["lang.logits.sad"]) < TOL
    finally:
        torch.set_default_dtype(torch.float32)


@pytest.mark.parametrize("name", list(CASES))
def test_port_matches_golden_adam(name):
    att, modes = CASES[name]
    rec = load_golden(name)
    torch.set_default_dtype(torch.float64)
    try:
        dec = build_port(name, rec)
        dec.train()
        cap = torch.from_numpy(rec["in.captions"])
        lens = [int(x) for x in rec["in.lengths"]]
        feats = torch.from_numpy(rec["in.features"])
        opt_a = torch.optim.Adam(dec.parameters(), lr=2e-4)
        opt_b = torch.optim.Adam(dec.parameters(), lr=5e-4)
        for opt, mode in [(opt_a, modes[0]), (opt_b, modes[-1]), (opt_a, modes[0])]:
            random.seed(1234)
            loss = port.train_step(dec, opt, cap, lens, feats, mode=mode, attention=att)
        assert abs(loss.item() - float(rec["adam3.loss_last"])) < 1e-9
        for k, v in dec.state_dict().items():
            assert rel_l2(v, rec["adam3.sd." + k]) < 1e-9, k
    finally:
        torch.set_default_dtype(torch.float32)


@pytest.mark.parametrize("name", list(CASES))
def test_port_matches_golden_decode(name):
    att, modes = CASES[name]
    rec = load_golden(name)
    torch.set_default_dtype(torch.float64)
    try:
        dec = build_port(name, rec, prefix="sharp.sd.")
        dec.eval()
        with torch.no_grad():
            out0, _, _, _ = _fwd(dec, rec, 0.0, modes[-1], att)
        assert np.array_equal(out0.argmax(1).numpy(), rec["sharp.tf0.argmax"])
        feats = torch.from_numpy(rec["in.features"])
        kw = {} if modes[-1] is None else {"mode": modes[-1]}
        variants = sorted({k.split(".")[1] for k in rec if k.startswith("sample.")})
        lens_seen = set()
        for v in variants:
            for img in range(3):
                for k in (1, 3, 5):
                    extra = dict(kw)
                    if v == "app":
                        extra["feed_image"] = True
                    with torch.no_grad():
                        ids = dec.sample(feats[img].unsqueeze(0), 1, 2, k=k, **extra)
                    want = rec["sample.%s.img%d.k%d" % (v, img, k)]
                    assert np.array_equal(ids.numpy(), want), (v, img, k)
                    lens_seen.add(want.shape[1])
        assert len(lens_seen) > 1  # the recipe yields captions of varied lengths
    finally:
        torch.set_default_dtype(torch.float32)


@pytest.mark.parametrize("name", list(CASES))
def test_port_fp32_matches_reference_vectors(name):
    """fp32 port == what the UNMODIFIED reference computed (tests/golden/*.npz, float64): teacher-forced logits, loss and
    attention weights of every mode at 1e-6 -- the stored-data form of the live fp32 comparison below."""
    att, modes = CASES[name]
    rec = load_golden(name)
    dec = build_port(name, rec, dtype=torch.float32)
    dec.train()
    cap = torch.from_numpy(rec["in.captions"])
    lens = [int(x) for x in rec["in.lengths"]]
    feats = torch.from_numpy(rec["in.features"]).float()
    for mode in modes:
        tag = "" if mode is None else "." + mode
        kw = {} if mode is None else {"mode": mode}
        random.seed(1234)
        with torch.no_grad():
            if att:
                l1 = [l - 1 for l in lens]
                out, alphas = dec(cap[:, :-1], l1, feats, teacher_forcing_ratio=1.0, **kw)
                loss = port.caption_loss(out, port.pack_targets(cap[:, 1:], l1), alphas)
                assert rel_l2(alphas, rec["tf1.alphas" + tag]) < 1e-6
            else:
                out = dec(cap, lens, feats, teacher_forcing_ratio=1.0, **kw)
                loss = port.caption_loss(out, port.pack_targets(cap, lens))
        assert out.dtype == torch.float32
        assert rel_l2(out, rec["tf1.logits" + tag]) < 1e-6
        assert abs(loss.item() - float(rec["tf1.loss" + tag])) < 1e-6 * abs(float(rec["tf1.loss" + tag]))


@pytest.mark.skipif(not rl.available(), reason="reference tree not present")
@pytest.mark.parametrize("name,mod,cls", [
    ("factored", "stylenet", "DecoderFactoredLSTM"),
    ("factored_att", "stylenet_att", "DecoderFactoredLSTMAtt"),
    ("nic", "nic", "DecoderRNN"),
    ("nic_att", "nic_att", "DecoderRNNAtt"),
])
def test_port_matches_live_reference_fp32(name, mod, cls):
    """fp32, fresh seed, bigger-than-golden shapes: port == unmodified reference module."""
    att, modes = CASES[name]
    V, E, H, F, A, D = 211, 30, 48, 40, 32, 56
    ref_cls = getattr(rl.load(mod), cls)
    port_cls = getattr(port, cls)
    args = {"factored": (E, H, F, V, 1), "factored_att": (A, E, H, F, V, 1),
            "nic": (E, H, V, 1), "nic_att": (A, E, H, V, 1)}[name]
    kw = {"dropout": 0.0}
    if att:
        kw["feature_size"] = D
    torch.manual_seed(11)
    ref = ref_cls(*args, **kw)
    mine = port_cls(*args, **kw)
    mine.load_state_dict(ref.state_dict())
    cap, lens, feats = port.synthetic_batch(9, 11, V, E=None if att else E,
                                            feat_shape=(4, 4, D) if att else None, ragged=True, seed=5)
    mkw = {} if modes[-1] is None else {"mode": modes[-1]}
    for tf in (1.0, 0.0, 0.6):
        outs = []
        for m in (ref, mine):
            random.seed(99)
            if att:
                o, a = m(cap[:, :-1], [l - 1 for l in lens], feats, teacher_forcing_ratio=tf, **mkw)
                outs.append((o, a))
            else:
                outs.append((m(cap, lens, feats, teacher_forcing_ratio=tf, **mkw),))
        for x, y in zip(*outs):
            assert torch.equal(x, y) or rel_l2(x.detach(), y.detach()) < 1e-6


def test_stack_oracle_matches_reference_composition():
    """oracle/stack.py over ORACLE-PORT layers == the same composition over unmodified reference layers
    (tests/golden/stack3.npz, oracle/make_golden_stack.py): logits, loss, gradients (fp64, 1e-10), greedy ids."""
    import random
    from oracle import port
    from oracle.stack import stack_forward
    rec = load_golden("stack3")
    V, E, H, F, L = (int(rec["meta." + k]) for k in ("V", "E", "H", "F", "L"))
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        layers = [port.DecoderFactoredLSTM(E if l == 0 else H, H, F, V, 1, dropout=0.0, max_seq_length=12) for l in range(L)]
        for l, layer in enumerate(layers):
            pre = "sd.%d." % l
            layer.load_state_dict({k[len(pre):]: torch.from_numpy(v) for k, v in rec.items() if k.startswith(pre)})
        cap = torch.from_numpy(rec["in.captions"])
        lens = [int(x) for x in rec["in.lengths"]]
        feats = torch.from_numpy(rec["in.features"])
        tgt = port.pack_targets(cap, lens)
        for mode in ("factual", "sad"):
            for layer in layers:
                layer.zero_grad()
            random.seed(1234)
            out = stack_forward(layers, cap, lens, feats, teacher_forcing_ratio=1.0, mode=mode)
            loss = torch.nn.functional.cross_entropy(out, tgt)
            loss.backward()
            assert rel_l2(out.detach(), rec["tf1.logits." + mode]) < 1e-10
            assert abs(loss.item() - float(rec["tf1.loss." + mode])) < 1e-10
            for l, layer in enumerate(layers):
                for n, p in layer.named_parameters():
                    key = "tf1.grad.%s.%d.%s" % (mode, l, n)
                    if p.grad is not None and key in rec:
                        assert rel_l2(p.grad, rec[key]) < 1e-10, key
            with torch.no_grad():
                random.seed(1234)
                out0 = stack_forward(layers, cap, lens, feats, teacher_forcing_ratio=0.0, mode=mode)
            assert np.array_equal(out0.argmax(1).numpy(), rec["tf0.argmax." + mode])
    finally:
        torch.set_default_dtype(old)
