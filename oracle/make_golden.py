"""Generate tests/golden/*.npz by executing the UNMODIFIED reference modules on CPU.

TEST INFRASTRUCTURE ONLY.  Needs a checkout of the original project:

    SN_REFERENCE_ROOT=<checkout> python -m oracle.make_golden

The reference ships no golden vectors (SURVEY.md section 8c), so these files ARE the pin: they
record what stylenet/model.py, stylenet/model_att.py, nic/model.py, nic/model_att.py and
app/backend/model.py (unmodified apart from the ``//`` shim of oracle/reference_loader.py)
compute on seeded synthetic inputs.  Everything is float64 so the vectors sit below the
fp32 noise floor of any implementation compared against them.
"""
import os
import random

import numpy as np
import torch

from oracle import reference_loader as rl
from oracle.port import pack_targets, synthetic_batch, lively_weights, STYLES

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# small, deliberately awkward sizes (E not a multiple of 8, V not a multiple of anything)
V, E, H, Fs, A, D, S = 53, 12, 16, 20, 16, 24, 3
B, T = 6, 7


def _sd_np(module, prefix="sd."):
    return {prefix + k: v.detach().numpy().copy() for k, v in module.state_dict().items()}


def _grads_np(module, prefix="grad."):
    return {prefix + n: p.grad.detach().numpy().copy() for n, p in module.named_parameters()
            if p.grad is not None}


def _run_forward(dec, cap, lens, feats, tf, mode, att):
    kw = {} if mode is None else {"mode": mode}
    random.seed(1234)
    if att:
        lens1 = [l - 1 for l in lens]
        out, alphas = dec(cap[:, :-1], lens1, feats, teacher_forcing_ratio=tf, **kw)
        tgt = pack_targets(cap[:, 1:], lens1)
        loss = torch.nn.functional.cross_entropy(out, tgt) + ((1. - alphas.sum(dim=1)) ** 2).mean()
        return out, alphas, loss
    out = dec(cap, lens, feats, teacher_forcing_ratio=tf, **kw)
    loss = torch.nn.CrossEntropyLoss()(out, pack_targets(cap, lens))
    return out, None, loss


def make_case(name, build, att, modes, sample_variants):
    torch.set_default_dtype(torch.float64)
    try:
        torch.manual_seed(7)
        dec = build()
        dec.train()
        rec = {"meta.V": V, "meta.E": E, "meta.H": H, "meta.F": Fs, "meta.A": A, "meta.D": D,
               "meta.S": S}
        rec.update(_sd_np(dec))
        cap, lens, feats = synthetic_batch(B, T, V, E=None if att else E,
                                           feat_shape=(S, S, D) if att else None, ragged=True, seed=3)
        feats = feats.double()
        rec["in.captions"] = cap.numpy()
        rec["in.lengths"] = np.asarray(lens)
        rec["in.features"] = feats.numpy()
        for mode in modes:
            tag = "" if mode is None else "." + mode
            # teacher forced forward + backward
            dec.zero_grad()
            f = feats.clone().requires_grad_(not att)
            out, alphas, loss = _run_forward(dec, cap, lens, f, 1.0, mode, att)
            loss.backward()
            rec["tf1.logits" + tag] = out.detach().numpy()
            rec["tf1.loss" + tag] = np.asarray(loss.item())
            if alphas is not None:
                rec["tf1.alphas" + tag] = alphas.detach().numpy()
            rec.update(_grads_np(dec, "tf1.grad%s." % tag))
            if not att:
                rec["tf1.dfeatures" + tag] = f.grad.numpy()
            # greedy (validation) forward, tf = 0
            with torch.no_grad():
                out0, _, loss0 = _run_forward(dec, cap, lens, feats, 0.0, mode, att)
            rec["tf0.logits" + tag] = out0.numpy()
            rec["tf0.argmax" + tag] = out0.argmax(1).numpy()
            # scheduled sampling, coin stream random.seed(1234), ratio 0.5
            dec.zero_grad()
            out5, _, loss5 = _run_forward(dec, cap, lens, feats, 0.5, mode, att)
            loss5.backward()
            rec["tf05.logits" + tag] = out5.detach().numpy()
            rec.update(_grads_np(dec, "tf05.grad%s." % tag))
        # language-only pass (features=None; stylenet/train.py:369-375)
        if not att and modes[0] is not None:
            random.seed(1234)
            lens1 = [l - 1 for l in lens]
            outl = dec(cap[:, :-1], lens1, None, teacher_forcing_ratio=1.0, mode="sad")
            rec["lang.logits.sad"] = outl.detach().numpy()
        # optimizer: 3 alternating steps with the reference's two Adams + clip 0.5
        utils = rl.load("stylenet_utils")
        opt_a = torch.optim.Adam(dec.parameters(), lr=2e-4)
        opt_b = torch.optim.Adam(dec.parameters(), lr=5e-4)
        sched = [(opt_a, modes[0]), (opt_b, modes[-1]), (opt_a, modes[0])]
        for opt, mode in sched:
            _, _, loss = _run_forward(dec, cap, lens, feats, 1.0, mode, att)
            dec.zero_grad()
            loss.backward()
            utils.clip_gradient(opt, 0.5)
            opt.step()
        rec.update(_sd_np(dec, "adam3.sd."))
        rec["adam3.loss_last"] = np.asarray(loss.item())
        # decode: restore the initial weights, sharpen, beam-search three images
        dec.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in rec.items() if k.startswith("sd.")})
        dec.eval()
        best = None
        for end_bias in (1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 8.0):   # pick the recipe with the most varied lengths
            lively_weights(dec, end_bias=end_bias)
            kw = {} if modes[-1] is None else {"mode": modes[-1]}
            with torch.no_grad():
                lens_seen = {dec.sample(sample_variants[0][3](feats[i]), 1, 2, k=k, **kw).shape[1]
                             for i in range(3) for k in (1, 3, 5)}
            score = len(lens_seen - {1})
            if best is None or score > best[0]:
                best = (score, end_bias)
        lively_weights(dec, end_bias=best[1])
        rec["sharp.end_bias"] = np.asarray(best[1])
        rec.update(_sd_np(dec, "sharp.sd."))
        with torch.no_grad():
            out0, _, _ = _run_forward(dec, cap, lens, feats, 0.0, modes[-1], att)
        rec["sharp.tf0.argmax"] = out0.argmax(1).numpy()
        for vname, mod_name, cls_name, kw_feat, extra in sample_variants:
            cls = getattr(rl.load(mod_name), cls_name)
            d2 = build(cls)
            d2.load_state_dict(dec.state_dict())
            d2.eval()
            for img in range(3):
                for k in (1, 3, 5):
                    for mode in (modes[-1],):
                        kw = dict(extra) if mode is None else {"mode": mode}
                        with torch.no_grad():
                            ids = d2.sample(kw_feat(feats[img]), 1, 2, k=k, **kw)
                        rec["sample.%s.img%d.k%d" % (vname, img, k)] = ids.numpy()
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **rec)
        print(name, "->", len(rec), "arrays")
    finally:
        torch.set_default_dtype(torch.float32)


def main():
    assert rl.available(), "set SN_REFERENCE_ROOT to a checkout of the original project"
    os.makedirs(OUT, exist_ok=True)
    sty, sty_att = rl.load("stylenet"), rl.load("stylenet_att")
    nic, nic_att = rl.load("nic"), rl.load("nic_att")

    make_case("factored", lambda c=sty.DecoderFactoredLSTM: c(E, H, Fs, V, 1, dropout=0.0, max_seq_length=12),
              False, ["factual", "happy"],
              [("stylenet", "stylenet", "DecoderFactoredLSTM", lambda f: f.unsqueeze(0), {}),
               ("app", "app", "DecoderFactoredLSTM", lambda f: f.reshape(1, 1, -1), {})])
    make_case("factored_att", lambda c=sty_att.DecoderFactoredLSTMAtt: c(A, E, H, Fs, V, 1, feature_size=D, dropout=0.0, max_seq_length=12),
              True, ["factual", "angry"],
              [("stylenet", "stylenet_att", "DecoderFactoredLSTMAtt", lambda f: f.unsqueeze(0), {})])
    make_case("nic", lambda c=nic.DecoderRNN: c(E, H, V, 1, dropout=0.0, max_seq_length=12),
              False, [None],
              [("nic", "nic", "DecoderRNN", lambda f: f.unsqueeze(0), {}),
               ("app", "app", "DecoderRNN", lambda f: f.reshape(1, 1, -1), {"mode": "factual"})])
    make_case("nic_att", lambda c=nic_att.DecoderRNNAtt: c(A, E, H, V, 1, feature_size=D, dropout=0.0, max_seq_length=12),
              True, [None],
              [("nic", "nic_att", "DecoderRNNAtt", lambda f: f.unsqueeze(0), {})])


if __name__ == "__main__":
    main()
