"""Generate tests/golden/stack3.npz: the 3-layer FactoredLSTM stack (BASELINE.json configs[3]) evaluated by composing
UNMODIFIED reference ``DecoderFactoredLSTM`` objects through ``oracle/stack.py`` (their own ``forward_step``,
stylenet/model.py:115-155, does all the arithmetic).  TEST INFRASTRUCTURE ONLY; needs a checkout of the original:

    SN_REFERENCE_ROOT=<checkout> python -m oracle.make_golden_stack
"""
import os
import random

import numpy as np
import torch

from oracle import reference_loader as rl
from oracle.port import pack_targets, synthetic_batch
from oracle.stack import stack_forward, stack_parameters

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
V, E, H, Fs, L = 53, 12, 16, 20, 3
B, T = 6, 7


def build_layers(cls, dropout=0.0):
    return [cls(E if l == 0 else H, H, Fs, V, 1, dropout=dropout, max_seq_length=12) for l in range(L)]


def run(layers, cap, lens, feats, tf, mode):
    random.seed(1234)
    out = stack_forward(layers, cap, lens, feats, teacher_forcing_ratio=tf, mode=mode)
    return out, torch.nn.CrossEntropyLoss()(out, pack_targets(cap, lens))


def zero_grad(layers):
    for layer in layers:
        layer.zero_grad()


def main():
    assert rl.available(), "set SN_REFERENCE_ROOT to a checkout of the original project"
    sty, utils = rl.load("stylenet"), rl.load("stylenet_utils")
    torch.set_default_dtype(torch.float64)
    try:
        torch.manual_seed(11)
        layers = build_layers(sty.DecoderFactoredLSTM)
        for layer in layers:
            layer.train()
        rec = {"meta.V": V, "meta.E": E, "meta.H": H, "meta.F": Fs, "meta.L": L}
        for l, layer in enumerate(layers):
            rec.update({"sd.%d.%s" % (l, k): v.detach().numpy().copy() for k, v in layer.state_dict().items()})
        cap, lens, feats = synthetic_batch(B, T, V, E=E, ragged=True, seed=5)
        feats = feats.double()
        rec["in.captions"], rec["in.lengths"], rec["in.features"] = cap.numpy(), np.asarray(lens), feats.numpy()
        for mode in ("factual", "sad"):
            zero_grad(layers)
            f = feats.clone().requires_grad_(True)
            out, loss = run(layers, cap, lens, f, 1.0, mode)
            loss.backward()
            rec["tf1.logits." + mode] = out.detach().numpy()
            rec["tf1.loss." + mode] = np.asarray(loss.item())
            rec["tf1.dfeatures." + mode] = f.grad.numpy()
            for l, layer in enumerate(layers):
                for n, p in layer.named_parameters():
                    if p.grad is not None:
                        rec["tf1.grad.%s.%d.%s" % (mode, l, n)] = p.grad.detach().numpy().copy()
            with torch.no_grad():
                out0, _ = run(layers, cap, lens, feats, 0.0, mode)
            rec["tf0.logits." + mode] = out0.numpy()
            rec["tf0.argmax." + mode] = out0.argmax(1).numpy()
            zero_grad(layers)
            out5, loss5 = run(layers, cap, lens, feats, 0.5, mode)
            loss5.backward()
            rec["tf05.logits." + mode] = out5.detach().numpy()
            for l, layer in enumerate(layers):
                for n, p in layer.named_parameters():
                    if p.grad is not None:
                        rec["tf05.grad.%s.%d.%s" % (mode, l, n)] = p.grad.detach().numpy().copy()
        # multitask alternation (train_multitask.py:192-235): factual pass / optimizer, emotion pass / lang_optimizer
        params = stack_parameters(layers)
        opt_a = torch.optim.Adam(params, lr=2e-4)
        opt_b = torch.optim.Adam(params, lr=5e-4)
        for opt, mode in [(opt_a, "factual"), (opt_b, "sad"), (opt_a, "factual"), (opt_b, "happy")]:
            _, loss = run(layers, cap, lens, feats, 1.0, mode)
            zero_grad(layers)
            loss.backward()
            utils.clip_gradient(opt, 0.5)
            opt.step()
        for l, layer in enumerate(layers):
            rec.update({"adam4.sd.%d.%s" % (l, k): v.detach().numpy().copy() for k, v in layer.state_dict().items()})
        rec["adam4.loss_last"] = np.asarray(loss.item())
        np.savez_compressed(os.path.join(OUT, "stack3.npz"), **rec)
        print("stack3 ->", len(rec), "arrays")
    finally:
        torch.set_default_dtype(torch.float32)


if __name__ == "__main__":
    main()
