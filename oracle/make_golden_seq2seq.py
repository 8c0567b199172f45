"""Generate tests/golden/seq2seq.npz from the UNMODIFIED reference seq2seq module (seq2seq/model.py of the original).
Needs a checkout of the original project:  SN_REFERENCE_ROOT=<checkout> python -m oracle.make_golden_seq2seq
Contents (float64): weights of a Seq2Seq(E=12, H=16, V=61, layers=2); inputs; encoder forward (TF = 1 / 0 / 0.5, coin
stream random.seed(1234)) logits + final states + every gradient; emotion decoder forward + gradients; greedy
sample() ids of the encoder (batch 3) and of the factual / happy paths (batch 1) with livelier weights."""
import os
import random
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import reference_loader as rl          # noqa: E402
from oracle.port import synthetic_batch            # noqa: E402


def main():
    torch.set_default_dtype(torch.float64)
    mod = rl.load("seq2seq")
    E, H, V, L, B, T = 12, 16, 61, 2, 5, 7
    torch.manual_seed(0)
    m = mod.Seq2Seq(E, H, V, L, dropout=0.0, max_seq_length=9)
    m.max_seq_length = 9
    m.encoder.max_seq_length = 9
    for d in (m.decoder_happy, m.decoder_sad, m.decoder_angry):
        d.max_seq_length = 9
    rec = {"meta.E": E, "meta.H": H, "meta.V": V, "meta.L": L}
    for k, v in m.state_dict().items():
        rec["sd." + k] = v.numpy().copy()
    cap, lens, feats = synthetic_batch(B, T, V, E=E, ragged=True, seed=3)
    feats = feats.double()
    dst, dlens, _ = synthetic_batch(B, T - 1, V, ragged=True, seed=4)
    rec.update({"in.src": cap.numpy(), "in.src_lengths": np.asarray(lens), "in.features": feats.numpy(),
                "in.dst": dst.numpy(), "in.dst_lengths": np.asarray(dlens)})
    for tf, tag in ((1.0, "tf1"), (0.0, "tf0"), (0.5, "tf05")):
        random.seed(1234)
        m.zero_grad()
        out, (h, c) = m.encoder(feats, cap, lens, tf)
        out.logsumexp(1).sum().backward()
        rec["enc.%s.logits" % tag] = out.detach().numpy()
        rec["enc.%s.h" % tag], rec["enc.%s.c" % tag] = h.detach().numpy(), c.detach().numpy()
        for n, p in m.encoder.named_parameters():
            rec["enc.%s.grad.%s" % (tag, n)] = p.grad.numpy().copy()
    random.seed(1234)
    m.zero_grad()
    out = m(feats, (cap, lens), (dst, dlens), 1.0, "happy")
    out.logsumexp(1).sum().backward()
    rec["s2s.happy.logits"] = out.detach().numpy()
    for n, p in m.decoder_happy.named_parameters():
        rec["s2s.happy.grad." + n] = p.grad.numpy().copy()
    # decode: livelier weights so that the arg-max sequences are not constant
    g = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for p in m.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * (2.5 / (p.shape[-1] ** 0.5) if p.dim() > 1 else 0.3))
        for sub in (m.encoder, m.decoder_happy):
            sub.embed.weight.copy_(torch.randn(sub.embed.weight.shape, generator=g) * 1.5)
            sub.linear.weight.mul_(8.0 / 2.5)
    for k, v in m.state_dict().items():
        rec["lively.sd." + k] = v.numpy().copy()
    with torch.no_grad():
        ids, (h, c) = m.encoder.sample(feats[:3])
        rec["sample.enc.ids"], rec["sample.enc.h"], rec["sample.enc.c"] = ids.numpy(), h.numpy(), c.numpy()
        rec["sample.factual.ids"] = m.sample(feats[:1], 1, mode="factual").numpy()
        rec["sample.happy.ids"] = m.sample(feats[:1], 1, mode="happy").numpy()
    out_path = os.path.join(ROOT, "tests", "golden", "seq2seq.npz")
    np.savez_compressed(out_path, **rec)
    print("wrote", out_path, len(rec), "arrays;", "encoder ids", rec["sample.enc.ids"][0][:9], "happy", rec["sample.happy.ids"])


if __name__ == "__main__":
    main()
