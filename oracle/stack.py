"""Oracle of the multi-layer FactoredLSTM stack (BASELINE.json configs[3]) -- TEST INFRASTRUCTURE ONLY.

The reference ignores ``num_layers`` (stylenet/model.py:37), so the stack is an EXTENSION whose definition is this
file (SURVEY.md section 8c): ``layers`` is a list of decoder objects exposing the reference's
``forward_step(embedded, states, mode)`` (stylenet/model.py:115-155) -- oracle-port decoders, or the UNMODIFIED
reference ``DecoderFactoredLSTM`` objects when the original is checked out -- composed the way
``nn.LSTM(num_layers)`` composes cells (seq2seq/model.py:46-49):

    layer 0:  forward_step(x_t,            (h0, c0), mode)      embedding B / dropout / feature row of layers[0]
    layer l:  forward_step(h_t^{l-1},      (hl, cl), mode)      layers[l] built with embed_size = hidden_size
    logits:   layers[0].C(h_t^{top})

with the unroll, packing, teacher-forcing coin and arg-max feedback of stylenet/model.py:157-196 around it.
"""
import random

import torch

from oracle.port import batch_sizes_of


def stack_forward(layers, captions, lengths, features=None, teacher_forcing_ratio=0.8, mode="factual",
                  return_hidden=False):
    l0 = layers[0]
    emb = l0.dropout(l0.B(captions))                                     # model.py:166-167
    if features is not None:
        emb = torch.cat([features.unsqueeze(1), emb], 1)                 # model.py:170-171
    bs = batch_sizes_of(list(lengths))                                   # model.py:173-174
    Bn = captions.size(0)
    hs = [emb.new_zeros(Bn, l0.hidden_size) for _ in layers]             # model.py:176-177, per layer
    cs = [emb.new_zeros(Bn, l0.hidden_size) for _ in layers]
    tops = []
    predicted = captions[:, 0]                                           # model.py:179
    for t, b in enumerate(bs):
        if random.random() < teacher_forcing_ratio:                      # model.py:181
            x = emb[:b, t]
        else:
            x = l0.B(predicted)[:b]                                      # model.py:184
        for l, layer in enumerate(layers):
            x, (hs[l], cs[l]) = layer.forward_step(x, (hs[l][:b], cs[l][:b]), mode)   # model.py:185-186
        tops.append(x)
        predicted = l0.C(x).max(1)[1]                                    # model.py:189-191
    tops = torch.cat(tops, 0)
    out = l0.C(tops)                                                     # model.py:193-194
    return (out, tops) if return_hidden else out


def stack_parameters(layers):
    """Parameters the stack owns: everything of layer 0, and V/S/U/W of the upper layers (their B and C are unused)."""
    ps = list(layers[0].parameters())
    for layer in layers[1:]:
        ps += [p for n, p in layer.named_parameters() if not (n.startswith("B.") or n.startswith("C."))]
    return ps


def stack_forward_step(layers, embedded, states, mode):
    """One step through the stack: ``states = (h, c)`` with shape [num_layers, R, H]; layer l > 0 reads layer l-1's new
    h (stylenet/model.py:115-155 per layer, seq2seq/model.py:46-49 for the stacking).  Returns (h_top, (h', c'))."""
    h, c = states
    hs, cs = [], []
    x = embedded
    for l, layer in enumerate(layers):
        x, (hl, cl) = layer.forward_step(x, (h[l], c[l]), mode)
        hs.append(hl)
        cs.append(cl)
    return x, (torch.stack(hs, 0), torch.stack(cs, 0))


def stack_sample(layers, features, start_token, end_token, k=5, mode="factual", feed_image=False):
    """Beam search of stylenet/model.py:198-294 (``feed_image``: the app/backend variant) through the stack: the beam
    state is one (h, c) per layer, re-ordered together (oracle.port.beam_search moves every state tensor along dim 0)."""
    from oracle.port import beam_search
    l0 = layers[0]
    L, H = len(layers), l0.hidden_size
    feat = features.reshape(1, -1)

    def step_fn(prev, state, step):
        x = feat.expand(prev.numel(), -1) if (feed_image and step == 1) else l0.B(prev)
        new = []
        for l, layer in enumerate(layers):
            x, (hl, cl) = layer.forward_step(x, (state[2 * l], state[2 * l + 1]), mode)
            new += [hl, cl]
        return l0.C(x), tuple(new)

    z = torch.zeros(k, H, dtype=l0.C.weight.dtype)
    return beam_search(step_fn, tuple(z.clone() for _ in range(2 * L)), l0.vocab_size, start_token, end_token, k,
                       l0.max_seq_length)
