"""CPU restatement ("port") of the reference caption-decoder hot path.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Plain PyTorch-on-CPU modules that
restate, independently written, what the reference's decoder classes compute, with the
same parameter names so ``state_dict``s interchange with both the reference modules and
the CUDA drop-in.  Every function cites the reference file:line it follows (paths
relative to the reference repository root).

Pin: ``tests/test_oracle_pin.py`` checks this port against golden vectors produced by
the unmodified reference modules (``oracle/make_golden.py`` -> ``tests/golden/*.npz``)
and, when ``SN_REFERENCE_ROOT`` names a checkout, against the live reference.  The reference
itself ships no tests or vectors ("parity unpinned" by upstream; SURVEY.md section 8c).

Semantics that matter (SURVEY.md "ten facts"):
  * FactoredLSTM cell has NO tanh on the cell output: h = o * c  (stylenet/model.py:152-153)
  * one ``random.random()`` coin per time step for the whole batch (stylenet/model.py:181)
  * non-teacher-forced input is B[argmax(previous logits)], step 0 uses captions[:,0]
    (stylenet/model.py:179,184)
  * ``sample()`` beam search bookkeeping (stylenet/model.py:198-294), integer ``//``
"""
import random
from typing import List, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

GATES = ("i", "f", "o", "c")
STYLES = ("factual", "happy", "sad", "angry")


def style_attr(style: str, gate: str) -> str:
    """Attribute name of the per-style S matrix (stylenet/model.py:56,61,66,71,76-91)."""
    return ("S_f" + gate) if style == "factual" else ("S_%s_%s" % (style, gate))


def att_attr(style: str) -> str:
    """Attribute name of the per-style attention net (stylenet/model_att.py:101,140,148,156)."""
    return "attention" if style == "factual" else "attention_" + style


def _ref_init(module: nn.Module, emb: nn.Embedding, out: nn.Linear) -> None:
    """reset_parameters + init_weights (stylenet/model.py:99-113, nic/model.py:58-72)."""
    for p in module.parameters():
        if p.dim() >= 2:
            nn.init.xavier_uniform_(p.data)
        else:
            nn.init.zeros_(p.data)
    emb.weight.data.uniform_(-0.1, 0.1)
    out.bias.data.fill_(0)
    out.weight.data.uniform_(-0.1, 0.1)


def batch_sizes_of(lengths: List[int]) -> List[int]:
    """b_t = #{b : L_b > t} -- what pack_padded_sequence(...).batch_sizes holds
    (stylenet/model.py:173-174).  ``lengths`` must be sorted descending."""
    assert all(lengths[i] >= lengths[i + 1] for i in range(len(lengths) - 1)), \
        "lengths must be sorted in decreasing order (pack_padded_sequence contract)"
    assert len(lengths) > 0 and lengths[-1] > 0
    return [sum(1 for L in lengths if L > t) for t in range(lengths[0])]


def pack_targets(captions: torch.Tensor, lengths: List[int]) -> torch.Tensor:
    """Time-major packed targets (stylenet/train_multitask.py:377-379)."""
    bs = batch_sizes_of(lengths)
    return torch.cat([captions[:b, t] for t, b in enumerate(bs)], 0)


# --------------------------------------------------------------------------------------
# beam search shared by every decoder (stylenet/model.py:198-294, model_att.py:307-426,
# nic/model.py:117-207, app/backend/model.py:386-487)
# --------------------------------------------------------------------------------------
def beam_search(step_fn, state, vocab_size, start_token, end_token, k, max_seq_length):
    """``step_fn(prev_words[s], state, step) -> (logits[s,V], state)``;
    ``state`` is a tuple of tensors whose dim 0 is the live-beam axis (re-ordered here)."""
    prev_words = torch.full((k,), start_token, dtype=torch.long)
    seqs = prev_words.unsqueeze(1)
    run_scores = torch.zeros(k, 1)
    done_seqs, done_scores = [], []
    step = 1
    while True:
        logits, state = step_fn(prev_words, state, step)
        scores = run_scores.expand_as(logits) + F.log_softmax(logits, dim=1)
        if step == 1:  # all beams identical: expand row 0 only (model.py:239-241)
            top_scores, top_idx = scores[0].topk(k, 0, True, True)
        else:
            top_scores, top_idx = scores.reshape(-1).topk(k, 0, True, True)
        src = top_idx // vocab_size           # model.py:249 (integer division)
        nxt = top_idx % vocab_size            # model.py:250
        seqs = torch.cat([seqs[src], nxt.unsqueeze(1)], 1)
        alive = [j for j in range(nxt.numel()) if int(nxt[j]) != end_token]
        dead = sorted(set(range(nxt.numel())) - set(alive))
        if dead:
            done_seqs.extend(seqs[dead].tolist())
            done_scores.extend(float(top_scores[j]) for j in dead)
        k -= len(dead)
        if k == 0:
            break
        seqs = seqs[alive]
        state = tuple(s[src[alive]] for s in state)
        run_scores = top_scores[alive].unsqueeze(1)
        prev_words = nxt[alive]
        if step > max_seq_length:             # model.py:283
            break
        step += 1
    if not done_scores:                       # model.py:288-289
        return torch.tensor([[end_token]], dtype=torch.long)
    best = done_scores.index(max(done_scores))  # first max, un-normalised (model.py:291)
    return torch.tensor([done_seqs[best]], dtype=torch.long)


class _FactoredBase(nn.Module):
    """Parameter set shared by the factored decoders (stylenet/model.py:52-94)."""

    def _build_factored(self, in_size, hidden_size, factored_size, vocab_size, bias):
        for g in GATES:
            setattr(self, "U_" + g, nn.Linear(factored_size, hidden_size, bias=bias))
            setattr(self, "V_" + g, nn.Linear(in_size, factored_size, bias=bias))
            setattr(self, "W_" + g, nn.Linear(hidden_size, hidden_size, bias=bias))
        for s in STYLES:
            for g in GATES:
                setattr(self, style_attr(s, g), nn.Linear(factored_size, factored_size, bias=bias))
        self.C = nn.Linear(hidden_size, vocab_size, bias=bias)

    def forward_step(self, embedded, states, mode):
        """One FactoredLSTM cell step (stylenet/model.py:115-155)."""
        h, c = states
        if mode not in STYLES:
            raise ValueError("mode name wrong: %r" % (mode,))
        z = {}
        for g in GATES:
            x = getattr(self, "V_" + g)(embedded)
            x = getattr(self, style_attr(mode, g))(x)
            z[g] = getattr(self, "U_" + g)(x) + getattr(self, "W_" + g)(h)
        i, f, o = torch.sigmoid(z["i"]), torch.sigmoid(z["f"]), torch.sigmoid(z["o"])
        c = f * c + i * torch.tanh(z["c"])
        h = o * c                              # no tanh (model.py:153)
        return h, (h, c)


class DecoderFactoredLSTM(_FactoredBase):
    """Restates stylenet/model.py:30-294."""

    def __init__(self, embed_size, hidden_size, factored_size, vocab_size, num_layers,
                 feature_size=2048, bias=True, dropout=0.22, max_seq_length=40):
        super().__init__()
        self.feature_size, self.hidden_size = feature_size, hidden_size
        self.vocab_size, self.max_seq_length = vocab_size, max_seq_length
        self.dropout = nn.Dropout(dropout)
        self.B = nn.Embedding(vocab_size, embed_size)
        self._build_factored(embed_size, hidden_size, factored_size, vocab_size, bias)
        _ref_init(self, self.B, self.C)

    def forward(self, captions, lengths, features=None, teacher_forcing_ratio=0.8,
                mode="factual", return_hidden=False):
        """stylenet/model.py:157-196."""
        emb = self.dropout(self.B(captions))
        if features is not None:
            emb = torch.cat([features.unsqueeze(1), emb], 1)
        bs = batch_sizes_of(list(lengths))
        B = captions.size(0)
        h = emb.new_zeros(B, self.hidden_size)
        c = emb.new_zeros(B, self.hidden_size)
        hs = []
        predicted = captions[:, 0]
        for t, b in enumerate(bs):
            if random.random() < teacher_forcing_ratio:
                x = emb[:b, t]
            else:
                x = self.B(predicted)[:b]
            hid, (h, c) = self.forward_step(x, (h[:b], c[:b]), mode)
            hs.append(hid)
            predicted = self.C(hid).max(1)[1]
        hs = torch.cat(hs, 0)
        out = self.C(hs)
        return (out, hs) if return_hidden else out

    def sample(self, features, start_token, end_token, k=5, factual_limit=-1,
               mode="factual", feed_image=False):
        """Beam search.  ``feed_image=False``: stylenet/model.py:198-294 (image never fed);
        ``feed_image=True``: app/backend/model.py:386-487 (image feature is the step-1 input)."""
        feat = features.reshape(1, -1)

        def step_fn(prev, state, step):
            if feed_image and step == 1:
                x = feat.expand(prev.numel(), -1)
            else:
                x = self.B(prev)
            hid, state = self.forward_step(x, state, mode)
            return self.C(hid), state

        z = torch.zeros(k, self.hidden_size)
        return beam_search(step_fn, (z, z.clone()), self.vocab_size, start_token, end_token,
                           k, self.max_seq_length)


class Attention(nn.Module):
    """Additive soft attention (stylenet/model_att.py:32-70)."""

    def __init__(self, encoder_dim, decoder_dim, attention_dim):
        super().__init__()
        self.encoder_att = nn.Linear(encoder_dim, attention_dim)
        self.decoder_att = nn.Linear(decoder_dim, attention_dim)
        self.full_att = nn.Linear(attention_dim, 1)

    def forward(self, encoder_out, decoder_hidden):
        att1 = self.encoder_att(encoder_out)
        att2 = self.decoder_att(decoder_hidden)
        e = self.full_att(torch.relu(att1 + att2.unsqueeze(1))).squeeze(2)
        alpha = torch.softmax(e, dim=1)
        return (encoder_out * alpha.unsqueeze(2)).sum(1), alpha


def _att_forward(dec, embed, captions, lengths, features, tf_ratio, attention, cell, return_hidden):
    """Shared teacher-forced unroll of the attention decoders
    (stylenet/model_att.py:238-305, nic/model_att.py forward)."""
    B = captions.size(0)
    feats = features.reshape(B, -1, features.size(-1))
    P = feats.size(1)
    emb = dec.dropout(embed(captions))
    bs = batch_sizes_of(list(lengths))
    h, c = dec.init_hidden_state(feats)
    alphas = emb.new_zeros(B, max(lengths), P)
    hs = []
    predicted = captions[:, 0]
    for t, b in enumerate(bs):
        awe, alpha = attention(feats[:b], h[:b])
        awe = torch.sigmoid(dec.f_beta(h[:b])) * awe
        if random.random() < tf_ratio:
            x = emb[:b, t]
        else:
            x = embed(predicted)[:b]
        hid, (h, c) = cell(torch.cat([x, awe], 1), (h[:b], c[:b]))
        hs.append(hid)
        alphas[:b, t] = alpha
        predicted = dec._out(hid).max(1)[1]
    hs = torch.cat(hs, 0)
    out = dec._out(hs)
    return (out, alphas, hs) if return_hidden else (out, alphas)


def _att_sample(dec, embed, features, start_token, end_token, k, attention, cell):
    """stylenet/model_att.py:307-426."""
    feats = features.reshape(1, -1, features.size(-1)).expand(k, -1, -1)
    h0, c0 = dec.init_hidden_state(feats)

    def step_fn(prev, state, step):
        h, c, fe = state
        awe, _ = attention(fe, h)
        awe = torch.sigmoid(dec.f_beta(h)) * awe
        hid, (h, c) = cell(torch.cat([embed(prev), awe], 1), (h, c))
        return dec._out(hid), (h, c, fe)

    return beam_search(step_fn, (h0, c0, feats), dec.vocab_size, start_token, end_token, k,
                       dec.max_seq_length)


class DecoderFactoredLSTMAtt(_FactoredBase):
    """Restates stylenet/model_att.py:73-426."""

    def __init__(self, attention_size, embed_size, hidden_size, factored_size, vocab_size,
                 num_layers, feature_size=2048, bias=True, dropout=0.22, max_seq_length=40):
        super().__init__()
        self.attention_size, self.feature_size = attention_size, feature_size
        self.hidden_size, self.vocab_size = hidden_size, vocab_size
        self.max_seq_length = max_seq_length
        self.init_h = nn.Linear(feature_size, hidden_size)
        self.init_c = nn.Linear(feature_size, hidden_size)
        self.dropout = nn.Dropout(dropout)
        for s in STYLES:
            setattr(self, att_attr(s), Attention(feature_size, hidden_size, attention_size))
        self.B = nn.Embedding(vocab_size, embed_size)
        self.f_beta = nn.Linear(hidden_size, feature_size)
        self._build_factored(embed_size + feature_size, hidden_size, factored_size, vocab_size, bias)
        _ref_init(self, self.B, self.C)

    def _out(self, h):
        return self.C(h)

    def init_hidden_state(self, feature):
        """stylenet/model_att.py:185-194."""
        m = feature.mean(dim=1)
        return self.init_h(m), self.init_c(m)

    def forward(self, captions, lengths, features, teacher_forcing_ratio=0.8, mode="factual",
                return_hidden=False):
        if mode not in STYLES:
            raise ValueError("mode name wrong: %r" % (mode,))
        att = getattr(self, att_attr(mode))
        cell = lambda x, st: self.forward_step(x, st, mode)
        return _att_forward(self, self.B, captions, lengths, features, teacher_forcing_ratio,
                            att, cell, return_hidden)

    def sample(self, features, start_token, end_token, k=5, factual_limit=-1, mode="factual"):
        att = getattr(self, att_attr(mode))
        cell = lambda x, st: self.forward_step(x, st, mode)
        return _att_sample(self, self.B, features, start_token, end_token, k, att, cell)


class DecoderRNN(nn.Module):
    """Restates nic/model.py:29-207 (nn.LSTMCell decoder)."""

    def __init__(self, embed_size, hidden_size, vocab_size, num_layers, feature_size=2048,
                 dropout=0.22, max_seq_length=40):
        super().__init__()
        self.feature_size, self.hidden_size = feature_size, hidden_size
        self.vocab_size, self.max_seq_length = vocab_size, max_seq_length
        self.dropout = nn.Dropout(dropout)
        self.embed = nn.Embedding(vocab_size, embed_size)
        self.lstm = nn.LSTMCell(embed_size, hidden_size, bias=True)
        self.linear = nn.Linear(hidden_size, vocab_size)
        _ref_init(self, self.embed, self.linear)

    def forward_step(self, embedded, states):
        """nic/model.py:74-79."""
        h, c = self.lstm(embedded, states)
        return h, (h, c)

    def forward(self, captions, lengths, features, teacher_forcing_ratio=0.8, return_hidden=False):
        """nic/model.py:81-115."""
        emb = self.dropout(self.embed(captions))
        emb = torch.cat([features.unsqueeze(1), emb], 1)
        bs = batch_sizes_of(list(lengths))
        B = captions.size(0)
        h = emb.new_zeros(B, self.hidden_size)
        c = emb.new_zeros(B, self.hidden_size)
        hs = []
        predicted = captions[:, 0]
        for t, b in enumerate(bs):
            if random.random() < teacher_forcing_ratio:
                x = emb[:b, t]
            else:
                x = self.embed(predicted)[:b]
            hid, (h, c) = self.forward_step(x, (h[:b], c[:b]))
            hs.append(hid)
            predicted = self.linear(hid).max(1)[1]
        hs = torch.cat(hs, 0)
        out = self.linear(hs)
        return (out, hs) if return_hidden else out

    def sample(self, features, start_token, end_token, k=5, feed_image=False):
        """nic/model.py:117-207 (``feed_image=True``: app/backend variant)."""
        feat = features.reshape(1, -1)

        def step_fn(prev, state, step):
            x = feat.expand(prev.numel(), -1) if (feed_image and step == 1) else self.embed(prev)
            hid, state = self.forward_step(x, state)
            return self.linear(hid), state

        z = torch.zeros(k, self.hidden_size)
        return beam_search(step_fn, (z, z.clone()), self.vocab_size, start_token, end_token,
                           k, self.max_seq_length)


class DecoderRNNAtt(nn.Module):
    """Restates nic/model_att.py:72-306 (LSTMCell(E+D,H) + one attention net)."""

    def __init__(self, attention_size, embed_size, hidden_size, vocab_size, num_layers,
                 feature_size=2048, dropout=0.22, max_seq_length=40):
        super().__init__()
        self.attention_size, self.feature_size = attention_size, feature_size
        self.hidden_size, self.vocab_size = hidden_size, vocab_size
        self.max_seq_length = max_seq_length
        self.init_h = nn.Linear(feature_size, hidden_size)
        self.init_c = nn.Linear(feature_size, hidden_size)
        self.dropout = nn.Dropout(dropout)
        self.attention = Attention(feature_size, hidden_size, attention_size)
        self.embed = nn.Embedding(vocab_size, embed_size)
        self.f_beta = nn.Linear(hidden_size, feature_size)
        self.lstm = nn.LSTMCell(embed_size + feature_size, hidden_size, bias=True)
        self.linear = nn.Linear(hidden_size, vocab_size)
        _ref_init(self, self.embed, self.linear)

    def _out(self, h):
        return self.linear(h)

    def init_hidden_state(self, feature):
        m = feature.mean(dim=1)
        return self.init_h(m), self.init_c(m)

    def forward_step(self, embedded, states):
        h, c = self.lstm(embedded, states)
        return h, (h, c)

    def forward(self, captions, lengths, features, teacher_forcing_ratio=0.8, return_hidden=False):
        return _att_forward(self, self.embed, captions, lengths, features, teacher_forcing_ratio,
                            self.attention, self.forward_step, return_hidden)

    def sample(self, features, start_token, end_token, k=5):
        return _att_sample(self, self.embed, features, start_token, end_token, k,
                           self.attention, self.forward_step)


# --------------------------------------------------------------------------------------
# loss + optimizer step around the decoder call (the L4 part of the hot path)
# --------------------------------------------------------------------------------------
def caption_loss(outputs, targets, alphas=None, alpha_c=1.0):
    """CrossEntropyLoss mean over packed tokens (stylenet/train_multitask.py:134,383);
    attention adds the doubly-stochastic term (train_multitask_att.py:409-411)."""
    loss = F.cross_entropy(outputs, targets)
    if alphas is not None:
        loss = loss + alpha_c * ((1.0 - alphas.sum(dim=1)) ** 2).mean()
    return loss


def clip_gradient(optimizer, grad_clip):
    """Element-wise clamp of every present gradient (stylenet/utils.py:51-60)."""
    for group in optimizer.param_groups:
        for p in group["params"]:
            if p.grad is not None:
                p.grad.data.clamp_(-grad_clip, grad_clip)


def train_step(decoder, optimizer, captions, lengths, features, mode=None, grad_clip=0.5,
               teacher_forcing_ratio=1.0, attention=False):
    """forward -> loss -> zero_grad -> backward -> clip -> Adam.step
    (stylenet/train_multitask.py:377-389; att: train_multitask_att.py:402-417)."""
    kw = {} if mode is None else {"mode": mode}
    if attention:
        lens = [l - 1 for l in lengths]
        targets = pack_targets(captions[:, 1:], lens)
        out, alphas = decoder(captions[:, :-1], lens, features,
                              teacher_forcing_ratio=teacher_forcing_ratio, **kw)
        loss = caption_loss(out, targets, alphas)
    else:
        targets = pack_targets(captions, lengths)
        out = decoder(captions, lengths, features, teacher_forcing_ratio=teacher_forcing_ratio, **kw)
        loss = caption_loss(out, targets)
    decoder.zero_grad()
    loss.backward()
    clip_gradient(optimizer, grad_clip)
    optimizer.step()
    return loss


def synthetic_batch(B, T, V, E=None, feat_shape=None, ragged=False, seed=0):
    """Synthetic inputs of SURVEY.md section 8d: captions ~ randint(4,V), col 0 = <start>=1, last
    token = <end>=2, lengths sorted descending (data_loader.py:133)."""
    g = torch.Generator().manual_seed(seed)
    cap = torch.randint(4, V, (B, T), generator=g)
    if ragged:
        lens = sorted(torch.randint(min(5, T), T + 1, (B,), generator=g).tolist(), reverse=True)
        lens[0] = T
    else:
        lens = [T] * B
    cap[:, 0] = 1
    for b, L in enumerate(lens):
        cap[b, L - 1] = 2
        cap[b, L:] = 0
    feats = None
    if feat_shape is not None:
        feats = torch.randn((B,) + tuple(feat_shape), generator=g)
    elif E is not None:
        feats = torch.randn(B, E, generator=g)
    return cap, lens, feats


def lively_weights(decoder, gain=1.5, out_gain=8.0, end_bias=2.0, end_token=2, seed=5):
    """Decode-test weights for SMALL models: with the reference init tiny models emit flat
    logits and beams never finish.  Re-draw every matrix ~ N(0, gain^2/fan_in), biases
    ~ N(0, 0.2^2), embedding ~ N(0,1), output projection ~ N(0, out_gain^2/H) and favour
    <end>.  Only used to build/consume decode fixtures (the weights themselves are stored)."""
    import math
    g = torch.Generator().manual_seed(seed)
    out = decoder.C if hasattr(decoder, "C") else decoder.linear
    emb = decoder.B if hasattr(decoder, "B") else decoder.embed
    with torch.no_grad():
        for p in decoder.parameters():
            if p.dim() >= 2:
                p.copy_(torch.randn(p.shape, generator=g, dtype=torch.float64) * gain / math.sqrt(p.shape[1]))
            else:
                p.copy_(torch.randn(p.shape, generator=g, dtype=torch.float64) * 0.2)
        emb.weight.copy_(torch.randn(emb.weight.shape, generator=g, dtype=torch.float64))
        out.weight.copy_(torch.randn(out.weight.shape, generator=g, dtype=torch.float64)
                         * out_gain / math.sqrt(out.weight.shape[1]))
        out.bias.zero_()
        out.bias[end_token] = end_bias


def sharpen_for_decode(decoder, end_token=2, scale=30.0, end_bias=2.0):
    """SURVEY.md section 8c decode recipe: with reference init the logits are flat and beams
    never end; scale the output projection and favour <end> so captions terminate."""
    out = decoder.C if hasattr(decoder, "C") else decoder.linear
    with torch.no_grad():
        out.weight.mul_(scale)
        out.bias[end_token] = end_bias
