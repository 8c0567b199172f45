"""Multi-layer FactoredLSTM stack (BASELINE.json configs[3]: "3-layer FactoredLSTM factored_size 1024 multitask").

EXTENSION, not reference behaviour: every reference decoder accepts ``num_layers`` and ignores it
(stylenet/model.py:37).  The stack is DEFINED by composing reference pieces (SURVEY.md section 8c):

  * layer 0 is ``DecoderFactoredLSTM.forward_step`` as is (stylenet/model.py:115-155) -- same parameters, same names;
  * layer l > 0 is the same ``forward_step`` with ``embed_size = hidden_size`` (``V_g`` is ``[F, H]``), fed by layer
    l-1's ``h_t`` of the same time step -- the ``nn.LSTM(num_layers)`` convention of seq2seq/model.py:46-49;
  * zero initial state per layer, the vocabulary projection ``C`` reads the top layer, the style matrices ``S`` of
    every layer switch with ``mode``.

Its oracle (``oracle/stack.py``) instantiates reference decoders and calls their ``forward_step`` in that order.
Parameters of layer l > 0 are named ``l{l}_<reference name>`` (``l1_V_i.weight`` ...) and live in the same flat arena
as layer 0, so the fused clamp+Adam kernel, the CUDA-graph step and the data-parallel exchange are unchanged.

Kernel schedule: with teacher forcing a layer's input does not depend on its own output, so the stack runs
LAYER-MAJOR -- all time steps of layer l (time-batched factored projection on tcgen05 + one persistent recurrence
launch) before layer l+1; scheduled-sampling steps run the layers step by step.
"""
import torch
import torch.nn as nn

from . import ops
from .decoders import DecoderFactoredLSTM, GATES, STYLES, style_attr, _Ctx, _ref_init


class DecoderFactoredLSTMStack(DecoderFactoredLSTM):
    """``num_layers`` stacked FactoredLSTM cells behind the ``DecoderFactoredLSTM`` surface."""

    _layered = True          # decode keeps one (h, c) per layer

    def __init__(self, embed_size, hidden_size, factored_size, vocab_size, num_layers, feature_size=2048,
                 bias=True, dropout=0.22, max_seq_length=40):
        super().__init__(embed_size, hidden_size, factored_size, vocab_size, num_layers, feature_size, bias, dropout,
                         max_seq_length)
        if int(num_layers) < 1:
            raise ValueError("num_layers must be >= 1")
        self.num_layers = int(num_layers)
        for l in range(1, self.num_layers):
            lp = self._lp(l)
            for g in GATES:
                setattr(self, lp + "U_" + g, nn.Linear(factored_size, hidden_size, bias=bias))
                setattr(self, lp + "V_" + g, nn.Linear(hidden_size, factored_size, bias=bias))
                setattr(self, lp + "W_" + g, nn.Linear(hidden_size, hidden_size, bias=bias))
                for s in STYLES:
                    setattr(self, lp + style_attr(s, g), nn.Linear(factored_size, factored_size, bias=bias))
        _ref_init(self, self.B, self.C)

    # -- layout ------------------------------------------------------------------------------------
    def _arena_groups(self):
        groups = super()._arena_groups()
        for l in range(1, self.num_layers):
            lp = self._lp(l)
            for pre in ("V_", "U_", "W_"):
                groups.append([lp + pre + g + ".weight" for g in GATES])
                groups.append([lp + pre + g + ".bias" for g in GATES])
            for s in STYLES:
                groups.append([lp + style_attr(s, g) + ".weight" for g in GATES])
                groups.append([lp + style_attr(s, g) + ".bias" for g in GATES])
        return groups

    def _seq_grad_names(self, mode):
        names = super()._seq_grad_names(mode)
        for l in range(1, self.num_layers):
            lp = self._lp(l)
            for pre in ("V_", "U_", "W_"):
                names += [lp + pre + g + sfx for g in GATES for sfx in (".weight", ".bias")]
            names += [lp + style_attr(mode, g) + sfx for g in GATES for sfx in (".weight", ".bias")]
        return names

    def load_layer_state_dicts(self, layer_state_dicts):
        """Copy parameters from one reference-style ``DecoderFactoredLSTM`` state_dict per layer (layer 0 also gives
        ``B`` and ``C``; upper layers' own ``B``/``C`` are unused, as in the oracle composition)."""
        if len(layer_state_dicts) != self.num_layers:
            raise ValueError("need one state_dict per layer")
        own = dict(self.named_parameters())
        with torch.no_grad():
            for l, sd in enumerate(layer_state_dicts):
                lp = self._lp(l)
                for k, v in sd.items():
                    if l > 0 and (k.startswith("B.") or k.startswith("C.")):
                        continue
                    own[lp + k].copy_(v)
        return self

    # -- forward -------------------------------------------------------------------------------------
    def _upper_layers_init(self, c, save):
        plan = c.plan
        dev = c.XP.device
        H, N, B = self.hidden_size, plan.N, plan.B
        f32 = dict(dtype=torch.float32, device=dev)
        b16 = dict(dtype=torch.bfloat16, device=dev)
        use_tc = self.bf16 and H % 32 == 0
        upper = []
        for l in range(1, self.num_layers):
            cl = _Ctx()
            cl.layer, cl.mode, cl.plan, cl.Ein = l, c.mode, plan, H
            cl.save = save
            cl.w16 = {}
            cl.X = cl.Xb = None
            cl.XP = torch.empty(N, 4 * H, **f32)
            cl.Hall = torch.empty(N, H, **f32)
            cl.Call = torch.empty(N, H, **f32) if save else None
            cl.Hprev = torch.empty(N, H, **f32) if (save and not use_tc) else None
            cl.gates = torch.empty(N, 4 * H, **f32) if save else None
            cl.c_state = torch.zeros(B, H, **f32)
            # chain intermediates: allocated up front because scheduled sampling projects segment by segment
            F = self.factored_size
            cl.A1 = torch.empty(N, 4 * F, **(b16 if self.bf16 else f32))
            cl.A2 = torch.empty(N, 4 * F, **(b16 if self.bf16 else f32))
            if self.bf16 and not use_tc:
                cl.Xb = torch.empty(N, (H + 7) // 8 * 8, **b16)
            cl.Hb = cl.Hpb = None
            cl.Whh, cl.bhh = self._recurrent_weights(l)
            cl.ev_pre = None
            if self.bf16:
                # this layer's weight shadows are cast on the side stream while the layers below run
                specs = [(cl.w16, "V", self._stack("V_", (4 * F, H), layer=l)),
                         (cl.w16, "S", self._style_stack(c.mode, (4 * F, F), layer=l)),
                         (cl.w16, "U", self._stack("U_", (4 * H, F), layer=l))]
                if use_tc:
                    specs.append((cl.w16, "Whh", cl.Whh))
                cl.ev_pre = self._shadows_async(specs)
            if use_tc:
                cl.Hb = torch.empty(N, H, **b16)
                cl.Hpb = torch.empty(N, H, **b16) if save else None
            upper.append(cl)
        return upper

    def _upper_layers_fwd(self, c, t0, t1):
        """Steps t0..t1 of every layer above the first: project layer l-1's hidden rows of the segment through
        U S V (K2), then one recurrence launch over the segment (K3)."""
        plan = c.plan
        r0 = plan.off[t0]
        n = (plan.off[t1] if t1 < plan.T else plan.N) - r0
        below = c
        for cl in c.upper:
            if self.bf16 and below.Hb is not None:
                cl.Xb, X = below.Hb, None            # the recurrence below already wrote its h_t as the bf16 operand
            else:
                cl.X = X = below.Hall
            if cl.ev_pre is not None:
                torch.cuda.current_stream().wait_event(cl.ev_pre)
                cl.ev_pre = None
            self._input_projection(cl, X, c.mode, r0, n)
            self._recur_fwd(c, cl, t0, t1)
            below = cl

    # -- decode ----------------------------------------------------------------------------------------
    def forward_step(self, embedded, states, mode):
        """One step through all layers.  ``states = (h, c)`` with h, c of shape [num_layers, R, H] (the nn.LSTM
        convention, seq2seq/model.py:46-49); returns ``(h_top [R, H], (h', c'))``.  Layer l > 0 reads layer l-1's new h
        (oracle/stack.py::stack_forward_step)."""
        from .decode import single_step
        return single_step(self, embedded, states, mode)

    def sample(self, features, start_token, end_token, k=5, factual_limit=-1, mode="factual", feed_image=False):
        """Beam search with the reference's semantics (stylenet/model.py:198-294) through the stack: every live beam
        carries one (h, c) per layer (oracle/stack.py::stack_sample)."""
        from .decode import beam_sample, require_one_style
        require_one_style(mode)
        return beam_sample(self, features, start_token, end_token, k, mode, feed_image)[0]


class MultitaskSchedule:
    """The reference's multitask alternation (stylenet/train_multitask.py:192-235, 363-405, 511-557): a factual pass
    (``mode='factual'``, ``optimizer``, lr 2e-4) followed by one emotion pass per style tag in random order
    (``mode=tag``, ``lang_optimizer``, lr 5e-4) -- two optimizer objects with their own Adam moments over the SAME
    decoder parameters.  ``trainer_factual`` / ``trainer_emotion`` are DataParallelTrainer objects over one decoder."""

    def __init__(self, trainer_factual, trainer_emotion, tags=("happy", "sad", "angry")):
        self.fac, self.emo, self.tags = trainer_factual, trainer_emotion, tuple(tags)

    def step(self, factual_batch, emotion_batches):
        """``factual_batch``: (captions, lengths, features); ``emotion_batches``: {tag: (captions, lengths, features)}.
        Returns {pass name: loss tensor}."""
        out = {}
        cap, lengths, feat = factual_batch
        out["factual"] = self.fac.step(cap, lengths, feat, mode="factual")[0]
        for tag in self.tags:
            if tag in emotion_batches:
                cap, lengths, feat = emotion_batches[tag]
                out[tag] = self.emo.step(cap, lengths, feat, mode=tag)[0]
        return out
