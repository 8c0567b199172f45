"""Drop-in decoder modules: the reference's ``nn.Module`` surface (constructor arguments, parameter names,
``forward`` / ``forward_step`` / ``sample`` signatures) over the sm_100a kernels of libsn100.so.

Reference surfaces mirrored here:
  DecoderFactoredLSTM      stylenet/model.py:30-294
  DecoderRNN               nic/model.py:29-207
(the attention variants live in decoders_att.py)

Host logic only: packing plans, the teacher-forcing coin sequence (one ``random.random()`` per step,
stylenet/model.py:181), kernel sequencing and autograd glue.  All arithmetic runs in libsn100.so; there is
no PyTorch/CPU fallback -- tensors must be CUDA tensors on an sm_100 device.
"""
import random
from collections import OrderedDict

import os

import torch
import torch.nn as nn

from . import ops
from .arena import ParamArena
from .packing import get_plan

# greedy decoding under no_grad replays a CUDA graph from the second identical call on (see _forward_greedy)
GREEDY_GRAPH = [True]

GATES = ("i", "f", "o", "c")
STYLES = ("factual", "happy", "sad", "angry")


def style_attr(style, gate):
    return ("S_f" + gate) if style == "factual" else ("S_%s_%s" % (style, gate))


def _ref_init(module, emb, out):
    """reset_parameters + init_weights, stylenet/model.py:99-113 (host-side init, not on the path)."""
    for p in module.parameters():
        if p.dim() >= 2:
            nn.init.xavier_uniform_(p.data)
        else:
            nn.init.zeros_(p.data)
    emb.weight.data.uniform_(-0.1, 0.1)
    out.bias.data.fill_(0)
    out.weight.data.uniform_(-0.1, 0.1)


class _Ctx:
    """Activations saved between forward and backward of one sequence."""
    pass


class _HiddenFn(torch.autograd.Function):
    """captions/features -> Hall [N,H] through K1, K2, K3; backward publishes parameter gradients into
    the arena and returns d features."""

    @staticmethod
    def forward(ctx, anchor, features, dec, plan, captions, coins, mode, save):
        c = dec._run_forward(plan, captions, features, coins, mode, save=save)
        ctx.dec, ctx.c = dec, c
        ctx.need_dfeat = features is not None and features.requires_grad
        return c.top.Hall

    @staticmethod
    def backward(ctx, dHall):
        dec, c = ctx.dec, ctx.c
        gbuf = dec._grad_target(c.grad_names)
        dfeat = dec._run_backward(c, dHall.contiguous(), gbuf, ctx.need_dfeat)
        dec._publish(c.grad_names, gbuf)
        return None, dfeat, None, None, None, None, None, None


class _LogitsFn(torch.autograd.Function):
    """Hall -> logits [N,V] (the tensor the reference's forward() returns, stylenet/model.py:193-194)."""

    @staticmethod
    def forward(ctx, Hall, anchor, dec):
        ctx.dec = dec
        ctx.save_for_backward(Hall)
        return dec._vocab_logits(Hall)

    @staticmethod
    def backward(ctx, dlogits):
        dec = ctx.dec
        (Hall,) = ctx.saved_tensors
        gbuf = dec._grad_target(dec._out_names())
        dHall = dec._vocab_backward(Hall, dlogits.contiguous(), gbuf)
        dec._publish(dec._out_names(), gbuf)
        return dHall, None, None


def _pad8(n):
    return (n + 7) // 8 * 8


class _DecoderBase(nn.Module):
    """Shared host logic of the non-attention decoders."""

    cell = ops.CELL_FACTORED
    precision = "fp32"

    # per-process caches that must not travel with a pickled decoder (CUDA graphs, streams and events cannot be
    # pickled; the arena is rebuilt on first use).  The reference pickles the whole decoder every epoch
    # (save_checkpoint, stylenet/utils.py:62-90) and un-pickles it to resume (train_multitask.py:169-176).
    _TRANSIENT = ("_greedy_graphs", "_decode_sessions", "_side_streams", "_out_w16", "_out_w16_pref", "_out_w16_ev",
                  "_out_h16", "_seed_dev", "_arena", "_att_cache", "_gate_flag", "_gate_armed", "_after_recur", "_bucket_hook",
                  "_emb_early")

    def __getstate__(self):
        st = self.__dict__.copy()
        for k in self._TRANSIENT:
            st.pop(k, None)
        return st

    def set_precision(self, precision):
        """"fp32": every GEMM in fp32 FFMA (reference-exact mode, <=1e-5).  "bf16": GEMM operands in bf16 on
        the tcgen05 tensor cores, fp32 accumulation in TMEM; recurrence state, gate math, softmax/NLL,
        gradients-as-accumulated, master weights and Adam moments stay fp32 (SURVEY.md Appendix A)."""
        if precision not in ("fp32", "bf16"):
            raise ValueError("precision must be 'fp32' or 'bf16'")
        self.precision = precision
        return self

    @property
    def bf16(self):
        return self.precision == "bf16"

    def _shadow(self, w, rows=None, cols=None):
        """bf16 operand copy of a 2-D fp32 weight view, K padded to a multiple of 8 (TMA 16-byte rule)."""
        return ops.to_bf16_padded(w)

    # ---- arena ----------------------------------------------------------------------------------
    def _arena_groups(self):
        raise NotImplementedError

    def arena(self):
        a = self.__dict__.get("_arena")
        if a is None:
            a = ParamArena(self, self._arena_groups())
            self.__dict__["_arena"] = a
        return a.ensure()

    def _grad_target(self, names):
        """Flat buffer the backward kernels write: the gradient arena itself, or a zeroed temporary when
        one of the parameters about to be written already holds a gradient (accumulation across
        backward calls without zero_grad)."""
        a = self.arena()
        if any(a.named[n].grad is not None for n in names):
            return torch.zeros_like(a.gflat)
        return a.gflat

    def _publish(self, names, gbuf):
        self.arena().publish_grads(names, gbuf)

    def _side(self, i=0):
        """Side CUDA streams for work that is independent of the critical chain: weight-gradient GEMMs (each has only
        45-320 tiles, two of them side by side fill the 148 SMs where one cannot), bf16 weight shadows, loss
        bookkeeping.  Works eagerly and under CUDA-graph capture (fork/join become parallel graph branches).
        Stream 0 and 1 carry the weight gradients, stream 2 the weight shadows of the forward pass."""
        sts = self.__dict__.setdefault("_side_streams", {})
        st = sts.get(i)
        if st is None:
            st = torch.cuda.Stream()
            sts[i] = st
        return st

    def _fork(self, i=0):
        side = self._side(i)
        side.wait_stream(torch.cuda.current_stream())
        return side

    def _join(self):
        for st in self.__dict__.get("_side_streams", {}).values():
            torch.cuda.current_stream().wait_stream(st)

    def _take_out_shadow(self):
        """The prefetched bf16 shadow of the vocabulary weight (or None), after making the current stream wait for it."""
        Wb = self.__dict__.pop("_out_w16_pref", None)
        ev = self.__dict__.pop("_out_w16_ev", None)
        if Wb is not None and ev is not None:
            torch.cuda.current_stream().wait_event(ev)
        return Wb

    def _shadows_async(self, specs, max_blocks=24):
        """bf16 operand shadows of fp32 weights, cast on side stream 2 while the main stream gathers / projects.
        ``specs``: [(dict, key, fp32 2-D weight)].  The output tensors are allocated on the CURRENT stream (so the
        caching allocator ties their lifetime to it) and only written on the side stream.  Returns the event the main
        stream must wait for before the first use (``_shadows_wait``)."""
        main = torch.cuda.current_stream()
        outs = []
        for dct, key, w in specs:
            R, C = w.shape
            Cp = (C + 7) // 8 * 8
            out = torch.empty(R, Cp, dtype=torch.bfloat16, device=w.device)
            dct[key] = out
            outs.append((w, out, R, C, Cp))
        side = self._side(2)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            for w, out, R, C, Cp in outs:
                ops.cast_bf16(w, R, C, w.stride(0), out, Cp, Cp, max_blocks=max_blocks)
            ev = torch.cuda.Event()
            ev.record(side)
        return ev

    def _next_seed(self, dev, p_drop):
        """Dropout randomness = hash(seed + device counter, row, col).  The counter lives in device memory
        and is bumped by a (graph-capturable) device op once per forward, so CUDA-graph replays draw a fresh
        mask every step."""
        base = int(self.__dict__.get("_seed", 0x5EED)) * 1000003
        if p_drop <= 0.0:
            return base, None
        sd = self.__dict__.get("_seed_dev")
        if sd is None or sd.device != dev:
            sd = torch.zeros(1, dtype=torch.int64, device=dev)
            self.__dict__["_seed_dev"] = sd
        sd.add_(1)
        return base, sd

    def _check_inputs(self, captions, features):
        if not captions.is_cuda:
            raise ops._lib.SnError("decoder inputs must be CUDA tensors: this path has no CPU fallback")
        ops.lib()

    # ---- pieces each subclass provides -----------------------------------------------------------
    def _emb(self):
        raise NotImplementedError

    def _out(self):
        raise NotImplementedError

    def _input_projection(self, c, X, mode, r0, n):
        raise NotImplementedError

    def _input_projection_bwd(self, c, dZ, gbuf):
        raise NotImplementedError

    # ---- forward ---------------------------------------------------------------------------------
    def _coins(self, T, teacher_forcing_ratio):
        # one coin per time step for the whole batch, drawn from Python's global RNG exactly like the
        # reference (stylenet/model.py:181); drawing them up front consumes the same stream.
        return [random.random() < teacher_forcing_ratio for _ in range(T)]

    def _run_forward(self, plan, captions, features, coins, mode, save):
        a = self.arena()
        dev = captions.device
        d = plan.dev(dev)
        H, N, B, T = self.hidden_size, plan.N, plan.B, plan.T
        emb = self._emb()
        E = emb.weight.shape[1]
        has_feat = features is not None
        c = _Ctx()
        c.plan, c.mode, c.has_feat, c.captions = plan, mode, has_feat, captions
        c.p_drop = float(self.dropout.p) if self.training else 0.0
        c.seed, c.seed_dev = self._next_seed(dev, c.p_drop)
        feats = None
        if has_feat:
            feats = features.detach()
            if feats.dtype != torch.float32 or not feats.is_contiguous():
                feats = feats.float().contiguous()
            if feats.dim() == 3:
                feats = feats.reshape(feats.shape[0], -1)
        all_tf = all(coins)
        c.tok_override = None
        if not all_tf:
            c.tok_override = torch.full((N,), -1, dtype=torch.int32, device=dev)
        c.emb_ws = c.emb_ev = c.emb_zeroed = None
        if self.__dict__.pop("_emb_early", False) and all_tf:
            # the token grouping of the embedding backward needs only the captions and the plan, and nothing reads the
            # embedding's gradient between the previous step's Adam and the backward's group sums: both run here, on
            # a side stream next to the forward, instead of on the tail of the step
            V = emb.weight.shape[0]
            c.emb_ws = ops.embed_plan_ws(V, N, dev)      # allocated on the current stream, written on the side stream
            c.emb_zeroed = a.gflat
            gE = self._gview(a.gflat, [self._emb_name()], emb.weight.shape)
            side = self._side(4)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                ops.embed_plan(captions, has_feat, d["row_b"], d["row_t"], None, N, V, c.emb_ws)
                gE.zero_()
                c.emb_ev = torch.cuda.Event()
                c.emb_ev.record(side)
        c.Ein = E
        c.w16 = {}      # bf16 weight shadows of this call (refreshed every forward)
        c.ev_early = c.ev_late = c.ev_first = None
        if self.bf16:
            # every weight shadow is cast on a side stream: the first GEMM's at full width next to the gather (it is on
            # the critical path), the others throttled (24 CTAs) under the gather / first GEMM
            early, late = self._shadow_specs(c, mode)
            first = c.__dict__.pop("first_specs", None)
            if first:
                c.ev_first = self._shadows_async(first, max_blocks=0)
            second = c.__dict__.pop("second_specs", None)
            c.ev_second = self._shadows_async(second, max_blocks=0) if second else None
            if early:
                c.ev_early = self._shadows_async(early)
            if late:
                c.ev_late = self._shadows_async(late)
            # the vocabulary weight (the largest cast) is only needed after the recurrence: its own event
            self.__dict__["_out_w16_ev"] = self._shadows_async([(self.__dict__, "_out_w16_pref", self._out().weight)])
        if self.bf16:
            # bf16 mode: the packed input rows are produced directly as the K-padded bf16 GEMM operand
            X = None
            c.Xb = torch.empty(N, _pad8(E), dtype=torch.bfloat16, device=dev)
        else:
            X = torch.empty(N, E, dtype=torch.float32, device=dev)
            c.Xb = None
        ops.gather_pack_fwd(captions, emb.weight, feats, has_feat, d["row_b"], d["row_t"], None, N, X,
                            c.p_drop, c.seed, seed_dev=c.seed_dev, Xb=c.Xb)
        c.X = X
        c.XP = torch.empty(N, 4 * H, dtype=torch.float32, device=dev)
        self._input_projection(c, X, mode, 0, N)
        c.Hall = torch.empty(N, H, dtype=torch.float32, device=dev)
        c.Call = torch.empty(N, H, dtype=torch.float32, device=dev) if save else None
        c.Hprev = torch.empty(N, H, dtype=torch.float32, device=dev) if save else None
        c.gates = torch.empty(N, 4 * H, dtype=torch.float32, device=dev) if save else None
        c_state = torch.zeros(B, H, dtype=torch.float32, device=dev)
        c.aux_argmax = None
        Whh, bhh = self._recurrent_weights()
        c.Whh, c.bhh = Whh, bhh
        use_tc = self.bf16 and H % 32 == 0
        c.Hb = c.Hpb = None
        if c.ev_late is not None:
            torch.cuda.current_stream().wait_event(c.ev_late)
        if use_tc:
            if "Whh" not in c.w16:
                c.w16["Whh"] = self._shadow(Whh)
            c.Hb = torch.empty(N, H, dtype=torch.bfloat16, device=dev)
            c.Hpb = torch.empty(N, H, dtype=torch.bfloat16, device=dev) if save else None
            c.Hprev = None
        c.upper = self._upper_layers_init(c, save)     # layers above the first (stack.py); [] for the reference models
        c.top = c.upper[-1] if c.upper else c

        c.c_state = c_state

        def run(t0, t1):
            self._recur_fwd(c, c, t0, t1)
            if c.upper:
                self._upper_layers_fwd(c, t0, t1)

        if all_tf:
            run(0, T)
        else:
            out = self._out()
            V = out.weight.shape[0]
            pred = captions[:, 0].to(torch.int32).contiguous()      # model.py:179
            am = torch.empty(B, dtype=torch.int64, device=dev)
            t = 0
            while t < T:
                if coins[t]:
                    t1 = t
                    while t1 < T and coins[t1]:
                        t1 += 1
                    run(t, t1)
                    t = t1
                else:
                    bt, r0 = plan.bs[t], plan.off[t]
                    if t > 0:
                        # predicted = argmax C(h_{t-1})  (model.py:189-191), lowest index on ties
                        bp, rp = plan.bs[t - 1], plan.off[t - 1]
                        lg = torch.empty(bp, V, dtype=torch.float32, device=dev)
                        ops.gemm(ops.OP_NT, c.top.Hall, out.weight, lg, bp, V, H, H, H, V, bias=out.bias,
                                 a_off=rp * H)
                        ops.softmax_nll(lg, bp, V, argmax=am)
                        pred = am[:bp].to(torch.int32)
                    c.tok_override[r0:r0 + bt] = pred[:bt]
                    ops.gather_pack_fwd(captions, emb.weight, feats, has_feat, d["row_b"], d["row_t"],
                                        c.tok_override, bt, X, c.p_drop, c.seed, row_off=r0, seed_dev=c.seed_dev,
                                        Xb=c.Xb)
                    self._input_projection(c, X, mode, r0, bt)
                    run(t, t + 1)
                    t += 1
        c.grad_names = self._seq_grad_names(mode)
        c.feat_shape = None if features is None else features.shape
        if not save:
            c.X = c.XP = None
        return c

    def _recur_fwd(self, c, cl, t0, t1):
        """K3 forward of one layer over steps [t0, t1).  Two kernels behind one call: the persistent, latency-optimised
        recurrence (any batch, any segment) and -- for whole teacher-forced sequences of >= ops.RECUR_GEMM_MIN_BATCH
        samples in bf16 mode -- one tcgen05 GEMM per step with the cell fused into the epilogue (throughput regime)."""
        plan = c.plan
        d = plan.dev(cl.XP.device)
        H, B, T = self.hidden_size, plan.B, plan.T
        Whh, bhh = cl.Whh, cl.bhh          # cached per forward: arena lookups are host work, this runs once per segment
        if cl.Hb is not None:
            if t0 == 0 and t1 == T and B >= ops.RECUR_GEMM_MIN_BATCH[0] and H % 64 == 0:
                if "Whh_il" not in cl.w16:
                    cl.w16["Whh_il"] = ops.cast_gate_interleave(Whh)
                if cl.Call is None:
                    cl.Call = torch.empty(plan.N, H, dtype=torch.float32, device=cl.XP.device)
                ops.recur_fwd_gemm(self.cell, H, B, plan, cl.XP, cl.w16["Whh_il"], bhh, cl.Hall, cl.Hb, cl.Call, cl.gates)
                if cl.Hpb is not None:
                    ops.recur_hprev(cl.Hb, d, plan.N, H, cl.Hpb)
                cl.recur_gemm = True
                return
            h_init = cl.Hall[plan.off[t0 - 1]:] if t0 > 0 else None
            ops.recur_fwd_bf16(self.cell, H, B, d["bs"], d["off"], t0, t1, cl.XP, cl.w16["Whh"], bhh, h_init,
                               cl.Hall, cl.Hb, cl.Hpb, cl.Call, cl.gates, cl.c_state)
        else:
            h_init = cl.Hall[plan.off[t0 - 1]:] if t0 > 0 else None
            ops.recur_fwd(self.cell, H, B, d["bs"], d["off"], t0, t1, cl.XP, Whh, bhh, h_init, cl.Hall,
                          cl.Call, cl.Hprev, cl.gates, cl.c_state)

    def _shadow_specs(self, c, mode):
        """(early, late) lists of (dict, key, fp32 weight) to cast to bf16 on the side stream at the start of a forward:
        `early` = needed by the second GEMM of the input projection, `late` = needed from the recurrence on."""
        H = self.hidden_size
        late = []
        if H % 32 == 0:
            late.append((c.w16, "Whh", self._recurrent_weights()[0]))
        return [], late

    def _upper_layers_init(self, c, save):
        return []

    def _upper_layers_fwd(self, c, t0, t1):
        pass

    def _layer_bwd(self, c, cl, dHall, gbuf):
        """Reverse-time recurrence of ONE layer (K3 backward), its recurrent weight / bias gradients and the
        backward of its input projection.  ``cl`` holds the layer's saved activations (``c`` itself for the first
        layer).  Returns the gradient w.r.t. the layer's input rows [N, Ein]."""
        plan = c.plan
        dev = dHall.device
        d = plan.dev(dev)
        H, N, B, T = self.hidden_size, plan.N, plan.B, plan.T
        L = getattr(cl, "layer", 0)
        Whh, _ = self._recurrent_weights(L)
        dZ = torch.empty(N, 4 * H, dtype=torch.float32, device=dev)
        dhc = torch.zeros(2, B, H, dtype=torch.float32, device=dev)      # (one fill kernel in front of the recurrence)
        dh, dc = dhc[0], dhc[1]
        gW, gbW = self._recurrent_grads(gbuf, L)
        if cl.Hpb is not None:
            cl.dZb = torch.empty(N, 4 * H, dtype=torch.bfloat16, device=dev)
            if getattr(cl, "recur_gemm", False):
                ops.recur_bwd_gemm(self.cell, H, B, plan, cl.w16["Whh"], cl.Call, cl.gates, dHall, dZ, cl.dZb, dc)
            else:
                ops.recur_bwd_bf16(self.cell, H, B, d["bs"], d["off"], 0, T, cl.w16["Whh"], None, cl.Call, cl.gates,
                                   dHall, dZ, cl.dZb, dh, dc, start_flag=self.__dict__.pop("_gate_armed", None))
            self._run_deferred()
            with torch.cuda.stream(self._fork()):
                ops.gemm_bf16(ops.OP_TN, cl.dZb, cl.Hpb, 4 * H, H, N, 4 * H, H, C=gW, ldc=H)
                ops.colsum(dZ, N, 4 * H, 4 * H, gbW, wide=bool(ops.TAIL_SCHEDULE[0]))
            # d b_U (factored input projection) is the same column sum of dZ: copied from d b_hh on this side stream
            cl.colsum_dZ = gbW if ops.TAIL_SCHEDULE[0] else None
            return self._input_projection_bwd(cl, dZ, gbuf)
        ops.recur_bwd(self.cell, H, B, d["bs"], d["off"], 0, T, Whh, None, cl.Call, cl.gates, dHall, dZ, dh, dc)
        # dW_hh = dZ^T Hprev ; d b_hh = colsum(dZ)
        if self.bf16:
            cl.dZb = ops.to_bf16_padded(dZ)
            Hpb = ops.to_bf16_padded(cl.Hprev)
            ops.gemm_bf16(ops.OP_TN, cl.dZb, Hpb, 4 * H, H, N, 4 * H, H, C=gW, ldc=H)
        else:
            ops.gemm(ops.OP_TN, dZ, cl.Hprev, gW, 4 * H, H, N, 4 * H, H, H)
        ops.colsum(dZ, N, 4 * H, 4 * H, gbW)
        return self._input_projection_bwd(cl, dZ, gbuf)

    def _run_backward(self, c, dHall, gbuf, need_dfeat):
        for cl in reversed(c.upper):
            dHall = self._layer_bwd(c, cl, dHall, gbuf)      # d(input of layer l) = d(hidden states of layer l-1)
        dX = self._layer_bwd(c, c, dHall, gbuf)
        out = self._embedding_bwd(c, dX, gbuf, need_dfeat)
        self._join()
        return out

    def _embedding_bwd(self, c, dX, gbuf, need_dfeat):
        plan = c.plan
        dev = dX.device
        d = plan.dev(dev)
        N, B = plan.N, plan.B
        emb = self._emb()
        E = emb.weight.shape[1]
        gE = self._gview(gbuf, [self._emb_name()], emb.weight.shape)
        dfeat = torch.empty(B, E, dtype=torch.float32, device=dev) if (need_dfeat and c.has_feat) else None
        if getattr(c, "emb_ws", None) is not None:
            # grouping and zeroing were issued by the forward (_run_forward): only the group sums are left
            torch.cuda.current_stream().wait_event(c.emb_ev)
            if gbuf is not c.emb_zeroed:
                gE.zero_()
            ops.embed_grad(gE, dfeat, c.has_feat, d["row_b"], d["row_t"], c.tok_override, N, dX, c.p_drop, c.seed,
                           c.emb_ws, seed_dev=c.seed_dev, wide=True)
        else:
            gE.zero_()
            ops.gather_pack_bwd(c.captions, gE, dfeat, c.has_feat, d["row_b"], d["row_t"], c.tok_override, N, dX,
                                c.p_drop, c.seed, seed_dev=c.seed_dev)
        if dfeat is not None and c.feat_shape is not None:
            dfeat = dfeat.view(c.feat_shape)
        # the embedding is the last gradient of the step: its bucket starts right here, next to the W_hh / U and S / V
        # buckets still running on the side streams, instead of behind the join of all of them
        self._bucket_final([self._emb_name()])
        return dfeat

    def _run_deferred(self):
        """Side-stream work of the vocabulary backward that was held back until the reverse recurrence was launched."""
        todo = self.__dict__.pop("_after_recur", None)
        for fn in todo or ():
            fn()

    def _bucket_final(self, names):
        """The gradients of ``names`` are final (all their kernels are queued on the CURRENT stream): publish them and
        let the trainer exchange / update this bucket now, under the rest of the backward."""
        hook = self.__dict__.get("_bucket_hook")
        if hook is None:
            return
        gbuf, fn = hook
        names = [n for n in names if n in self.arena().named]
        self._publish(names, gbuf)
        fn(names)

    def _gview(self, gbuf, names, shape):
        a = self.arena()
        o, n = a._span(names)
        return gbuf[o:o + n].view(shape)

    # ---- vocabulary projection ---------------------------------------------------------------------
    def _vocab_logits(self, Hall, Hb=None):
        out = self._out()
        if self.bf16:
            V, H = out.weight.shape
            N = Hall.shape[0]
            if Hb is None:
                Hb = ops.to_bf16_padded(Hall.contiguous())
            Wb = self._take_out_shadow()
            if Wb is None:
                Wb = ops.to_bf16_padded(out.weight)
            self.__dict__["_out_w16"] = Wb          # reused by the matching backward of this step
            logits = torch.empty(N, V, dtype=torch.float32, device=Hall.device)
            ops.gemm_bf16(ops.OP_NT, Hb, Wb, N, V, H, Hb.stride(0), Wb.stride(0), C=logits, ldc=V, bias=out.bias)
            return logits
        return ops.linear_nt(Hall.contiguous(), out.weight, out.bias)

    def _vocab_backward(self, Hall, dlogits, gbuf, Hb=None, dLb=None, defer=None, gate_B=None):
        out = self._out()
        V, H = out.weight.shape
        N = Hall.shape[0]
        wn, bn = self._out_names()
        gC = self._gview(gbuf, [wn], (V, H))
        gb = self._gview(gbuf, [bn], (V,))
        dHall = torch.empty(N, H, dtype=torch.float32, device=Hall.device)
        if self.bf16:
            have_b16 = dLb is not None
            if not have_b16:
                dLb = ops.to_bf16_padded(dlogits)
            hb_stash = self.__dict__.pop("_out_h16", None)
            if Hb is None:
                Hb = hb_stash if (have_b16 and hb_stash is not None) else ops.to_bf16_padded(Hall.contiguous())
            Wb = self.__dict__.pop("_out_w16", None) if dLb is not None and have_b16 else None
            if Wb is None:
                Wb = ops.to_bf16_padded(out.weight)
            if have_b16:
                # dH feeds the reverse recurrence: issued FIRST so its tiles get the SMs; dC / db_C do not feed anything
                # before Adam: side stream, joined by the caller (_join)
                mode_dc = ops.DC_SCHEDULE[0] if defer is not None else 0
                side = self._side(0)
                if mode_dc != 2:
                    side.wait_stream(torch.cuda.current_stream())           # dLb / Hb exist
                ops.gemm_bf16(ops.OP_NN, dLb, Wb, N, H, V, dLb.stride(0), Wb.stride(0), C=dHall, ldc=H)
                if mode_dc == 1:
                    # the cluster-form recurrence needs 16 completely free SMs per cluster: dC must not grab SMs before its
                    # clusters are placed.  dC becomes runnable together with the recurrence (both wait for dH) but is
                    # LAUNCHED after it, and is capped to the SMs the 6 clusters leave free.
                    side.wait_stream(torch.cuda.current_stream())

                gate = None
                if mode_dc == 0 and gate_B is not None and ops.GATE_DC[0] and ops.recur_cluster_ok(H, gate_B):
                    # the cluster-form reverse recurrence needs 16 completely free SMs per cluster: everything queued on
                    # this side stream (dC, db_C, the bucket's exchange / Adam) waits behind a gate that opens once the
                    # recurrence's CTAs are resident, and then runs on the SMs it leaves free
                    gate = self.__dict__.get("_gate_flag")
                    if gate is None or gate.device != dHall.device:
                        gate = self.__dict__["_gate_flag"] = torch.zeros(3, dtype=torch.int32, device=dHall.device)
                    self.__dict__["_gate_armed"] = gate

                def side_work():
                    if mode_dc == 2:
                        side.wait_stream(torch.cuda.current_stream())       # after the reverse recurrence, full width
                    with torch.cuda.stream(side):
                        if gate is not None:
                            ops.gate_wait(gate)
                        ops.gemm_bf16(ops.OP_TN, dLb, Hb, V, H, N, dLb.stride(0), Hb.stride(0), C=gC, ldc=H,
                                      max_pairs=0 if mode_dc == 2 else ops.DC_MAX_PAIRS[0])
                        ops.colsum_bf16(dLb, N, V, dLb.stride(0), gb, wide=bool(ops.TAIL_SCHEDULE[0]))
                if mode_dc == 0:
                    side_work()
                else:
                    defer.append(side_work)
                return dHall
            ops.gemm_bf16(ops.OP_NN, dLb, Wb, N, H, V, dLb.stride(0), Wb.stride(0), C=dHall, ldc=H)
            ops.gemm_bf16(ops.OP_TN, dLb, Hb, V, H, N, dLb.stride(0), Hb.stride(0), C=gC, ldc=H)
        else:
            ops.gemm(ops.OP_NN, dlogits, out.weight, dHall, N, H, V, dlogits.stride(0), H, H)
            ops.gemm(ops.OP_TN, dlogits, Hall, gC, V, H, N, dlogits.stride(0), H, H)
        ops.colsum(dlogits, N, V, dlogits.stride(0), gb)
        return dHall

    def _vocab_nll(self, Hall, Hb, targets, denom, backward, row_weight=None):
        """Vocabulary projection + log-softmax + NLL (+ gradient w.r.t. the logits) + arg-max + top-5
        (stylenet/model.py:193-194, train_multitask.py:377-383, utils.py:127-140).
        bf16 mode: K5 fused with the projection -- logits live only in TMEM, never in HBM.  Pass 1 -> log-sum-exp,
        target logit, loss, arg-max; pass 2 recomputes the tiles and emits the gradient directly as the bf16
        operand of the dH / dC GEMMs (or only ranks the target when not training).
        fp32 mode: fp32 FFMA logits + the one-pass softmax kernel (gradient in place).
        ``row_weight`` (float32 [N] or None): the gradient of row r is scaled by row_weight[r].
        Returns (row_loss, argmax, top5hit, dlogits_fp32 | None, dlogits_bf16 | None)."""
        out = self._out()
        V, H = out.weight.shape
        N, dev = Hall.shape[0], Hall.device
        row_loss = torch.empty(N, dtype=torch.float32, device=dev)
        argmax = torch.empty(N, dtype=torch.int64, device=dev)
        top5 = torch.empty(N, dtype=torch.int32, device=dev)
        if self.bf16:
            if Hb is None:
                Hb = ops.to_bf16_padded(Hall.contiguous())
            Wb = self._take_out_shadow()                      # cast on the side stream at the start of the forward
            if Wb is None:
                Wb = ops.to_bf16_padded(out.weight)
            self.__dict__["_out_w16"] = Wb              # reused by the matching _vocab_backward
            self.__dict__["_out_h16"] = Hb
            tl = torch.empty(N, dtype=torch.float32, device=dev)
            lse = torch.empty(N, dtype=torch.float32, device=dev)
            above = torch.empty(N, dtype=torch.int32, device=dev)
            ops.vocab_nll_fwd(Hb, Wb, out.bias, targets, N, V, H, tl, lse, row_loss=row_loss, argmax=argmax, above=above)
            dLb = torch.empty(N, _pad8(V), dtype=torch.bfloat16, device=dev) if backward else None
            ops.vocab_nll_bwd(Hb, Wb, out.bias, targets, N, V, H, tl, lse, 1.0 / denom, dLb=dLb, above=above,
                              top5hit=top5, row_weight=row_weight)
            return row_loss, argmax, top5, None, dLb
        logits = self._vocab_logits(Hall, Hb)
        ops.softmax_nll(logits, N, V, targets=targets, row_loss=row_loss, dlogits=logits if backward else None,
                        grad_scale=1.0 / denom, argmax=argmax, top5hit=top5, row_weight=row_weight)
        return row_loss, argmax, top5, logits, None

    # ---- sampling decode (self-critical training, scst.py) ----------------------------------------------------------
    def sample_captions(self, features, start_token, end_token, n=1, temperature=1.0, seed=0, mode="factual",
                        greedy=False):
        """Draw ``n`` captions for each row of ``features [n_img, E]`` (K12, one pass over each step's logits with the
        bookkeeping on the device; dropout off).  Returns device tensors
          seqs     int64 [n_img * n, max_seq_length + 2], zero-padded; row i * n + j = sample j of image i,
                   [<start>, w1, ..., <end>] (no <end> when the row ran out of steps);
          lengths  int64 [n_img * n], counting <start> and <end>;
          logprob  float32 [n_img * n, max_seq_length + 1]: column t - 1 = log-probability at temperature 1 of the
                   token drawn at step t (zeros after the row's end).
        Conditioning: step 0 feeds the image feature and discards its output, step 1 feeds <start>, step t the token
        drawn at step t - 1; a row stops at its first <end> or after max_seq_length + 1 draws.  This is exactly the
        teacher-forced ``forward_loss(seqs, lengths, features)``, so a sample is trained on as it is.  It is neither of
        ``sample()``'s semantics: the reference's beam search never feeds the image, and ``feed_image=True`` (the app
        back end) takes the first word from the image step.
        Draw: token = argmax_v logit_v / temperature + g_v, Gumbel noise from a counter-based hash of (seed, step, row,
        v) (include/sn100.h, sn_sample_step); ties to the lowest index.  ``greedy=True``: the plain arg-max.  The same
        seed gives the same samples, eagerly or replayed from the session's CUDA graphs.
        ``mode``: one style name (factored decoders; ignored by DecoderRNN).  Raises ValueError, before any device
        work, for n < 1, a temperature that is not finite or not > 0, a seed outside 0 .. 2^63 - 1 and a style list."""
        import math
        import numbers
        from .decode import sample_decode
        if isinstance(n, bool) or not isinstance(n, numbers.Integral) or n < 1:
            raise ValueError("n must be an integer >= 1; got %r" % (n,))
        if not isinstance(temperature, numbers.Real) or not math.isfinite(temperature) or not temperature > 0:
            raise ValueError("temperature must be finite and > 0; got %r" % (temperature,))
        if isinstance(seed, bool) or not isinstance(seed, numbers.Integral) or not 0 <= seed < 1 << 63:
            raise ValueError("seed must be an integer in 0 .. 2^63 - 1; got %r" % (seed,))
        if isinstance(mode, (list, tuple)):
            raise ValueError("sample_captions takes one style name, not a style list")
        if self.cell == ops.CELL_FACTORED:
            if mode not in STYLES:
                raise ValueError("mode name wrong: %r (expected one of %s)" % (mode, STYLES))
        else:
            mode = None
        return sample_decode(self, features, int(start_token), int(end_token), int(n), mode, float(temperature),
                             int(seed), bool(greedy))

    # ---- greedy decoding (validation path) replayed from a CUDA graph ------------------------------------
    def _forward_greedy(self, captions, lengths, features, mode):
        """``forward(teacher_forcing_ratio=0)`` under ``no_grad`` -- the reference's validation / greedy-decode path
        (stylenet/train_multitask.py:296-299): every step feeds back the arg-max of the previous step, all on the
        device, so the ~10 launches x T steps are host-bound when issued one by one.  From the second call with the
        same (lengths, shapes, mode, precision) the whole forward is replayed from a captured CUDA graph; inputs are
        copied into its static buffers, the returned logits are a copy of its static output."""
        key = (tuple(int(l) for l in lengths), mode, tuple(captions.shape),
               None if features is None else tuple(features.shape), self.precision, self.training,
               captions.device.index, self.arena().version)
        cache = self.__dict__.setdefault("_greedy_graphs", OrderedDict())
        sess = cache.get(key)
        if sess is None:
            sess = cache[key] = _Ctx()
            sess.calls, sess.graph = 0, None
            while len(cache) > 4:                      # each entry pins its logits and activations
                cache.popitem(last=False)
        cache.move_to_end(key)
        sess.calls += 1
        plan = get_plan(lengths)
        coins = self._coins(plan.T, 0.0)               # consumes the host RNG stream exactly like the reference
        if sess.graph is None and sess.calls < 2:
            c = self._run_forward(plan, captions.contiguous(), features, coins, mode, save=False)
            return self._vocab_logits(c.top.Hall, c.top.Hb)
        if sess.graph is None:
            sess.captions = captions.contiguous().clone()
            sess.features = None if features is None else features.detach().clone()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with ops.no_gc_during_capture(), torch.cuda.graph(g):
                c = self._run_forward(plan, sess.captions, sess.features, coins, mode, save=False)
                sess.out = self._vocab_logits(c.top.Hall, c.top.Hb)
            sess.graph = g
        sess.captions.copy_(captions, non_blocking=True)
        if features is not None:
            sess.features.copy_(features, non_blocking=True)
        sess.graph.replay()
        return sess.out.clone()

    # ---- public API --------------------------------------------------------------------------------
    def _greedy_eligible(self, captions, lengths, features, teacher_forcing_ratio):
        if torch.is_grad_enabled() or teacher_forcing_ratio > 0.0 or not GREEDY_GRAPH[0] or not captions.is_cuda:
            return False
        if torch.cuda.is_current_stream_capturing():
            return False
        if features is not None and features.shape[-1] != self._emb().weight.shape[1]:
            return False                      # let the regular path raise its error
        plan = get_plan(lengths)
        T_in = captions.shape[1] + (1 if features is not None else 0)
        return plan.B == captions.shape[0] and plan.T <= T_in

    def _forward_hidden(self, captions, lengths, features, teacher_forcing_ratio, mode):
        self._check_inputs(captions, features)
        if features is not None and features.shape[-1] != self._emb().weight.shape[1]:
            raise RuntimeError("features must be [B, embed_size]")
        plan = get_plan(lengths)
        if plan.B != captions.shape[0]:
            raise RuntimeError("len(lengths) != batch size")
        T_in = captions.shape[1] + (1 if features is not None else 0)
        if plan.T > T_in:
            raise RuntimeError("lengths exceed the (feature +) caption length")
        coins = self._coins(plan.T, teacher_forcing_ratio)
        captions = captions.contiguous()
        anchor = self._out().weight
        save = torch.is_grad_enabled()
        return _HiddenFn.apply(anchor, features, self, plan, captions, coins, mode, save), plan

    def forward_loss(self, captions, lengths, features=None, targets=None, teacher_forcing_ratio=1.0,
                     mode="factual", backward=True, n_global=None, grad_hook=None, early_step=None, early_embed=False,
                     token_weights=None):
        """Fused training entry point (an addition beside the kept surface, SURVEY.md section 8b):
        forward -> mean token NLL -> (optionally) backward, with log-softmax/NLL/gradient fused in one
        pass over the logits and no autograd graph.  Populates ``.grad`` like ``loss.backward()`` after
        ``zero_grad()`` would.  Returns ``(loss[1], stats)`` with stats = dict(argmax, top5hit).
        ``n_global``: token count to normalise by (data parallel: the global count).
        ``early_step(names) -> bool``: called (bf16 mode, on side stream 0, right behind dC / db_C) when the gradients
        of the vocabulary projection are final, so that the optimizer can update them under the reverse recurrence.
        ``early_embed``: in a teacher-forced bf16 step, issue the embedding backward's token grouping and gradient
        zeroing from the forward, on a side stream (the same results, off the tail of the step).
        ``token_weights``: float32 CUDA tensor [N] in packed row order (or None): the loss becomes
        sum_r w_r * NLL_r / denom and every gradient is that loss's (weights may be negative, e.g. the advantages of
        self-critical training, scst.py).  ``stats["argmax"]`` / ``"top5hit"`` and the per-row NLL do not depend on
        it; weights of 1 give the unweighted results bit for bit."""
        self._check_inputs(captions, features)
        plan = get_plan(lengths)
        if token_weights is not None:
            if (not isinstance(token_weights, torch.Tensor) or token_weights.dtype != torch.float32
                    or tuple(token_weights.shape) != (plan.N,) or token_weights.device != captions.device):
                raise ValueError("token_weights must be a float32 tensor of shape [%d] on %s" % (plan.N, captions.device))
            token_weights = token_weights.contiguous()
        coins = self._coins(plan.T, teacher_forcing_ratio)
        captions = captions.contiguous()
        dev = captions.device
        # (the gradient arena's embedding rows are zeroed early only when they hold no live gradient)
        self.__dict__["_emb_early"] = bool(early_embed and backward and self.bf16 and self._emb().weight.grad is None)
        with torch.no_grad():
            c = self._run_forward(plan, captions, features, coins, mode, save=backward)
            N = plan.N
            out = self._out()
            V = out.weight.shape[0]
            if targets is None:
                if features is None:
                    raise ValueError("forward_loss: pass `targets` when features is None (language-only "
                                     "pass: inputs captions[:, :-1], targets packed captions[:, 1:])")
                if self.bf16:
                    # gathered on the shadow stream (forked from the main stream at the start of this forward, after
                    # `captions` existed) while the recurrence runs; allocated here, written there
                    targets = torch.empty(N, dtype=captions.dtype, device=dev)
                    side = self._side(2)
                    with torch.cuda.stream(side):
                        self._default_targets(captions, plan, True, out=targets)
                        ev = torch.cuda.Event()
                        ev.record(side)
                    torch.cuda.current_stream().wait_event(ev)
                else:
                    targets = self._default_targets(captions, plan, True)
            denom = float(n_global if n_global is not None else N)
            row_loss, argmax, top5, logits, dLb = self._vocab_nll(c.top.Hall, c.top.Hb, targets, denom, backward,
                                                                  row_weight=token_weights)
            loss = torch.empty(1, dtype=torch.float32, device=dev)
            if not (backward and dLb is not None):
                ops.reduce_sum(row_loss, N, 1.0 / denom, loss, row_weight=token_weights)
            if backward:
                gbuf = self._grad_target(c.grad_names + list(self._out_names()))
                deferred = []
                gate_B = plan.B if (c.top.Hpb is not None and not (plan.B >= ops.RECUR_GEMM_MIN_BATCH[0] and self.hidden_size % 64 == 0)) else None
                dHall = self._vocab_backward(c.top.Hall, logits, gbuf, c.top.Hb, dLb, defer=deferred, gate_B=gate_B)
                if dLb is not None:
                    def loss_and_bucket():
                        # the scalar loss is bookkeeping: reduce it behind dC on side stream 0, not in front of dH
                        with torch.cuda.stream(self._side(0)):
                            ops.reduce_sum(row_loss, N, 1.0 / denom, loss, row_weight=token_weights)
                            if early_step is not None and gbuf is self.arena().gflat:
                                self._publish(list(self._out_names()), gbuf)
                                early_step(list(self._out_names()))
                    if deferred:
                        deferred.append(loss_and_bucket)
                    else:
                        loss_and_bucket()
                # (work deferred until the reverse recurrence of the top layer has been launched, see _layer_bwd)
                self.__dict__["_after_recur"] = deferred
                if grad_hook is not None and gbuf is self.arena().gflat:
                    self._run_deferred()
                    self._join()
                    grad_hook(list(self._out_names()))       # bucket 0 is final: overlap its all-reduce
                need_dfeat = features is not None and features.requires_grad
                # further buckets (W_hh / U, S / V of every layer) are handed to `early_step` by the backward itself
                self.__dict__["_bucket_hook"] = (gbuf, early_step) if (early_step is not None and gbuf is self.arena().gflat) else None
                try:
                    dfeat = self._run_backward(c, dHall, gbuf, need_dfeat)
                finally:
                    self.__dict__["_bucket_hook"] = None
                self._run_deferred()
                self._join()
                self._publish(c.grad_names + list(self._out_names()), gbuf)
                if grad_hook is not None:
                    grad_hook(c.grad_names if gbuf is self.arena().gflat else c.grad_names + list(self._out_names()))
                if dfeat is not None:
                    features.grad = dfeat if features.grad is None else features.grad + dfeat
        return loss, {"argmax": argmax, "top5hit": top5, "n_tokens": N}

    def _default_targets(self, captions, plan, has_feat, out=None):
        """Packed targets = what pack_padded_sequence(captions, lengths)[0] holds (train_multitask.py:377-379):
        one gather through a flat (b*T + t) index cached with the plan."""
        d = plan.dev(captions.device)
        key = "tgt_idx_%d_%d" % (captions.shape[1], 0 if has_feat else 1)
        idx = d.get(key)
        if idx is None:
            idx = (d["row_b"].long() * captions.shape[1] + d["row_t"].long() + (0 if has_feat else 1)).contiguous()
            d[key] = idx
        if out is not None:
            return torch.index_select(captions.reshape(-1), 0, idx, out=out)
        return captions.reshape(-1).index_select(0, idx)


V_CAST_SIDE = [os.environ.get("SN_V_CAST_SIDE", "1") == "1"]


class DecoderFactoredLSTM(_DecoderBase):
    """StyleNet FactoredLSTM decoder -- signature of stylenet/model.py:32-41."""

    cell = ops.CELL_FACTORED

    def __init__(self, embed_size, hidden_size, factored_size, vocab_size, num_layers, feature_size=2048,
                 bias=True, dropout=0.22, max_seq_length=40):
        super().__init__()
        if not bias:
            raise NotImplementedError("bias=False is not supported by the fused path")
        self.feature_size, self.hidden_size = feature_size, hidden_size
        self.factored_size, self.embed_size = factored_size, embed_size
        self.vocab_size, self.max_seq_length = vocab_size, max_seq_length
        self.num_layers = num_layers   # accepted and ignored, like the reference (model.py:37)
        self.dropout = nn.Dropout(dropout)
        self.B = nn.Embedding(vocab_size, embed_size)
        for g in GATES:
            setattr(self, "U_" + g, nn.Linear(factored_size, hidden_size, bias=bias))
            setattr(self, style_attr("factual", g), nn.Linear(factored_size, factored_size, bias=bias))
            setattr(self, "V_" + g, nn.Linear(embed_size, factored_size, bias=bias))
            setattr(self, "W_" + g, nn.Linear(hidden_size, hidden_size, bias=bias))
        for s in STYLES[1:]:
            for g in GATES:
                setattr(self, style_attr(s, g), nn.Linear(factored_size, factored_size, bias=bias))
        self.C = nn.Linear(hidden_size, vocab_size, bias=bias)
        _ref_init(self, self.B, self.C)

    # -- layout ------------------------------------------------------------------------------------
    def _arena_groups(self):
        groups = [["B.weight"]]
        for pre in ("V_", "U_", "W_"):
            groups.append([pre + g + ".weight" for g in GATES])
            groups.append([pre + g + ".bias" for g in GATES])
        for s in STYLES:
            groups.append([style_attr(s, g) + ".weight" for g in GATES])
            groups.append([style_attr(s, g) + ".bias" for g in GATES])
        groups += [["C.weight"], ["C.bias"]]
        return groups

    def _emb(self):
        return self.B

    def _emb_name(self):
        return "B.weight"

    def _out(self):
        return self.C

    def _out_names(self):
        return ("C.weight", "C.bias")

    @staticmethod
    def _lp(layer):
        """Parameter-name prefix of stack layer ``layer`` (the first layer keeps the reference names)."""
        return "" if layer == 0 else "l%d_" % layer

    def _stack(self, pre, shape, grad=False, gbuf=None, bias=False, layer=0):
        names = [self._lp(layer) + pre + g + (".bias" if bias else ".weight") for g in GATES]
        if gbuf is not None:
            return self._gview(gbuf, names, shape)
        return self.arena().block(names, shape, grad=grad)

    def _style_stack(self, mode, shape, gbuf=None, bias=False, layer=0):
        names = [self._lp(layer) + style_attr(mode, g) + (".bias" if bias else ".weight") for g in GATES]
        if gbuf is not None:
            return self._gview(gbuf, names, shape)
        return self.arena().block(names, shape)

    def _shadow_specs(self, c, mode):
        H, F = self.hidden_size, self.factored_size
        early, late = super()._shadow_specs(c, mode)
        if mode in STYLES:
            # (V's K = 300 -> 304 padded cast is the scalar kernel, 39 us under the block cap: cast at full width)
            if V_CAST_SIDE[0]:
                # V and S feed the first two GEMMs of the critical chain: full width, one event each (S must not wait for
                # U's throttled cast: that left a 7 us bubble between the V and the S stage)
                c.first_specs = [(c.w16, "V", self._stack("V_", (4 * F, c.Ein)))]
                c.second_specs = [(c.w16, "S", self._style_stack(mode, (4 * F, F)))]
                early = [(c.w16, "U", self._stack("U_", (4 * H, F)))]
            else:
                early = [(c.w16, "S", self._style_stack(mode, (4 * F, F))), (c.w16, "U", self._stack("U_", (4 * H, F)))]
        return early, late

    def _recurrent_weights(self, layer=0):
        H = self.hidden_size
        return self._stack("W_", (4 * H, H), layer=layer), self._stack("W_", (4 * H,), bias=True, layer=layer)

    def _recurrent_grads(self, gbuf, layer=0):
        H = self.hidden_size
        return (self._stack("W_", (4 * H, H), gbuf=gbuf, layer=layer),
                self._stack("W_", (4 * H,), gbuf=gbuf, bias=True, layer=layer))

    def _seq_grad_names(self, mode):
        names = ["B.weight"]
        for pre in ("V_", "U_", "W_"):
            names += [pre + g + sfx for g in GATES for sfx in (".weight", ".bias")]
        names += [style_attr(mode, g) + sfx for g in GATES for sfx in (".weight", ".bias")]
        return names

    # -- K2: factored input projection U S V ----------------------------------------------------------
    def _input_projection(self, c, X, mode, r0, n):
        """XP[r0:r0+n] = U_g(S_{mode,g}(V_g x)) for the four gates (stylenet/model.py:119-150), as one
        stacked GEMM and two 4-group batched GEMMs; biases of every stage included."""
        if mode not in STYLES:
            raise ValueError("mode name wrong: %r (expected one of %s)" % (mode, STYLES))
        H, F = self.hidden_size, self.factored_size
        Ein = X.shape[1] if X is not None else c.Ein
        dev = c.XP.device
        full = (r0 == 0 and n == c.XP.shape[0])
        if full and not self.bf16:
            c.A1 = torch.empty(n, 4 * F, dtype=torch.float32, device=dev)
            c.A2 = torch.empty(n, 4 * F, dtype=torch.float32, device=dev)
        A1, A2 = c.__dict__.get("A1"), c.__dict__.get("A2")
        L = getattr(c, "layer", 0)
        Vc, bV = self._stack("V_", (4 * F, Ein), layer=L), self._stack("V_", (4 * F,), bias=True, layer=L)
        Sc, bS = self._style_stack(mode, (4 * F, F), layer=L), self._style_stack(mode, (4 * F,), bias=True, layer=L)
        Uc, bU = self._stack("U_", (4 * H, F), layer=L), self._stack("U_", (4 * H,), bias=True, layer=L)
        if self.bf16:
            w16 = c.__dict__.setdefault("w16", {})
            if "V" not in w16:
                w16["V"] = self._shadow(Vc)
            if "S" not in w16:
                w16["S"], w16["U"] = self._shadow(Sc), self._shadow(Uc)
            Vb, Sb, Ub = w16["V"], w16["S"], w16["U"]
            Ep, Fp = Vb.stride(0), Sb.stride(0)
            if full:
                if X is not None:
                    c.Xb = torch.empty(n, Ep, dtype=torch.bfloat16, device=dev)
                c.A1 = torch.empty(n, 4 * F, dtype=torch.bfloat16, device=dev)
                c.A2 = torch.empty(n, 4 * F, dtype=torch.bfloat16, device=dev)
            if X is not None:
                ops.cast_bf16(X, n, Ein, Ein, c.Xb, Ep, Ep, src_off=r0 * Ein, dst_off=r0 * Ep)
            ev = c.__dict__.get("ev_first")
            if ev is not None:                  # the V shadow comes from the side stream
                torch.cuda.current_stream().wait_event(ev)
                c.ev_first = None
            ops.gemm_bf16(ops.OP_NT, c.Xb, Vb, n, 4 * F, Ep, Ep, Ep, Cb=c.A1, ldcb=4 * F, bias=bV, a_off=r0 * Ep,
                          cb_off=r0 * 4 * F)
            ev2 = c.__dict__.get("ev_second")
            ev = c.__dict__.get("ev_early")
            if ev2 is not None:                 # the S shadow has its own event, U's is awaited in front of the U stage
                torch.cuda.current_stream().wait_event(ev2)
                c.ev_second = None
            elif ev is not None:                # the S / U shadows come from the side stream
                torch.cuda.current_stream().wait_event(ev)
                c.ev_early = ev = None
            ops.gemm_bf16(ops.OP_NT, c.A1, Sb, n, F, F, 4 * F, Fp, Cb=c.A2, ldcb=4 * F, bias=bS, batch=4, sA=F,
                          sB=F * Fp, sCb=F, sBias=F, a_off=r0 * 4 * F, cb_off=r0 * 4 * F)
            if ev is not None:
                torch.cuda.current_stream().wait_event(ev)
                c.ev_early = None
            ops.gemm_bf16(ops.OP_NT, c.A2, Ub, n, H, F, 4 * F, Fp, C=c.XP, ldc=4 * H, bias=bU, batch=4, sA=F,
                          sB=H * Fp, sC=H, sBias=H, a_off=r0 * 4 * F, c_off=r0 * 4 * H)
            return
        ops.gemm(ops.OP_NT, X, Vc, A1, n, 4 * F, Ein, Ein, Ein, 4 * F, bias=bV, a_off=r0 * Ein,
                 c_off=r0 * 4 * F)
        ops.gemm(ops.OP_NT, A1, Sc, A2, n, F, F, 4 * F, F, 4 * F, bias=bS, batch=4, sA=F, sB=F * F, sC=F,
                 sBias=F, a_off=r0 * 4 * F, c_off=r0 * 4 * F)
        ops.gemm(ops.OP_NT, A2, Uc, c.XP, n, H, F, 4 * F, F, 4 * H, bias=bU, batch=4, sA=F, sB=H * F, sC=H,
                 sBias=H, a_off=r0 * 4 * F, c_off=r0 * 4 * H)

    def _input_projection_bwd(self, c, dZ, gbuf):
        H, F = self.hidden_size, self.factored_size
        N, Ein = dZ.shape[0], c.Ein
        dev = dZ.device
        mode = c.mode
        L = getattr(c, "layer", 0)
        Vc = self._stack("V_", (4 * F, Ein), layer=L)
        Sc = self._style_stack(mode, (4 * F, F), layer=L)
        Uc = self._stack("U_", (4 * H, F), layer=L)
        gV, gbV = (self._stack("V_", (4 * F, Ein), gbuf=gbuf, layer=L),
                   self._stack("V_", (4 * F,), gbuf=gbuf, bias=True, layer=L))
        gS, gbS = (self._style_stack(mode, (4 * F, F), gbuf=gbuf, layer=L),
                   self._style_stack(mode, (4 * F,), gbuf=gbuf, bias=True, layer=L))
        gU, gbU = (self._stack("U_", (4 * H, F), gbuf=gbuf, layer=L),
                   self._stack("U_", (4 * H,), gbuf=gbuf, bias=True, layer=L))
        if self.bf16:
            return self._input_projection_bwd_bf16(c, dZ, gV, gbV, gS, gbS, gU, gbU)
        # U stage: dU_g = dZ_g^T A2_g ; dbU = colsum(dZ) ; dA2_g = dZ_g U_g
        ops.gemm(ops.OP_TN, dZ, c.A2, gU, H, F, N, 4 * H, 4 * F, F, batch=4, sA=H, sB=F, sC=H * F)
        ops.colsum(dZ, N, 4 * H, 4 * H, gbU)
        dA2 = torch.empty(N, 4 * F, dtype=torch.float32, device=dev)
        ops.gemm(ops.OP_NN, dZ, Uc, dA2, N, F, H, 4 * H, F, 4 * F, batch=4, sA=H, sB=H * F, sC=F)
        # S stage
        ops.gemm(ops.OP_TN, dA2, c.A1, gS, F, F, N, 4 * F, 4 * F, F, batch=4, sA=F, sB=F, sC=F * F)
        ops.colsum(dA2, N, 4 * F, 4 * F, gbS)
        dA1 = torch.empty(N, 4 * F, dtype=torch.float32, device=dev)
        ops.gemm(ops.OP_NN, dA2, Sc, dA1, N, F, F, 4 * F, F, 4 * F, batch=4, sA=F, sB=F * F, sC=F)
        # V stage
        ops.gemm(ops.OP_TN, dA1, c.X, gV, 4 * F, Ein, N, 4 * F, Ein, Ein)
        ops.colsum(dA1, N, 4 * F, 4 * F, gbV)
        dX = torch.empty(N, Ein, dtype=torch.float32, device=dev)
        ops.gemm(ops.OP_NN, dA1, Vc, dX, N, Ein, 4 * F, 4 * F, Ein, Ein)
        return dX

    def _input_projection_bwd_bf16(self, c, dZ, gV, gbV, gS, gbS, gU, gbU):
        """Backward of the factored chain with every GEMM on tcgen05 (bf16 operands, fp32 results)."""
        H, F = self.hidden_size, self.factored_size
        N, Ein = dZ.shape[0], c.Ein
        dev = dZ.device
        Vb, Sb, Ub = c.w16["V"], c.w16["S"], c.w16["U"]
        Ep, Fp = Vb.stride(0), Sb.stride(0)
        dZb = c.dZb
        f32 = dict(dtype=torch.float32, device=dev)
        b16 = dict(dtype=torch.bfloat16, device=dev)
        main = torch.cuda.current_stream()
        sa, sb = self._side(0), self._side(1)
        # critical chain (main stream): dZ -> dA2 -> dA1 -> dX ; the weight / bias gradients trail on TWO side streams
        # (U on stream 0 behind dW_hh, S and V on stream 1) so that Adam does not wait for a serial tail of GEMMs
        dA2, dA2b = torch.empty(N, 4 * F, **f32), torch.empty(N, 4 * F, **b16)
        dA1, dA1b = torch.empty(N, 4 * F, **f32), torch.empty(N, 4 * F, **b16)
        dX = torch.empty(N, Ein, **f32)
        L = getattr(c, "layer", 0)
        lp = self._lp(L)
        sa.wait_stream(main)
        with torch.cuda.stream(sa):
            ops.gemm_bf16(ops.OP_TN, dZb, c.A2, H, F, N, 4 * H, 4 * F, C=gU, ldc=F, batch=4, sA=H, sB=F, sC=H * F)
            wide = bool(ops.TAIL_SCHEDULE[0])
            if getattr(c, "colsum_dZ", None) is not None:
                gbU.copy_(c.colsum_dZ)          # written by _layer_bwd on this stream: the same sum, bit for bit
            else:
                ops.colsum(dZ, N, 4 * H, 4 * H, gbU, wide=wide)
            # stream 0 also carried dW_hh / db_hh of this layer (_layer_bwd): bucket {W_hh, U} is final here
            self._bucket_final([lp + pre + g + sfx for pre in ("W_", "U_") for g in GATES for sfx in (".weight", ".bias")])
        ops.gemm_bf16(ops.OP_NN, dZb, Ub, N, F, H, 4 * H, Fp, C=dA2, ldc=4 * F, Cb=dA2b, ldcb=4 * F, batch=4, sA=H,
                      sB=H * Fp, sC=F, sCb=F)
        sb.wait_stream(main)
        with torch.cuda.stream(sb):
            ops.gemm_bf16(ops.OP_TN, dA2b, c.A1, F, F, N, 4 * F, 4 * F, C=gS, ldc=F, batch=4, sA=F, sB=F, sC=F * F)
            ops.colsum(dA2, N, 4 * F, 4 * F, gbS, wide=wide)
        ops.gemm_bf16(ops.OP_NN, dA2b, Sb, N, F, F, 4 * F, Fp, C=dA1, ldc=4 * F, Cb=dA1b, ldcb=4 * F, batch=4, sA=F,
                      sB=F * Fp, sC=F, sCb=F)
        sb.wait_stream(main)
        with torch.cuda.stream(sb):
            ops.gemm_bf16(ops.OP_TN, dA1b, c.Xb, 4 * F, Ein, N, 4 * F, Ep, C=gV, ldc=Ein)
            ops.colsum(dA1, N, 4 * F, 4 * F, gbV, wide=wide)
            self._bucket_final([lp + style_attr(c.mode, g) + sfx for g in GATES for sfx in (".weight", ".bias")] +
                               [lp + "V_" + g + sfx for g in GATES for sfx in (".weight", ".bias")])
        ops.gemm_bf16(ops.OP_NN, dA1b, Vb, N, Ein, 4 * F, 4 * F, Ep, C=dX, ldc=Ein)
        return dX

    def _collapse_chain(self, ctx, mode, layer=0):
        """Inference only, once per decode call: the factored chain U_g S_g V_g of ``mode`` as ONE matrix per gate,
        Wc_g = U_g (S_g V_g) [H, Ein], bc_g = U_g (S_g bV_g + bS_g) + bU_g (stylenet/model.py:119-150 is linear in x
        between the embedding and the gate sums).  ``_small_step`` then runs a decode step as a single kernel.  The
        result buffers live in ``ctx`` (fixed addresses: the steps are CUDA-graph captured) and are refreshed in place."""
        if mode not in STYLES:
            raise ValueError("mode name wrong: %r (expected one of %s)" % (mode, STYLES))
        H, F = self.hidden_size, self.factored_size
        Ein = self._chain_in(layer)
        col = ctx.__dict__.setdefault("collapsed", {})
        ent = col.get(layer)
        key = (mode, self.arena().content_key())
        if ent is not None and ent.get("key") == key:
            return ent                         # same weights as at the last call (evaluation loops): nothing to refresh
        if ent is None or ent["Wc"].shape != (4 * H, Ein):
            f32 = dict(dtype=torch.float32, device=self.B.weight.device)
            ent = col[layer] = {"Wc": torch.empty(4 * H, Ein, **f32), "bc": torch.empty(4 * H, **f32),
                                "SV": torch.empty(4 * F, Ein, **f32), "t": torch.empty(4 * F, **f32)}
        self._collapse_into(mode, layer, ent["Wc"], ent["bc"], ent["SV"], ent["t"])
        ent["mode"], ent["key"] = mode, key
        return ent

    def _chain_in(self, layer):
        """Input width of layer ``layer``'s factored chain (E for the first layer, H above it)."""
        return self.arena().named[self._lp(layer) + "V_" + GATES[0] + ".weight"].shape[1]

    def _collapse_into(self, mode, layer, Wc, bc, SV, t):
        """The GEMMs of ``_collapse_chain``: Wc [4H, Ein], bc [4H] of ``mode``; SV [4F, Ein] and t [4F] are scratch."""
        H, F = self.hidden_size, self.factored_size
        Ein = Wc.shape[1]
        Vc, bV = self._stack("V_", (4 * F, Ein), layer=layer), self._stack("V_", (4 * F,), bias=True, layer=layer)
        Sc, bS = self._style_stack(mode, (4 * F, F), layer=layer), self._style_stack(mode, (4 * F,), bias=True, layer=layer)
        Uc, bU = self._stack("U_", (4 * H, F), layer=layer), self._stack("U_", (4 * H,), bias=True, layer=layer)
        with torch.no_grad():
            ops.gemm(ops.OP_NN, Sc, Vc, SV, F, Ein, F, F, Ein, Ein, batch=4, sA=F * F, sB=F * Ein, sC=F * Ein)
            ops.gemm(ops.OP_NN, Uc, SV, Wc, H, Ein, F, F, Ein, Ein, batch=4, sA=H * F, sB=F * Ein, sC=H * Ein)
            ops.gemm(ops.OP_NN, Sc, bV, t, F, 1, F, F, 1, 1, batch=4, sA=F * F, sB=F, sC=F)
            t.add_(bS)
            ops.gemm(ops.OP_NN, Uc, t, bc, H, 1, F, F, 1, 1, batch=4, sA=H * F, sB=F, sC=H)
            bc.add_(bU)

    def _collapse_styles(self, ctx, styles, layer=0):
        """``_collapse_chain`` for several styles of one decode call (``sample_batch`` with a per-image style list):
        Wc [G, 4H, Ein] / bc [G, 4H], entry g the collapsed chain of ``styles[g]`` -- the same GEMMs, so bit for bit
        the single-style matrices.  Fixed addresses (graph-captured steps read them), refreshed in place whenever the
        weights have changed since the last call."""
        for mode in styles:
            if mode not in STYLES:
                raise ValueError("mode name wrong: %r (expected one of %s)" % (mode, STYLES))
        H, F = self.hidden_size, self.factored_size
        Ein, G = self._chain_in(layer), len(styles)
        col = ctx.__dict__.setdefault("collapsed_groups", {})
        ent = col.get(layer)
        key = (tuple(styles), self.arena().content_key())
        if ent is not None and ent.get("key") == key:
            return ent
        if ent is None or ent["Wc"].shape != (G, 4 * H, Ein):
            f32 = dict(dtype=torch.float32, device=self.B.weight.device)
            ent = col[layer] = {"Wc": torch.empty(G, 4 * H, Ein, **f32), "bc": torch.empty(G, 4 * H, **f32),
                                "SV": torch.empty(4 * F, Ein, **f32), "t": torch.empty(4 * F, **f32)}
        for g, mode in enumerate(styles):
            self._collapse_into(mode, layer, ent["Wc"][g], ent["bc"][g], ent["SV"], ent["t"])
        ent["key"] = key
        return ent

    def _small_step(self, ctx, X, mode, R, h_prev, c_prev, src_row, h_out, c_out, layer=0, x_rows=None):
        """forward_step for R <= ops.SKINNY_MAX_ROWS rows on the matrix-vector kernels (sn_decode.cu): V and S stages as
        skinny linears, the U stage + W_hh + gates + cell update fused (stylenet/model.py:119-153); with the chain
        collapsed for this call (``_collapse_chain``) the whole step is the fused kernel alone."""
        if mode not in STYLES:
            raise ValueError("mode name wrong: %r (expected one of %s)" % (mode, STYLES))
        H, F = self.hidden_size, self.factored_size
        Ein = X.shape[1]
        ent = ctx.__dict__.get("collapsed", {}).get(layer)
        if ent is not None and ent.get("mode") == mode and ent["Wc"].shape[1] == Ein:
            Whh, bhh = self._recurrent_weights(layer)
            ops.decode_cell(self.cell, H, R, ent["Wc"], Ein, X, 0, ent["bc"], Whh, bhh, h_prev, c_prev, src_row, h_out,
                            c_out, x_rows=x_rows)
            return
        a1, a2 = ctx.__dict__.get("sk_a1"), ctx.__dict__.get("sk_a2")
        if a1 is None or a1.shape[0] < R:
            a1 = ctx.sk_a1 = torch.empty(max(R, ops.SKINNY_MAX_ROWS), 4 * F, dtype=torch.float32, device=X.device)
            a2 = ctx.sk_a2 = torch.empty_like(a1)
        ops.skinny_linear(self._stack("V_", (4 * F, Ein), layer=layer), X, a1, R,
                          bias=self._stack("V_", (4 * F,), bias=True, layer=layer), x_rows=x_rows)
        Sc = self._style_stack(mode, (4 * F, F), layer=layer)
        bS = self._style_stack(mode, (4 * F,), bias=True, layer=layer)
        if F % 32 == 0:
            ops.skinny_linear(Sc, a1, a2, R, bias=bS, group_n=F, group_x=F)
        else:                      # odd factored sizes: one call per gate block
            for g in range(4):
                ops.skinny_linear(Sc[g * F:(g + 1) * F], a1[:, g * F:(g + 1) * F], a2[:, g * F:(g + 1) * F], R,
                                  bias=bS[g * F:(g + 1) * F])
        Whh, bhh = self._recurrent_weights(layer)
        ops.decode_cell(self.cell, H, R, self._stack("U_", (4 * H, F), layer=layer), F, a2, F,
                        self._stack("U_", (4 * H,), bias=True, layer=layer), Whh, bhh, h_prev, c_prev, src_row, h_out, c_out)

    # -- reference surface ---------------------------------------------------------------------------
    def forward(self, captions, lengths, features=None, teacher_forcing_ratio=0.8, mode="factual"):
        """Same call and return as stylenet/model.py:157-196: packed logits [sum(lengths), V]."""
        if mode not in STYLES:
            raise ValueError("mode name wrong: %r (expected one of %s)" % (mode, STYLES))
        if self._greedy_eligible(captions, lengths, features, teacher_forcing_ratio):
            return self._forward_greedy(captions, lengths, features, mode)
        hall, _ = self._forward_hidden(captions, lengths, features, teacher_forcing_ratio, mode)
        return _LogitsFn.apply(hall, self.C.weight, self)

    def forward_step(self, embedded, states, mode):
        """One cell step (stylenet/model.py:115-155) on the kernels: K2 projection + one K3 step."""
        from .decode import single_step
        return single_step(self, embedded, states, mode)

    def sample(self, features, start_token, end_token, k=5, factual_limit=-1, mode="factual",
               feed_image=False):
        """Beam search with the reference's semantics (stylenet/model.py:198-294; ``feed_image=True`` is
        the app/backend/model.py:386-487 variant).  Returns LongTensor [1, L]."""
        from .decode import beam_sample, require_one_style
        require_one_style(mode)
        return beam_sample(self, features, start_token, end_token, k, mode, feed_image)[0]

    def sample_batch(self, features, start_token, end_token, k=5, mode="factual", feed_image=False):
        """``sample()`` for every row of ``features [n_img, E]`` in one batched beam search (an addition beside the kept
        surface, SURVEY.md section 8b; replaces the per-image loop of stylenet/evaluator.py:74-81).  Returns a list of
        LongTensor [1, L_i], element i identical to ``sample(features[i:i+1], ...)``.
        ``mode`` may also be a list / tuple of n_img style names: image i is captioned in style ``mode[i]`` (element i
        identical to ``sample_batch(features[i:i+1], ..., mode=mode[i])[0]``), all styles in one beam search -- e.g.
        ``sample_batch(feature.expand(4, -1), start, end, k, mode=list(STYLES))`` captions one image in every style."""
        from .decode import beam_sample
        return beam_sample(self, features, start_token, end_token, k, mode, feed_image)


class DecoderRNN(_DecoderBase):
    """NIC LSTM decoder -- signature of nic/model.py:31-38."""

    cell = ops.CELL_LSTM

    def __init__(self, embed_size, hidden_size, vocab_size, num_layers, feature_size=2048, dropout=0.22,
                 max_seq_length=40):
        super().__init__()
        self.feature_size, self.hidden_size, self.embed_size = feature_size, hidden_size, embed_size
        self.vocab_size, self.max_seq_length = vocab_size, max_seq_length
        self.num_layers = num_layers
        self.dropout = nn.Dropout(dropout)
        self.embed = nn.Embedding(vocab_size, embed_size)
        self.lstm = nn.LSTMCell(embed_size, hidden_size, bias=True)
        self.linear = nn.Linear(hidden_size, vocab_size)
        _ref_init(self, self.embed, self.linear)

    def _arena_groups(self):
        return [["embed.weight"], ["lstm.weight_ih"], ["lstm.weight_hh"], ["lstm.bias_ih"], ["lstm.bias_hh"],
                ["linear.weight"], ["linear.bias"]]

    def _emb(self):
        return self.embed

    def _emb_name(self):
        return "embed.weight"

    def _out(self):
        return self.linear

    def _out_names(self):
        return ("linear.weight", "linear.bias")

    def _recurrent_weights(self, layer=0):
        self.arena()
        return self.lstm.weight_hh, self.lstm.bias_hh

    def _recurrent_grads(self, gbuf, layer=0):
        H = self.hidden_size
        return self._gview(gbuf, ["lstm.weight_hh"], (4 * H, H)), self._gview(gbuf, ["lstm.bias_hh"], (4 * H,))

    def _seq_grad_names(self, mode):
        return ["embed.weight", "lstm.weight_ih", "lstm.weight_hh", "lstm.bias_ih", "lstm.bias_hh"]

    def _input_projection(self, c, X, mode, r0, n):
        """XP = x W_ih^T + b_ih (the first addmm of nn.LSTMCell, nic/model.py:77)."""
        H = self.hidden_size
        Ein = X.shape[1] if X is not None else c.Ein
        if self.bf16:
            w16 = c.__dict__.setdefault("w16", {})
            if "Wih" not in w16:
                w16["Wih"] = self._shadow(self.lstm.weight_ih)
            Wb = w16["Wih"]
            Ep = Wb.stride(0)
            if X is not None:
                if r0 == 0 and n == X.shape[0]:
                    c.Xb = torch.empty(n, Ep, dtype=torch.bfloat16, device=X.device)
                ops.cast_bf16(X, n, Ein, Ein, c.Xb, Ep, Ep, src_off=r0 * Ein, dst_off=r0 * Ep)
            ops.gemm_bf16(ops.OP_NT, c.Xb, Wb, n, 4 * H, Ep, Ep, Ep, C=c.XP, ldc=4 * H, bias=self.lstm.bias_ih,
                          a_off=r0 * Ep, c_off=r0 * 4 * H)
            return
        ops.gemm(ops.OP_NT, X, self.lstm.weight_ih, c.XP, n, 4 * H, Ein, Ein, Ein, 4 * H,
                 bias=self.lstm.bias_ih, a_off=r0 * Ein, c_off=r0 * 4 * H)

    def _input_projection_bwd(self, c, dZ, gbuf):
        H = self.hidden_size
        N, Ein = dZ.shape[0], c.Ein
        gW = self._gview(gbuf, ["lstm.weight_ih"], (4 * H, Ein))
        gb = self._gview(gbuf, ["lstm.bias_ih"], (4 * H,))
        dX = torch.empty(N, Ein, dtype=torch.float32, device=dZ.device)
        if self.bf16:
            Wb = c.w16["Wih"]
            Ep = Wb.stride(0)
            ops.gemm_bf16(ops.OP_TN, c.dZb, c.Xb, 4 * H, Ein, N, 4 * H, Ep, C=gW, ldc=Ein)
            ops.colsum(dZ, N, 4 * H, 4 * H, gb)
            ops.gemm_bf16(ops.OP_NN, c.dZb, Wb, N, Ein, 4 * H, 4 * H, Ep, C=dX, ldc=Ein)
            return dX
        ops.gemm(ops.OP_TN, dZ, c.X, gW, 4 * H, Ein, N, 4 * H, Ein, Ein)
        ops.colsum(dZ, N, 4 * H, 4 * H, gb)
        ops.gemm(ops.OP_NN, dZ, self.lstm.weight_ih, dX, N, Ein, 4 * H, 4 * H, Ein, Ein)
        return dX

    def _small_step(self, ctx, X, mode, R, h_prev, c_prev, src_row, h_out, c_out):
        """nn.LSTMCell step (nic/model.py:74-79) for R <= ops.SKINNY_MAX_ROWS rows: one fused matrix-vector kernel."""
        H = self.hidden_size
        self.arena()
        ops.decode_cell(self.cell, H, R, self.lstm.weight_ih, X.shape[1], X, 0, self.lstm.bias_ih, self.lstm.weight_hh,
                        self.lstm.bias_hh, h_prev, c_prev, src_row, h_out, c_out)

    def forward(self, captions, lengths, features, teacher_forcing_ratio=0.8):
        """Same call and return as nic/model.py:81-115."""
        if self._greedy_eligible(captions, lengths, features, teacher_forcing_ratio):
            return self._forward_greedy(captions, lengths, features, None)
        hall, _ = self._forward_hidden(captions, lengths, features, teacher_forcing_ratio, None)
        return _LogitsFn.apply(hall, self.linear.weight, self)

    def forward_step(self, embedded, states):
        from .decode import single_step
        return single_step(self, embedded, states, None)

    def sample(self, features, start_token, end_token, k=5, feed_image=False):
        """Beam search, nic/model.py:117-207 (``feed_image=True``: app/backend variant)."""
        from .decode import beam_sample
        return beam_sample(self, features, start_token, end_token, k, None, feed_image)[0]

    def sample_batch(self, features, start_token, end_token, k=5, feed_image=False):
        """Batched ``sample()``: one beam search over every row of ``features [n_img, E]`` (see DecoderFactoredLSTM)."""
        from .decode import beam_sample
        return beam_sample(self, features, start_token, end_token, k, None, feed_image)
