"""Soft-attention decoders: DecoderFactoredLSTMAtt (stylenet/model_att.py:73-426) and DecoderRNNAtt
(nic/model_att.py:72-306) on the sm_100a kernels.

What is time-parallel is hoisted out of the step loop (identical results, SURVEY.md Appendix B):
  * att1 = encoder_att(features) -- the reference recomputes it every step (model_att.py:59)
  * the embedding columns of V (resp. W_ih): the chain is linear, so V x = V_emb emb + V_ctx ctx
  * every weight gradient (one GEMM over all packed rows after the reverse-time loop)
Per step only what depends on h_{t-1} runs: decoder_att / f_beta GEMMs, the fused attention kernel (K4),
the context columns of the input projection, and one recurrence step (K3).
"""
import torch
import torch.nn as nn

from . import ops
from .decoders import GATES, STYLES, _Ctx, _DecoderBase, _ref_init, style_attr
from .packing import get_plan


def att_attr(style):
    return "attention" if style == "factual" else "attention_" + style


class Attention(nn.Module):
    """Parameter container with the reference's names (model_att.py:32-49); the arithmetic of its
    forward (model_att.py:51-70) runs in sn_att_step_fwd."""

    def __init__(self, encoder_dim, decoder_dim, attention_dim):
        super().__init__()
        self.encoder_att = nn.Linear(encoder_dim, attention_dim)
        self.decoder_att = nn.Linear(decoder_dim, attention_dim)
        self.full_att = nn.Linear(attention_dim, 1)

    def forward(self, encoder_out, decoder_hidden):
        """(attention_weighted_encoding [b,D], alpha [b,P]) for one step, on the kernels."""
        b, P, D = encoder_out.shape
        A = self.encoder_att.weight.shape[0]
        dev = encoder_out.device
        with torch.no_grad():
            feat = encoder_out.detach().float().contiguous()
            att1 = ops.linear_nt(feat.view(b * P, D), self.encoder_att.weight, self.encoder_att.bias)
            att2 = ops.linear_nt(decoder_hidden.detach().float().contiguous(), self.decoder_att.weight,
                                 self.decoder_att.bias)
            alpha = torch.empty(b, P, dtype=torch.float32, device=dev)
            ctx = torch.empty(b, D, dtype=torch.float32, device=dev)
            big = torch.full((b, D), 1e4, dtype=torch.float32, device=dev)   # sigmoid(1e4) == 1: ungated
            ops.att_step_fwd(att1, att2, feat, self.full_att.weight.view(-1), float(self.full_att.bias.item()),
                             big, b, P, A, D, alpha, P, ctx, D)
        return ctx, alpha


class _HiddenAttFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, features, dec, plan, captions, coins, mode, save):
        c = dec._run_forward_att(plan, captions, features, coins, mode, save)
        ctx.dec, ctx.c = dec, c
        ctx.need_dfeat = features.requires_grad
        return c.Hall, c.alphas

    @staticmethod
    def backward(ctx, dHall, dAlphas):
        dec, c = ctx.dec, ctx.c
        gbuf = dec._grad_target(c.grad_names)
        dfeat = dec._run_backward_att(c, dHall.contiguous(), dAlphas, gbuf, ctx.need_dfeat)
        dec._publish(c.grad_names, gbuf)
        return None, dfeat, None, None, None, None, None, None


class _AttBase(_DecoderBase):
    """Host logic shared by the two attention decoders."""

    def _att_module(self, mode):
        raise NotImplementedError

    def _att_prefix(self, mode):
        raise NotImplementedError

    def init_hidden_state(self, feature):
        """(h0, c0) from the mean feature (model_att.py:185-194) on the kernels."""
        with torch.no_grad():
            f = feature.detach().float().contiguous()
            B, P, D = f.shape
            mean = torch.empty(B, D, dtype=torch.float32, device=f.device)
            ops.mean_pixels(f, B, P, D, mean)
            h = ops.linear_nt(mean, self.init_h.weight, self.init_h.bias)
            c = ops.linear_nt(mean, self.init_c.weight, self.init_c.bias)
        return h, c

    # ---- forward -----------------------------------------------------------------------------------
    def _tc_ok(self):
        """bf16 mode needs TMA-legal operand shapes (every K and group offset a multiple of 8 elements)."""
        dims = [self.hidden_size, self.attention_size, self.feature_size]
        if hasattr(self, "factored_size"):
            dims.append(self.factored_size)
        return self.bf16 and self.hidden_size % 32 == 0 and all(x % 8 == 0 for x in dims)

    def _lin(self, c, x, xb, w, wkey, bias, out, n, r0_out=0, x_off_rows=0):
        """out[r0_out:r0_out+n] = x W^T + b for a small per-step Linear; tcgen05 in bf16 mode."""
        N_out, K = w.shape
        if c.tc:
            wb = c.w16[wkey]
            ops.gemm_bf16(ops.OP_NT, xb, wb, n, N_out, K, xb.stride(0), wb.stride(0), C=out, ldc=N_out, bias=bias,
                          a_off=x_off_rows * xb.stride(0), c_off=r0_out * N_out)
        else:
            ops.gemm(ops.OP_NT, x, w, out, n, N_out, K, K, K, N_out, bias=bias, a_off=x_off_rows * K,
                     c_off=r0_out * N_out)

    def _run_forward_att(self, plan, captions, features, coins, mode, save):
        a = self.arena()
        dev = captions.device
        d = plan.dev(dev)
        H, N, B, T = self.hidden_size, plan.N, plan.B, plan.T
        emb = self._emb()
        E = emb.weight.shape[1]
        D, A = self.feature_size, self.attention_size
        feats = features.detach()
        if feats.dtype != torch.float32:
            feats = feats.float()
        feats = feats.reshape(B, -1, D).contiguous()
        P = feats.shape[1]
        # produced by the fused encoder tail (encoders.EncoderCNNAtt) in the same pass that wrote `features`
        pre_mean = getattr(features, "sn_mean", None)
        pre_b16 = getattr(features, "sn_bf16", None)
        att = self._att_module(mode)
        c = _Ctx()
        c.plan, c.mode, c.captions, c.has_feat = plan, mode, captions, False
        c.feats, c.P, c.Ein = feats, P, E
        c.tc = self._tc_ok()
        c.w16 = {}
        c.p_drop = float(self.dropout.p) if self.training else 0.0
        c.seed, c.seed_dev = self._next_seed(dev, c.p_drop)
        f32 = dict(dtype=torch.float32, device=dev)
        b16 = dict(dtype=torch.bfloat16, device=dev)
        Whh, bhh = self._recurrent_weights()
        # hoisted, time-invariant pieces
        if pre_mean is not None and tuple(pre_mean.shape) == (B, D) and pre_mean.device == dev:
            c.mean = pre_mean
        else:
            c.mean = torch.empty(B, D, **f32)
            ops.mean_pixels(feats, B, P, D, c.mean)
        h0 = torch.empty(B, H, **f32)
        c.c0 = torch.empty(B, H, **f32)
        c.att1 = torch.empty(B * P, A, **f32)
        if c.tc:
            for key, w in (("init_h", self.init_h.weight), ("init_c", self.init_c.weight), ("Wd", att.decoder_att.weight),
                           ("We", att.encoder_att.weight), ("Wbeta", self.f_beta.weight), ("Whh", Whh)):
                c.w16[key] = ops.to_bf16_padded(w)
            c.meanb = ops.to_bf16_padded(c.mean)
            if pre_b16 is not None and pre_b16.numel() == B * P * D and pre_b16.device == dev:
                c.featsb = pre_b16.view(B * P, D)
            else:
                c.featsb = ops.to_bf16_padded(feats.view(B * P, D))
        else:
            c.meanb = c.featsb = None
        self._lin(c, c.mean, c.meanb, self.init_h.weight, "init_h", self.init_h.bias, h0, B)
        self._lin(c, c.mean, c.meanb, self.init_c.weight, "init_c", self.init_c.bias, c.c0, B)
        # att1 (and att2 below) feed relu(att1 + att2): their sum decides a 0/1 mask, so an operand rounded to bf16 flips
        # the mask wherever |att1 + att2| is below the rounding error and the attention net's gradients pick up a full
        # w_f * dE term per flip (2.6e-2 at configs[2] dimensions, over the 2e-2 budget).  Both stay exact fp32
        # contractions in bf16 mode; only GEMMs whose result is used linearly run on bf16 operands.
        ops.gemm(ops.OP_NT, feats.view(B * P, D), att.encoder_att.weight, c.att1, B * P, A, D, D, D, A,
                 bias=att.encoder_att.bias)
        all_tf = all(coins)
        c.tok_override = None if all_tf else torch.full((N,), -1, dtype=torch.int32, device=dev)
        if c.tc:
            c.X = None
            c.Xb = torch.empty(N, (E + 7) // 8 * 8, **b16)
        else:
            c.X = torch.empty(N, E, **f32)
            c.Xb = None
        ops.gather_pack_fwd(captions, emb.weight, None, False, d["row_b"], d["row_t"], None, N, c.X, c.p_drop, c.seed,
                            seed_dev=c.seed_dev, Xb=c.Xb)
        c.XP = torch.empty(N, 4 * H, **f32)
        self._proj_prepare(c)
        self._proj_embed_part(c, 0, N)
        c.CTX = torch.empty(N, D, **f32)
        c.CTXb = torch.empty(N, D, **b16) if c.tc else None
        c.att2 = torch.empty(N, A, **f32)
        c.gate_pre = torch.empty(N, D, **f32)
        Tmax = max(plan.lengths)
        c.alphas = torch.zeros(B, Tmax, P, **f32)
        c.Hall = torch.empty(N, H, **f32)
        c.Call = torch.empty(N, H, **f32) if save else None
        c.gates = torch.empty(N, 4 * H, **f32) if save else None
        if c.tc:
            c.Hprev = None
            c.Hb = torch.empty(N, H, **b16)
            c.Hpb = torch.empty(N, H, **b16)
            h0b = ops.to_bf16_padded(h0)
        else:
            c.Hprev = torch.empty(N, H, **f32)
            c.Hb = c.Hpb = None
        c_state = c.c0.clone()
        wfull = att.full_att.weight.view(-1)
        out = self._out()
        V = out.weight.shape[0]
        pred = captions[:, 0].to(torch.int32).contiguous()
        am = torch.empty(B, dtype=torch.int64, device=dev)
        # the scalar full_att bias shifts every score of a row equally and cancels in the softmax
        # (model_att.py:63-65): it is passed as 0 to avoid a device->host read on the hot path.
        for t in range(T):
            n, r0 = plan.bs[t], plan.off[t]
            rp = plan.off[t - 1] if t > 0 else 0
            hprev = h0 if t == 0 else c.Hall[rp:rp + n]
            if c.tc:
                hprev_b, hoff = (h0b, 0) if t == 0 else (c.Hb, rp)
            else:
                hprev_b, hoff = None, 0
            if not coins[t]:
                if t > 0:
                    bp = plan.bs[t - 1]
                    lg = torch.empty(bp, V, **f32)
                    ops.gemm(ops.OP_NT, c.Hall, out.weight, lg, bp, V, H, H, H, V, bias=out.bias, a_off=rp * H)
                    ops.softmax_nll(lg, bp, V, argmax=am)
                    pred = am[:bp].to(torch.int32)
                c.tok_override[r0:r0 + n] = pred[:n]
                ops.gather_pack_fwd(captions, emb.weight, None, False, d["row_b"], d["row_t"], c.tok_override, n,
                                    c.X, c.p_drop, c.seed, row_off=r0, seed_dev=c.seed_dev, Xb=c.Xb)
                self._proj_embed_part(c, r0, n)
            ops.gemm(ops.OP_NT, hprev, att.decoder_att.weight, c.att2, n, A, H, H, H, A, bias=att.decoder_att.bias,
                     c_off=r0 * A)
            self._lin(c, hprev, hprev_b, self.f_beta.weight, "Wbeta", self.f_beta.bias, c.gate_pre, n, r0_out=r0,
                      x_off_rows=hoff)
            ops.att_step_fwd(c.att1, c.att2[r0:], feats, wfull, 0.0, c.gate_pre[r0:], n, P, A, D,
                             c.alphas[:, t], Tmax * P, c.CTX[r0:], D, feat_b16=c.featsb)
            if c.tc:
                ops.cast_bf16(c.CTX, n, D, D, c.CTXb, D, D, src_off=r0 * D, dst_off=r0 * D)
            self._proj_step(c, r0, n)
            if c.tc:
                ops.recur_fwd_bf16(self.cell, H, B, d["bs"], d["off"], t, t + 1, c.XP, c.w16["Whh"], bhh, hprev, c.Hall,
                                   c.Hb, c.Hpb, c.Call, c.gates, c_state)
            else:
                ops.recur_fwd(self.cell, H, B, d["bs"], d["off"], t, t + 1, c.XP, Whh, bhh, hprev, c.Hall, c.Call,
                              c.Hprev, c.gates, c_state)
        c.grad_names = self._seq_grad_names(mode)
        return c

    # ---- backward ----------------------------------------------------------------------------------
    def _tn(self, c, dY, dYb, Xf, Xb, out, M, Nn, K, lda, ldb, ldc, c_off=0):
        """out[M,Nn] = dY^T X over K packed rows (a time-batched weight gradient)."""
        if c.tc:
            ops.gemm_bf16(ops.OP_TN, dYb, Xb, M, Nn, K, dYb.stride(0), Xb.stride(0), C=out, ldc=ldc, c_off=c_off)
        else:
            ops.gemm(ops.OP_TN, dY, Xf, out, M, Nn, K, lda, ldb, ldc, c_off=c_off)

    def _run_backward_att(self, c, dHall, dAlphas, gbuf, need_dfeat):
        a = self.arena()
        plan = c.plan
        dev = dHall.device
        d = plan.dev(dev)
        H, N, B, T = self.hidden_size, plan.N, plan.B, plan.T
        D, A, P = self.feature_size, self.attention_size, c.P
        emb = self._emb()
        E = emb.weight.shape[1]
        att = self._att_module(c.mode)
        pre = self._att_prefix(c.mode)
        f32 = dict(dtype=torch.float32, device=dev)
        b16 = dict(dtype=torch.bfloat16, device=dev)
        Whh, _ = self._recurrent_weights()
        wfull = att.full_att.weight.view(-1)
        dZ = torch.empty(N, 4 * H, **f32)
        c.dZb = torch.empty(N, 4 * H, **b16) if c.tc else None
        dh = torch.zeros(B, H, **f32)
        dc = torch.zeros(B, H, **f32)
        c.dCTX = torch.empty(N, D, **f32)
        datt2 = torch.empty(N, A, **f32)
        dgate = torch.empty(N, D, **f32)
        datt2b = torch.empty(N, A, **b16) if c.tc else None
        dgateb = torch.empty(N, D, **b16) if c.tc else None
        datt1 = torch.zeros(B * P, A, **f32)
        gwf = self._gview(gbuf, [pre + "full_att.weight"], (A,))
        gwf.zero_()
        self._gview(gbuf, [pre + "full_att.bias"], (1,)).zero_()   # exactly zero (softmax shift invariance)
        dfeat = torch.zeros(B, P, D, **f32) if need_dfeat else None
        Tmax = c.alphas.shape[1]
        dAl = None
        if dAlphas is not None:
            dAl = dAlphas.contiguous()
        self._proj_bwd_begin(c, N)
        for t in range(T - 1, -1, -1):
            n, r0 = plan.bs[t], plan.off[t]
            if c.tc:
                ops.recur_bwd_bf16(self.cell, H, B, d["bs"], d["off"], t, t + 1, c.w16["Whh"], c.c0, c.Call, c.gates,
                                   dHall, dZ, c.dZb, dh, dc)
            else:
                ops.recur_bwd(self.cell, H, B, d["bs"], d["off"], t, t + 1, Whh, c.c0, c.Call, c.gates, dHall, dZ, dh, dc)
            self._proj_step_bwd(c, dZ, r0, n)        # -> c.dCTX rows
            ops.att_step_bwd(c.att1, c.att2[r0:], c.feats, wfull, 0.0, c.gate_pre[r0:], c.alphas[:, t], Tmax * P,
                             c.dCTX[r0:], D, dAl[:, t] if dAl is not None else None, Tmax * P, n, P, A, D,
                             datt2[r0:], dgate[r0:], datt1, gwf, dfeat, feat_b16=c.featsb)
            # into h_{t-1}: through decoder_att and f_beta
            if c.tc:
                ops.cast_bf16(datt2, n, A, A, datt2b, A, A, src_off=r0 * A, dst_off=r0 * A)
                ops.cast_bf16(dgate, n, D, D, dgateb, D, D, src_off=r0 * D, dst_off=r0 * D)
                ops.gemm_bf16(ops.OP_NN, datt2b, c.w16["Wd"], n, H, A, A, H, C=dh, ldc=H, beta=1.0, a_off=r0 * A)
                ops.gemm_bf16(ops.OP_NN, dgateb, c.w16["Wbeta"], n, H, D, D, H, C=dh, ldc=H, beta=1.0, a_off=r0 * D)
            else:
                ops.gemm(ops.OP_NN, datt2, att.decoder_att.weight, dh, n, H, A, A, H, H, beta=1.0, a_off=r0 * A)
                ops.gemm(ops.OP_NN, dgate, self.f_beta.weight, dh, n, H, D, D, H, H, beta=1.0, a_off=r0 * D)
        # time-batched weight gradients
        gW, gbW = self._recurrent_grads(gbuf)
        if c.tc:
            datt1b = ops.to_bf16_padded(datt1)
        else:
            datt1b = None
        self._tn(c, dZ, c.dZb, c.Hprev, c.Hpb, gW, 4 * H, H, N, 4 * H, H, H)
        ops.colsum(dZ, N, 4 * H, 4 * H, gbW)
        self._tn(c, datt2, datt2b, c.Hprev, c.Hpb, self._gview(gbuf, [pre + "decoder_att.weight"], (A, H)), A, H, N, A, H, H)
        ops.colsum(datt2, N, A, A, self._gview(gbuf, [pre + "decoder_att.bias"], (A,)))
        self._tn(c, dgate, dgateb, c.Hprev, c.Hpb, self._gview(gbuf, ["f_beta.weight"], (D, H)), D, H, N, D, H, H)
        ops.colsum(dgate, N, D, D, self._gview(gbuf, ["f_beta.bias"], (D,)))
        self._tn(c, datt1, datt1b, c.feats.view(B * P, D), c.featsb,
                 self._gview(gbuf, [pre + "encoder_att.weight"], (A, D)), A, D, B * P, A, D, D)
        ops.colsum(datt1, B * P, A, A, self._gview(gbuf, [pre + "encoder_att.bias"], (A,)))
        # init_h / init_c: dh, dc now hold dL/dh0, dL/dc0.  K = B rows only: kept in fp32 FFMA in both modes (these
        # gradients sit at the end of the longest backward chain and are the most rounding-sensitive).
        ops.gemm(ops.OP_TN, dh, c.mean, self._gview(gbuf, ["init_h.weight"], (H, D)), H, D, B, H, D, D)
        ops.colsum(dh, B, H, H, self._gview(gbuf, ["init_h.bias"], (H,)))
        ops.gemm(ops.OP_TN, dc, c.mean, self._gview(gbuf, ["init_c.weight"], (H, D)), H, D, B, H, D, D)
        ops.colsum(dc, B, H, H, self._gview(gbuf, ["init_c.bias"], (H,)))
        dX = self._proj_weight_grads(c, dZ, gbuf)
        gE = self._gview(gbuf, [self._emb_name()], emb.weight.shape)
        gE.zero_()
        ops.gather_pack_bwd(c.captions, gE, None, False, d["row_b"], d["row_t"], c.tok_override, N, dX, c.p_drop, c.seed,
                            seed_dev=c.seed_dev)
        if need_dfeat:
            dmean = torch.empty(B, D, **f32)
            ops.gemm(ops.OP_NN, dh, self.init_h.weight, dmean, B, D, H, H, D, D)
            ops.gemm(ops.OP_NN, dc, self.init_c.weight, dmean, B, D, H, H, D, D, beta=1.0)
            dfeat += (dmean / P).unsqueeze(1)
            # through the hoisted encoder_att GEMM
            ops.gemm(ops.OP_NN, datt1, att.encoder_att.weight, dfeat.view(B * P, D), B * P, D, A, A, D, D, beta=1.0)
        return dfeat

    # ---- public ------------------------------------------------------------------------------------
    def _forward_att(self, captions, lengths, features, teacher_forcing_ratio, mode):
        self._check_inputs(captions, features)
        plan = get_plan(lengths)
        if plan.B != captions.shape[0]:
            raise RuntimeError("len(lengths) != batch size")
        if plan.T > captions.shape[1]:
            raise RuntimeError("lengths exceed the caption length")
        coins = self._coins(plan.T, teacher_forcing_ratio)
        captions = captions.contiguous()
        save = torch.is_grad_enabled()
        hall, alphas = _HiddenAttFn.apply(self._out().weight, features, self, plan, captions, coins, mode, save)
        from .decoders import _LogitsFn
        return _LogitsFn.apply(hall, self._out().weight, self), alphas

    def forward_loss(self, captions, lengths, features, targets=None, teacher_forcing_ratio=1.0, mode="factual",
                     backward=True, n_global=None, b_global=None, alpha_c=1.0, full_captions=None,
                     grad_hook=None):
        """Fused training entry point for the attention decoders: CE mean + alpha_c * mean((1-sum_t a)^2)
        (stylenet/train_multitask_att.py:402-411), forward and backward without an autograd graph.
        ``captions`` are the INPUT tokens (reference passes captions[:, :-1]); give the packed ``targets``
        or ``full_captions`` (then targets = packed full_captions[:, 1:])."""
        self._check_inputs(captions, features)
        plan = get_plan(lengths)
        coins = self._coins(plan.T, teacher_forcing_ratio)
        captions = captions.contiguous()
        dev = captions.device
        with torch.no_grad():
            c = self._run_forward_att(plan, captions, features, coins, mode, backward)
            N, B, P = plan.N, plan.B, c.P
            if targets is None:
                if full_captions is None:
                    raise ValueError("forward_loss: pass `targets` or `full_captions`")
                d = plan.dev(dev)
                targets = full_captions[d["row_b"].long(), d["row_t"].long() + 1].contiguous()
            out = self._out()
            V = out.weight.shape[0]
            denom = float(n_global if n_global is not None else N)
            row_loss, argmax, top5, logits, dLb = self._vocab_nll(c.Hall, None, targets, denom, backward)
            loss = torch.empty(1, dtype=torch.float32, device=dev)
            ops.reduce_sum(row_loss, N, 1.0 / denom, loss)
            # doubly stochastic regulariser: tiny [B,P] reduction (plumbing-size torch ops)
            bp = float((b_global if b_global is not None else B) * P)
            resid = 1.0 - c.alphas.sum(dim=1)
            loss += alpha_c * (resid * resid).sum() / bp
            if backward:
                dAl = (-2.0 * alpha_c / bp) * resid                       # d/d alpha[b,t,p], same for every t
                dAl = dAl.unsqueeze(1).expand(B, c.alphas.shape[1], P).contiguous()
                names = c.grad_names + list(self._out_names())
                gbuf = self._grad_target(names)
                dHall = self._vocab_backward(c.Hall, logits, gbuf, None, dLb)
                self._join()
                if grad_hook is not None and gbuf is self.arena().gflat:
                    grad_hook(list(self._out_names()))
                dfeat = self._run_backward_att(c, dHall, dAl, gbuf, features.requires_grad)
                self._publish(names, gbuf)
                if grad_hook is not None:
                    grad_hook(c.grad_names if gbuf is self.arena().gflat else names)
                if dfeat is not None:
                    dfeat = dfeat.view(features.shape)
                    features.grad = dfeat if features.grad is None else features.grad + dfeat
        return loss, {"argmax": argmax, "top5hit": top5, "n_tokens": N, "alphas": c.alphas}


class DecoderFactoredLSTMAtt(_AttBase):
    """Signature of stylenet/model_att.py:75-85."""

    cell = ops.CELL_FACTORED

    def __init__(self, attention_size, embed_size, hidden_size, factored_size, vocab_size, num_layers,
                 feature_size=2048, bias=True, dropout=0.22, max_seq_length=40):
        super().__init__()
        if not bias:
            raise NotImplementedError("bias=False is not supported by the fused path")
        self.attention_size, self.feature_size = attention_size, feature_size
        self.hidden_size, self.factored_size, self.embed_size = hidden_size, factored_size, embed_size
        self.vocab_size, self.max_seq_length, self.num_layers = vocab_size, max_seq_length, num_layers
        self.init_h = nn.Linear(feature_size, hidden_size)
        self.init_c = nn.Linear(feature_size, hidden_size)
        self.dropout = nn.Dropout(dropout)
        self.attention = Attention(feature_size, hidden_size, attention_size)
        self.B = nn.Embedding(vocab_size, embed_size)
        self.f_beta = nn.Linear(hidden_size, feature_size)
        for g in GATES:
            setattr(self, "U_" + g, nn.Linear(factored_size, hidden_size, bias=bias))
            setattr(self, style_attr("factual", g), nn.Linear(factored_size, factored_size, bias=bias))
            setattr(self, "V_" + g, nn.Linear(embed_size + feature_size, factored_size, bias=bias))
            setattr(self, "W_" + g, nn.Linear(hidden_size, hidden_size, bias=bias))
        for s in STYLES[1:]:
            setattr(self, att_attr(s), Attention(feature_size, hidden_size, attention_size))
            for g in GATES:
                setattr(self, style_attr(s, g), nn.Linear(factored_size, factored_size, bias=bias))
        self.C = nn.Linear(hidden_size, vocab_size, bias=bias)
        _ref_init(self, self.B, self.C)

    # reuse the non-attention factored helpers
    from .decoders import DecoderFactoredLSTM as _F
    _lp = staticmethod(_F._lp)
    _stack = _F._stack
    _style_stack = _F._style_stack
    _recurrent_weights = _F._recurrent_weights
    _recurrent_grads = _F._recurrent_grads
    _input_projection = _F._input_projection
    _small_step = _F._small_step
    del _F

    def _arena_groups(self):
        groups = [["B.weight"]]
        for pre in ("V_", "U_", "W_"):
            groups.append([pre + g + ".weight" for g in GATES])
            groups.append([pre + g + ".bias" for g in GATES])
        for s in STYLES:
            groups.append([style_attr(s, g) + ".weight" for g in GATES])
            groups.append([style_attr(s, g) + ".bias" for g in GATES])
        for s in STYLES:
            p = att_attr(s) + "."
            groups += [[p + "encoder_att.weight"], [p + "encoder_att.bias"], [p + "decoder_att.weight"],
                       [p + "decoder_att.bias"], [p + "full_att.weight"], [p + "full_att.bias"]]
        groups += [["init_h.weight"], ["init_h.bias"], ["init_c.weight"], ["init_c.bias"],
                   ["f_beta.weight"], ["f_beta.bias"], ["C.weight"], ["C.bias"]]
        return groups

    def _emb(self):
        return self.B

    def _emb_name(self):
        return "B.weight"

    def _out(self):
        return self.C

    def _out_names(self):
        return ("C.weight", "C.bias")

    def _att_module(self, mode):
        if mode not in STYLES:
            raise ValueError("mode name wrong: %r (expected one of %s)" % (mode, STYLES))
        return getattr(self, att_attr(mode))

    def _att_prefix(self, mode):
        return att_attr(mode) + "."

    def _seq_grad_names(self, mode):
        names = ["B.weight"]
        for pre in ("V_", "U_", "W_"):
            names += [pre + g + sfx for g in GATES for sfx in (".weight", ".bias")]
        names += [style_attr(mode, g) + sfx for g in GATES for sfx in (".weight", ".bias")]
        p = att_attr(mode) + "."
        names += [p + n for n in ("encoder_att.weight", "encoder_att.bias", "decoder_att.weight", "decoder_att.bias",
                                  "full_att.weight", "full_att.bias")]
        names += ["init_h.weight", "init_h.bias", "init_c.weight", "init_c.bias", "f_beta.weight", "f_beta.bias"]
        return names

    # -- projection pieces: V x = V[:, :E] emb + V[:, E:] ctx ----------------------------------------------
    def _proj_prepare(self, c):
        if not c.tc:
            return
        H, F, E, D = self.hidden_size, self.factored_size, self.embed_size, self.feature_size
        Vc = self._stack("V_", (4 * F, E + D))
        Ep = (E + 7) // 8 * 8
        Vemb = torch.empty(4 * F, Ep, dtype=torch.bfloat16, device=Vc.device)
        Vctx = torch.empty(4 * F, D, dtype=torch.bfloat16, device=Vc.device)
        ops.cast_bf16(Vc, 4 * F, E, E + D, Vemb, Ep, Ep)
        ops.cast_bf16(Vc, 4 * F, D, E + D, Vctx, D, D, src_off=E)
        c.w16["Vemb"], c.w16["Vctx"] = Vemb, Vctx
        c.w16["S"] = ops.to_bf16_padded(self._style_stack(c.mode, (4 * F, F)))
        c.w16["U"] = ops.to_bf16_padded(self._stack("U_", (4 * H, F)))

    def _proj_embed_part(self, c, r0, n):
        H, F, E, D = self.hidden_size, self.factored_size, self.embed_size, self.feature_size
        dev = c.XP.device
        if r0 == 0 and n == c.XP.shape[0]:
            c.A1 = torch.empty(n, 4 * F, dtype=torch.float32, device=dev)
            if c.tc:
                c.A1b = torch.empty(n, 4 * F, dtype=torch.bfloat16, device=dev)
                c.A2 = torch.empty(n, 4 * F, dtype=torch.bfloat16, device=dev)
            else:
                c.A2 = torch.empty(n, 4 * F, dtype=torch.float32, device=dev)
        bV = self._stack("V_", (4 * F,), bias=True)
        if c.tc:
            Vb = c.w16["Vemb"]
            Ep = Vb.stride(0)
            ops.gemm_bf16(ops.OP_NT, c.Xb, Vb, n, 4 * F, Ep, Ep, Ep, C=c.A1, ldc=4 * F, bias=bV, a_off=r0 * Ep,
                          c_off=r0 * 4 * F)
            return
        Vc = self._stack("V_", (4 * F, E + D))
        ops.gemm(ops.OP_NT, c.X, Vc, c.A1, n, 4 * F, E, E, E + D, 4 * F, bias=bV, a_off=r0 * E, c_off=r0 * 4 * F)

    def _proj_step(self, c, r0, n):
        H, F, E, D = self.hidden_size, self.factored_size, self.embed_size, self.feature_size
        bS = self._style_stack(c.mode, (4 * F,), bias=True)
        bU = self._stack("U_", (4 * H,), bias=True)
        if c.tc:
            Vx, Sb, Ub = c.w16["Vctx"], c.w16["S"], c.w16["U"]
            ops.gemm_bf16(ops.OP_NT, c.CTXb, Vx, n, 4 * F, D, D, D, C=c.A1, ldc=4 * F, Cb=c.A1b, ldcb=4 * F, beta=1.0,
                          a_off=r0 * D, c_off=r0 * 4 * F, cb_off=r0 * 4 * F)
            ops.gemm_bf16(ops.OP_NT, c.A1b, Sb, n, F, F, 4 * F, F, Cb=c.A2, ldcb=4 * F, bias=bS, batch=4, sA=F, sB=F * F,
                          sCb=F, sBias=F, a_off=r0 * 4 * F, cb_off=r0 * 4 * F)
            ops.gemm_bf16(ops.OP_NT, c.A2, Ub, n, H, F, 4 * F, F, C=c.XP, ldc=4 * H, bias=bU, batch=4, sA=F, sB=H * F,
                          sC=H, sBias=H, a_off=r0 * 4 * F, c_off=r0 * 4 * H)
            return
        Vc = self._stack("V_", (4 * F, E + D))
        Sc = self._style_stack(c.mode, (4 * F, F))
        Uc = self._stack("U_", (4 * H, F))
        ops.gemm(ops.OP_NT, c.CTX, Vc, c.A1, n, 4 * F, D, D, E + D, 4 * F, beta=1.0, a_off=r0 * D, b_off=E,
                 c_off=r0 * 4 * F)
        ops.gemm(ops.OP_NT, c.A1, Sc, c.A2, n, F, F, 4 * F, F, 4 * F, bias=bS, batch=4, sA=F, sB=F * F, sC=F,
                 sBias=F, a_off=r0 * 4 * F, c_off=r0 * 4 * F)
        ops.gemm(ops.OP_NT, c.A2, Uc, c.XP, n, H, F, 4 * F, F, 4 * H, bias=bU, batch=4, sA=F, sB=H * F, sC=H,
                 sBias=H, a_off=r0 * 4 * F, c_off=r0 * 4 * H)

    def _proj_bwd_begin(self, c, N):
        F = self.factored_size
        dev = c.XP.device
        c.dA2 = torch.empty(N, 4 * F, dtype=torch.float32, device=dev)
        c.dA1 = torch.empty(N, 4 * F, dtype=torch.float32, device=dev)
        if c.tc:
            c.dA2b = torch.empty(N, 4 * F, dtype=torch.bfloat16, device=dev)
            c.dA1b = torch.empty(N, 4 * F, dtype=torch.bfloat16, device=dev)

    def _proj_step_bwd(self, c, dZ, r0, n):
        H, F, E, D = self.hidden_size, self.factored_size, self.embed_size, self.feature_size
        if c.tc:
            Vx, Sb, Ub = c.w16["Vctx"], c.w16["S"], c.w16["U"]
            ops.gemm_bf16(ops.OP_NN, c.dZb, Ub, n, F, H, 4 * H, F, C=c.dA2, ldc=4 * F, Cb=c.dA2b, ldcb=4 * F, batch=4,
                          sA=H, sB=H * F, sC=F, sCb=F, a_off=r0 * 4 * H, c_off=r0 * 4 * F, cb_off=r0 * 4 * F)
            ops.gemm_bf16(ops.OP_NN, c.dA2b, Sb, n, F, F, 4 * F, F, C=c.dA1, ldc=4 * F, Cb=c.dA1b, ldcb=4 * F, batch=4,
                          sA=F, sB=F * F, sC=F, sCb=F, a_off=r0 * 4 * F, c_off=r0 * 4 * F, cb_off=r0 * 4 * F)
            ops.gemm_bf16(ops.OP_NN, c.dA1b, Vx, n, D, 4 * F, 4 * F, D, C=c.dCTX, ldc=D, a_off=r0 * 4 * F, c_off=r0 * D)
            return
        Vc = self._stack("V_", (4 * F, E + D))
        Sc = self._style_stack(c.mode, (4 * F, F))
        Uc = self._stack("U_", (4 * H, F))
        ops.gemm(ops.OP_NN, dZ, Uc, c.dA2, n, F, H, 4 * H, F, 4 * F, batch=4, sA=H, sB=H * F, sC=F,
                 a_off=r0 * 4 * H, c_off=r0 * 4 * F)
        ops.gemm(ops.OP_NN, c.dA2, Sc, c.dA1, n, F, F, 4 * F, F, 4 * F, batch=4, sA=F, sB=F * F, sC=F,
                 a_off=r0 * 4 * F, c_off=r0 * 4 * F)
        ops.gemm(ops.OP_NN, c.dA1, Vc, c.dCTX, n, D, 4 * F, 4 * F, E + D, D, a_off=r0 * 4 * F, b_off=E, c_off=r0 * D)

    def _proj_weight_grads(self, c, dZ, gbuf):
        H, F, E, D = self.hidden_size, self.factored_size, self.embed_size, self.feature_size
        N = dZ.shape[0]
        mode = c.mode
        gV, gbV = self._stack("V_", (4 * F, E + D), gbuf=gbuf), self._stack("V_", (4 * F,), gbuf=gbuf, bias=True)
        gS, gbS = self._style_stack(mode, (4 * F, F), gbuf=gbuf), self._style_stack(mode, (4 * F,), gbuf=gbuf, bias=True)
        gU, gbU = self._stack("U_", (4 * H, F), gbuf=gbuf), self._stack("U_", (4 * H,), gbuf=gbuf, bias=True)
        ops.colsum(dZ, N, 4 * H, 4 * H, gbU)
        ops.colsum(c.dA2, N, 4 * F, 4 * F, gbS)
        ops.colsum(c.dA1, N, 4 * F, 4 * F, gbV)
        dX = torch.empty(N, E, dtype=torch.float32, device=dZ.device)
        if c.tc:
            Vb = c.w16["Vemb"]
            Ep = Vb.stride(0)
            ops.gemm_bf16(ops.OP_TN, c.dZb, c.A2, H, F, N, 4 * H, 4 * F, C=gU, ldc=F, batch=4, sA=H, sB=F, sC=H * F)
            ops.gemm_bf16(ops.OP_TN, c.dA2b, c.A1b, F, F, N, 4 * F, 4 * F, C=gS, ldc=F, batch=4, sA=F, sB=F, sC=F * F)
            ops.gemm_bf16(ops.OP_TN, c.dA1b, c.Xb, 4 * F, E, N, 4 * F, Ep, C=gV, ldc=E + D)
            ops.gemm_bf16(ops.OP_TN, c.dA1b, c.CTXb, 4 * F, D, N, 4 * F, D, C=gV, ldc=E + D, c_off=E)
            ops.gemm_bf16(ops.OP_NN, c.dA1b, Vb, N, E, 4 * F, 4 * F, Ep, C=dX, ldc=E)
            return dX
        Vc = self._stack("V_", (4 * F, E + D))
        ops.gemm(ops.OP_TN, dZ, c.A2, gU, H, F, N, 4 * H, 4 * F, F, batch=4, sA=H, sB=F, sC=H * F)
        ops.gemm(ops.OP_TN, c.dA2, c.A1, gS, F, F, N, 4 * F, 4 * F, F, batch=4, sA=F, sB=F, sC=F * F)
        ops.gemm(ops.OP_TN, c.dA1, c.X, gV, 4 * F, E, N, 4 * F, E, E + D)
        ops.gemm(ops.OP_TN, c.dA1, c.CTX, gV, 4 * F, D, N, 4 * F, D, E + D, c_off=E)
        ops.gemm(ops.OP_NN, c.dA1, Vc, dX, N, E, 4 * F, 4 * F, E + D, E)
        return dX

    # -- reference surface ----------------------------------------------------------------------------
    def forward(self, captions, lengths, features, teacher_forcing_ratio=0.8, mode="factual"):
        """(outputs [sum(lengths), V], alphas [B, max(lengths), P]) like model_att.py:238-305."""
        self._att_module(mode)
        return self._forward_att(captions, lengths, features, teacher_forcing_ratio, mode)

    def forward_step(self, embedded, states, mode):
        from .decode import single_step
        return single_step(self, embedded, states, mode)

    def sample(self, features, start_token, end_token, k=5, factual_limit=-1, mode="factual"):
        """Beam search with attention, stylenet/model_att.py:307-426."""
        from .decode import beam_sample_att, require_one_style
        require_one_style(mode)
        return beam_sample_att(self, features, start_token, end_token, k, mode)[0]

    def sample_batch(self, features, start_token, end_token, k=5, mode="factual"):
        """``sample()`` for every image of ``features [n_img, S, S, D]`` in one batched beam search; returns a list of
        LongTensor [1, L_i] (replaces the per-image loop of stylenet/evaluator.py:74-81).  ``mode`` may be a list /
        tuple of n_img style names: image i in style ``mode[i]``, all in one beam search."""
        from .decode import beam_sample_att
        return beam_sample_att(self, features, start_token, end_token, k, mode)


class DecoderRNNAtt(_AttBase):
    """Signature of nic/model_att.py:74-82."""

    cell = ops.CELL_LSTM

    def __init__(self, attention_size, embed_size, hidden_size, vocab_size, num_layers, feature_size=2048,
                 dropout=0.22, max_seq_length=40):
        super().__init__()
        self.attention_size, self.feature_size = attention_size, feature_size
        self.hidden_size, self.embed_size = hidden_size, embed_size
        self.vocab_size, self.max_seq_length, self.num_layers = vocab_size, max_seq_length, num_layers
        self.init_h = nn.Linear(feature_size, hidden_size)
        self.init_c = nn.Linear(feature_size, hidden_size)
        self.dropout = nn.Dropout(dropout)
        self.attention = Attention(feature_size, hidden_size, attention_size)
        self.embed = nn.Embedding(vocab_size, embed_size)
        self.f_beta = nn.Linear(hidden_size, feature_size)
        self.lstm = nn.LSTMCell(embed_size + feature_size, hidden_size, bias=True)
        self.linear = nn.Linear(hidden_size, vocab_size)
        _ref_init(self, self.embed, self.linear)

    def _arena_groups(self):
        p = "attention."
        return [["embed.weight"], ["lstm.weight_ih"], ["lstm.weight_hh"], ["lstm.bias_ih"], ["lstm.bias_hh"],
                [p + "encoder_att.weight"], [p + "encoder_att.bias"], [p + "decoder_att.weight"],
                [p + "decoder_att.bias"], [p + "full_att.weight"], [p + "full_att.bias"],
                ["init_h.weight"], ["init_h.bias"], ["init_c.weight"], ["init_c.bias"],
                ["f_beta.weight"], ["f_beta.bias"], ["linear.weight"], ["linear.bias"]]

    def _emb(self):
        return self.embed

    def _emb_name(self):
        return "embed.weight"

    def _out(self):
        return self.linear

    def _out_names(self):
        return ("linear.weight", "linear.bias")

    def _att_module(self, mode):
        return self.attention

    def _att_prefix(self, mode):
        return "attention."

    def _recurrent_weights(self):
        self.arena()
        return self.lstm.weight_hh, self.lstm.bias_hh

    def _recurrent_grads(self, gbuf):
        H = self.hidden_size
        return self._gview(gbuf, ["lstm.weight_hh"], (4 * H, H)), self._gview(gbuf, ["lstm.bias_hh"], (4 * H,))

    def _seq_grad_names(self, mode):
        p = "attention."
        return ["embed.weight", "lstm.weight_ih", "lstm.weight_hh", "lstm.bias_ih", "lstm.bias_hh"] + \
            [p + n for n in ("encoder_att.weight", "encoder_att.bias", "decoder_att.weight", "decoder_att.bias",
                             "full_att.weight", "full_att.bias")] + \
            ["init_h.weight", "init_h.bias", "init_c.weight", "init_c.bias", "f_beta.weight", "f_beta.bias"]

    def _small_step(self, ctx, X, mode, R, h_prev, c_prev, src_row, h_out, c_out):
        H = self.hidden_size
        self.arena()
        ops.decode_cell(self.cell, H, R, self.lstm.weight_ih, X.shape[1], X, 0, self.lstm.bias_ih, self.lstm.weight_hh,
                        self.lstm.bias_hh, h_prev, c_prev, src_row, h_out, c_out)

    def _input_projection(self, c, X, mode, r0, n):
        """Full-width projection (used by forward_step / decode where the input is already [emb, ctx])."""
        H = self.hidden_size
        Ein = X.shape[1]
        ops.gemm(ops.OP_NT, X, self.lstm.weight_ih, c.XP, n, 4 * H, Ein, Ein, Ein, 4 * H, bias=self.lstm.bias_ih,
                 a_off=r0 * Ein, c_off=r0 * 4 * H)

    def _proj_prepare(self, c):
        if not c.tc:
            return
        H, E, D = self.hidden_size, self.embed_size, self.feature_size
        W = self.lstm.weight_ih
        Ep = (E + 7) // 8 * 8
        Wemb = torch.empty(4 * H, Ep, dtype=torch.bfloat16, device=W.device)
        Wctx = torch.empty(4 * H, D, dtype=torch.bfloat16, device=W.device)
        ops.cast_bf16(W, 4 * H, E, E + D, Wemb, Ep, Ep)
        ops.cast_bf16(W, 4 * H, D, E + D, Wctx, D, D, src_off=E)
        c.w16["Wemb"], c.w16["Wctx"] = Wemb, Wctx

    def _proj_embed_part(self, c, r0, n):
        H, E, D = self.hidden_size, self.embed_size, self.feature_size
        if c.tc:
            Wb = c.w16["Wemb"]
            Ep = Wb.stride(0)
            ops.gemm_bf16(ops.OP_NT, c.Xb, Wb, n, 4 * H, Ep, Ep, Ep, C=c.XP, ldc=4 * H, bias=self.lstm.bias_ih,
                          a_off=r0 * Ep, c_off=r0 * 4 * H)
            return
        ops.gemm(ops.OP_NT, c.X, self.lstm.weight_ih, c.XP, n, 4 * H, E, E, E + D, 4 * H, bias=self.lstm.bias_ih,
                 a_off=r0 * E, c_off=r0 * 4 * H)

    def _proj_step(self, c, r0, n):
        H, E, D = self.hidden_size, self.embed_size, self.feature_size
        if c.tc:
            ops.gemm_bf16(ops.OP_NT, c.CTXb, c.w16["Wctx"], n, 4 * H, D, D, D, C=c.XP, ldc=4 * H, beta=1.0,
                          a_off=r0 * D, c_off=r0 * 4 * H)
            return
        ops.gemm(ops.OP_NT, c.CTX, self.lstm.weight_ih, c.XP, n, 4 * H, D, D, E + D, 4 * H, beta=1.0,
                 a_off=r0 * D, b_off=E, c_off=r0 * 4 * H)

    def _proj_bwd_begin(self, c, N):
        pass

    def _proj_step_bwd(self, c, dZ, r0, n):
        H, E, D = self.hidden_size, self.embed_size, self.feature_size
        if c.tc:
            ops.gemm_bf16(ops.OP_NN, c.dZb, c.w16["Wctx"], n, D, 4 * H, 4 * H, D, C=c.dCTX, ldc=D, a_off=r0 * 4 * H,
                          c_off=r0 * D)
            return
        ops.gemm(ops.OP_NN, dZ, self.lstm.weight_ih, c.dCTX, n, D, 4 * H, 4 * H, E + D, D, a_off=r0 * 4 * H,
                 b_off=E, c_off=r0 * D)

    def _proj_weight_grads(self, c, dZ, gbuf):
        H, E, D = self.hidden_size, self.embed_size, self.feature_size
        N = dZ.shape[0]
        gW = self._gview(gbuf, ["lstm.weight_ih"], (4 * H, E + D))
        ops.colsum(dZ, N, 4 * H, 4 * H, self._gview(gbuf, ["lstm.bias_ih"], (4 * H,)))
        dX = torch.empty(N, E, dtype=torch.float32, device=dZ.device)
        if c.tc:
            Wb = c.w16["Wemb"]
            Ep = Wb.stride(0)
            ops.gemm_bf16(ops.OP_TN, c.dZb, c.Xb, 4 * H, E, N, 4 * H, Ep, C=gW, ldc=E + D)
            ops.gemm_bf16(ops.OP_TN, c.dZb, c.CTXb, 4 * H, D, N, 4 * H, D, C=gW, ldc=E + D, c_off=E)
            ops.gemm_bf16(ops.OP_NN, c.dZb, Wb, N, E, 4 * H, 4 * H, Ep, C=dX, ldc=E)
            return dX
        ops.gemm(ops.OP_TN, dZ, c.X, gW, 4 * H, E, N, 4 * H, E, E + D)
        ops.gemm(ops.OP_TN, dZ, c.CTX, gW, 4 * H, D, N, 4 * H, D, E + D, c_off=E)
        ops.gemm(ops.OP_NN, dZ, self.lstm.weight_ih, dX, N, E, 4 * H, 4 * H, E + D, E)
        return dX

    def forward(self, captions, lengths, features, teacher_forcing_ratio=0.8):
        """(outputs, alphas) like nic/model_att.py:152-202."""
        return self._forward_att(captions, lengths, features, teacher_forcing_ratio, None)

    def forward_step(self, embedded, states):
        from .decode import single_step
        return single_step(self, embedded, states, None)

    def sample(self, features, start_token, end_token, k=5):
        """Beam search with attention, nic/model_att.py:204-306."""
        from .decode import beam_sample_att
        return beam_sample_att(self, features, start_token, end_token, k, None)[0]

    def sample_batch(self, features, start_token, end_token, k=5):
        """Batched ``sample()`` over every image of ``features [n_img, S, S, D]``."""
        from .decode import beam_sample_att
        return beam_sample_att(self, features, start_token, end_token, k, None)
