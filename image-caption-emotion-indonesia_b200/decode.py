"""Batched beam / greedy decoding on the kernels (K8): the reference's ``sample()`` semantics
(stylenet/model.py:198-294, nic/model.py:117-207, app/backend/model.py:386-487) for n_img images at
once, with all bookkeeping on the device and no host synchronisation inside the step loop."""
import ctypes
import weakref

import torch

from . import ops
from .ops import check

_small = {}


def _i32(device, vals):
    key = (str(device), tuple(vals))
    t = _small.get(key)
    if t is None:
        t = torch.tensor(list(vals), dtype=torch.int32, device=device)
        _small[key] = t
    return t


class _StepCtx:
    pass


class StyleGroups(tuple):
    """The style groups of a mixed-style decode call: ``(styles, counts)``, group g = ``counts[g]`` consecutive images
    captioned in ``styles[g]``.  Hashable: it is the ``mode`` part of the session key."""

    @property
    def styles(self):
        return self[0]

    @property
    def counts(self):
        return self[1]


def group_styles(modes, n_img, styles):
    """Stable grouping of a per-image style list (``sample_batch(..., mode=[...])``) in the order of ``styles``.
    Returns (StyleGroups, order): ``order[j]`` is the input index of the j-th image in grouped order.  Raises
    ValueError for an empty list, a length other than ``n_img`` or an unknown style -- before any device work."""
    if not isinstance(modes, (list, tuple)):
        raise ValueError("mode must be a style name or a list / tuple of them, got %r" % (modes,))
    if len(modes) == 0:
        raise ValueError("empty style list")
    if len(modes) != n_img:
        raise ValueError("style list of length %d for %d images" % (len(modes), n_img))
    for m in modes:
        if not isinstance(m, str) or m not in styles:
            raise ValueError("mode name wrong: %r (expected one of %s)" % (m, tuple(styles)))
    present = [s for s in styles if s in modes]
    order = [i for s in present for i in range(n_img) if modes[i] == s]
    counts = tuple(sum(1 for m in modes if m == s) for s in present)
    return StyleGroups((tuple(present), counts)), order


def require_one_style(mode):
    """``sample()`` captions one image in one style; a style list is ``sample_batch``'s."""
    if isinstance(mode, (list, tuple)):
        raise ValueError("sample() takes one style name; pass a per-image style list to sample_batch()")


def ungroup(results, order):
    """Results in grouped order back to input order."""
    out = [None] * len(order)
    for j, i in enumerate(order):
        out[i] = results[j]
    return out


def _n_layers(dec):
    """Stacked decoders (stack.DecoderFactoredLSTMStack) keep one (h, c) per layer; the reference models have one."""
    return int(dec.num_layers) if getattr(dec, "_layered", False) else 1


def _rw(dec, layer):
    return dec._recurrent_weights(layer) if layer else dec._recurrent_weights()


def single_step(dec, embedded, states, mode):
    """forward_step(embedded, states[, mode]) -> (h, (h, c)) on the kernels (inference only).  Stacked decoders take and
    return states of shape [num_layers, R, H]."""
    h, c = states
    L = _n_layers(dec)
    stacked = h.dim() == 3
    if L > 1 and not stacked:
        raise ValueError("the stack's forward_step takes states of shape [num_layers, R, H]")
    hs = h.detach().float().contiguous().reshape(L, -1, h.shape[-1])
    cs = c.detach().float().contiguous().reshape(L, -1, h.shape[-1])
    R, H = hs.shape[1], hs.shape[2]
    dev = h.device
    X = embedded.detach().float().contiguous()
    h_new = torch.empty(L, R, H, dtype=torch.float32, device=dev)
    c_new = torch.empty(L, R, H, dtype=torch.float32, device=dev)
    with torch.no_grad():
        ops.lib()
        dec.arena()
        for l in range(L):
            ctx = _StepCtx()
            ctx.layer = l
            kw = {"layer": l} if l else {}
            if R <= ops.SKINNY_MAX_ROWS:
                dec._small_step(ctx, X, mode, R, hs[l], cs[l], None, h_new[l], c_new[l], **kw)
            else:
                ctx.XP = torch.empty(R, 4 * H, dtype=torch.float32, device=dev)
                dec._input_projection(ctx, X, mode, 0, R)
                Whh, bhh = _rw(dec, l)
                c_new[l].copy_(cs[l])
                ops.recur_fwd(dec.cell, H, R, _i32(dev, [R]), _i32(dev, [0]), 0, 1, ctx.XP, Whh, bhh, hs[l], h_new[l],
                              None, None, None, c_new[l])
            X = h_new[l]
    if stacked:
        return h_new[L - 1], (h_new, c_new)
    return h_new[0], (h_new[0], c_new[0])


def _vocab_step(dec, h_new, logits, cache):
    """logits = C(h) for one decode step; bf16 mode runs it on tcgen05 with a cached bf16 copy of C."""
    out = dec._out()
    V, H = out.weight.shape
    R = h_new.shape[0]
    if dec.bf16 and H % 8 == 0:
        if "Wb" not in cache:
            cache["Wb"] = ops.to_bf16_padded(out.weight)
            cache["hb"] = torch.empty(R, H, dtype=torch.bfloat16, device=h_new.device)
        ops.cast_bf16(h_new, R, H, H, cache["hb"], H, H)
        ops.gemm_bf16(ops.OP_NT, cache["hb"], cache["Wb"], R, V, H, H, cache["Wb"].stride(0), C=logits, ldc=V,
                      bias=out.bias)
    else:
        ops.gemm(ops.OP_NT, h_new, out.weight, logits, R, V, H, H, H, V, bias=out.bias)


class BeamState:
    reorders = True          # the state rows follow the surviving beams (src_row) after every step

    def __init__(self, n_img, kmax, max_len, start_token, device):
        L = max_len + 2
        R = n_img * kmax
        self.n_img, self.kmax, self.max_len, self.L, self.R = n_img, kmax, max_len, L, R
        i32 = dict(dtype=torch.int32, device=device)
        self.k_live = torch.full((n_img,), kmax, **i32)
        self.run_score = torch.zeros(R, dtype=torch.float32, device=device)
        self.prev_word = torch.full((R,), start_token, **i32)
        self.src_row = torch.arange(R, **i32)
        self.cur_buf = torch.zeros(n_img, **i32)
        self.seqs = torch.zeros(2, R, L, **i32)
        self.seqs[:, :, 0] = start_token
        self.done_seq = torch.zeros(R, L, **i32)
        self.done_len = torch.zeros(R, **i32)
        self.done_score = torch.zeros(R, dtype=torch.float32, device=device)
        self.n_done = torch.zeros(n_img, **i32)
        self.out_seq = torch.zeros(n_img, L, **i32)
        self.out_len = torch.zeros(n_img, **i32)
        self.n_unfinished = torch.full((1,), n_img, **i32)
        self.step_dev = torch.ones(1, **i32)
        self.start_token = start_token
        self._arange = torch.arange(R, **i32)

    def reset(self):
        """Back to the state before step 1 (in place: the buffers may be baked into a CUDA graph)."""
        self.k_live.fill_(self.kmax)
        self.run_score.zero_()
        self.prev_word.fill_(self.start_token)
        self.src_row.copy_(self._arange)
        self.cur_buf.zero_()
        self.seqs[:, :, 0] = self.start_token
        self.n_done.zero_()
        self.out_len.zero_()
        self.n_unfinished.fill_(self.n_img)
        self.step_dev.fill_(1)

    SPLIT_MAX_IMAGES = 8          # up to here one CTA per image leaves the GPU idle: spread each image over chunks

    def step(self, logits, step, end_token, device_step=False, advance=False):
        """One beam step.  ``advance``: also add 1 to the device-side step counter (returns True when the kernel did it,
        False when the caller has to)."""
        p = ops._ptr
        V = logits.shape[1]
        if self.n_img <= self.SPLIT_MAX_IMAGES and V >= 256:
            nch = max(1, min(16, V // 128))
            ws = self.__dict__.get("_split_ws")
            if ws is None:
                n = ops.lib().sn_beam_split_ws_floats(self.n_img, self.kmax, nch)
                ws = self._split_ws = torch.zeros(n, dtype=torch.float32, device=logits.device)
            check(ops.lib().sn_beam_step_split(
                p(logits), logits.stride(0), V, self.n_img, self.kmax, step, self.max_len, end_token,
                p(self.k_live), p(self.run_score), p(self.prev_word), p(self.src_row), p(self.cur_buf), p(self.seqs),
                p(self.done_seq), p(self.done_len), p(self.done_score), p(self.n_done), p(self.out_seq),
                p(self.out_len), p(self.n_unfinished), p(self.step_dev) if device_step else None, nch, p(ws),
                1 if (advance and device_step) else 0, ops._stream()), "sn_beam_step_split")
            ops.LAUNCHES[0] += 2
            return bool(advance and device_step)
        check(ops.lib().sn_beam_step(
            p(logits), logits.stride(0), logits.shape[1], self.n_img, self.kmax, step, self.max_len, end_token,
            p(self.k_live), p(self.run_score), p(self.prev_word), p(self.src_row), p(self.cur_buf), p(self.seqs),
            p(self.done_seq), p(self.done_len), p(self.done_score), p(self.n_done), p(self.out_seq),
            p(self.out_len), p(self.n_unfinished), p(self.step_dev) if device_step else None, ops._stream()),
            "sn_beam_step")

    def results(self):
        pk = torch.cat([self.out_seq, self.out_len.unsqueeze(1)], 1).cpu()        # one device->host copy, one sync
        L = self.out_seq.shape[1]
        return [pk[i, :int(pk[i, L])].long().unsqueeze(0) for i in range(self.n_img)]


class SampleState:
    """Device state of a sampling decode (K12, ``sample_captions``): n independent samples of each of n_img images, row
    i * n + j = sample j of image i.  No beam re-ordering: ``src_row`` is the identity.  ``seed_dev`` and ``step_dev``
    feed the noise from device memory (include/sn100.h, sn_sample_step)."""
    reorders = False

    def __init__(self, n_img, n, max_len, start_token, temperature, greedy, device):
        L = max_len + 2
        R = n_img * n
        self.n_img, self.kmax, self.max_len, self.L, self.R = n_img, n, max_len, L, R
        self.start_token, self.temperature, self.greedy = start_token, float(temperature), bool(greedy)
        i32 = dict(dtype=torch.int32, device=device)
        self.prev_word = torch.full((R,), start_token, **i32)
        self.src_row = torch.arange(R, **i32)
        self.seqs = torch.zeros(R, L, dtype=torch.int64, device=device)
        self.lengths = torch.zeros(R, dtype=torch.int64, device=device)
        self.logprob = torch.zeros(R, L - 1, dtype=torch.float32, device=device)
        self.done = torch.zeros(R, **i32)
        self.n_unfinished = torch.full((1,), R, **i32)
        self.step_dev = torch.ones(1, **i32)
        self.seed_dev = torch.zeros(1, dtype=torch.int64, device=device)
        self.reset()

    def reset(self):
        """Back to the state before the first draw (in place: the buffers may be baked into a CUDA graph)."""
        self.prev_word.fill_(self.start_token)
        self.seqs.zero_()
        self.seqs[:, 0] = self.start_token
        self.lengths.zero_()
        self.logprob.zero_()
        self.done.zero_()
        self.n_unfinished.fill_(self.R)
        self.step_dev.fill_(1)

    def step(self, logits, step, end_token, device_step=False, advance=False):
        """One draw per live row; the step index comes from ``step_dev``, which the caller advances (returns False)."""
        ops.sample_step(logits, logits.shape[1], self.R, self.max_len, end_token, self.temperature, self.greedy,
                        self.seed_dev, self.step_dev, self.prev_word, self.seqs, self.lengths, self.logprob, self.done,
                        self.n_unfinished)
        return False

    def results(self):
        return self.seqs.clone(), self.lengths.clone(), self.logprob.clone()


class _DecodeSession:
    """Static buffers + (lazily captured) CUDA graphs of one decode step for a fixed (decoder, n_img, k, mode,
    start/end token).  ``sample()`` is called once per image by the reference's evaluation loops
    (stylenet/evaluator.py:74-81): replaying the captured step removes the ~12 Python-issued launches per step
    that otherwise make a single-image beam search launch-bound."""

    def __init__(self, dec, n_img, k, mode, start_token, end_token, state=None):
        emb = dec._emb()
        dev = emb.weight.device
        E, H = emb.weight.shape[1], dec.hidden_size
        out = dec._out()
        V = out.weight.shape[0]
        self._dec = weakref.ref(dec)          # the decoder owns its sessions: no reference cycle
        self.mode, self.end_token = mode, end_token
        self.st = state if state is not None else BeamState(n_img, k, dec.max_seq_length, start_token, dev)
        R = self.st.R
        f32 = dict(dtype=torch.float32, device=dev)
        self.L = L = _n_layers(dec)
        self.h, self.c = torch.zeros(L, R, H, **f32), torch.zeros(L, R, H, **f32)      # one state per layer
        self.h_new = torch.empty(L, R, H, **f32)
        self.logits = torch.empty(R, V, **f32)
        self.X = torch.empty(R, E, **f32)
        self.ctx = _StepCtx()
        self.ctx.XP = torch.empty(R, 4 * H, **f32)
        self.ctx.w16 = {}
        self.row_img = (torch.arange(R, device=dev, dtype=torch.int32) // k).contiguous()
        self.row_zero = torch.zeros(R, dtype=torch.int32, device=dev)
        self.dummy_cap = torch.zeros(1, 1, dtype=torch.int64, device=dev)
        self.feats = torch.zeros(n_img, E, **f32)
        self.bs1, self.off1 = _i32(dev, [R]), _i32(dev, [0])
        self.cache = {}
        self.graph = None          # generic step (steps >= 2)
        self.calls = 0
        self.arena_version = dec.arena().version
        # mixed styles: group g = rows [row_off[g], row_off[g+1]) in style groups.styles[g]
        self.groups = mode if isinstance(mode, StyleGroups) else None
        if self.groups is not None:
            self.row_off = [0]
            for n in self.groups.counts:
                self.row_off.append(self.row_off[-1] + n * k)
            self.row_off_dev = _i32(dev, self.row_off)
            self.rows_max = max(self.groups.counts) * k
            self.gctx = [[_StepCtx() for _ in self.groups.styles] for _ in range(L)]
            for l in range(L):
                for g, gc in enumerate(self.gctx[l]):
                    gc.layer, gc.w16 = l, {}
                    gc.XP = self.ctx.XP[self.row_off[g]:self.row_off[g + 1]]     # the group's rows of the shared XP
        # few rows (single-image beam search): matrix-vector kernels, state double-buffered (A -> B -> A ...), the beam
        # re-ordering of the state folded into the next step's read (no index_select kernels)
        self.skinny = R <= (ops.SKINNY_MAX_ROWS if self.groups is None else
                            min(STYLES_SKINNY_MAX_ROWS[0], ops.SKINNY_LINEAR_MAX_ROWS))
        if self.skinny:
            self.hB, self.cB = torch.zeros(L, R, H, **f32), torch.zeros(L, R, H, **f32)
            self.flip = 0              # 0: the state is in (h, c); 1: in (hB, cB)

    def step(self, step, feed_image, device_step, draw=True):
        """One decode step.  ``draw=False``: advance the state only (the image step of sampling decode, whose output
        is discarded)."""
        dec, st = self._dec(), self.st
        emb, out = dec._emb(), dec._out()
        R, H = st.R, dec.hidden_size
        if feed_image and step == 1:
            ops.gather_pack_fwd(self.dummy_cap, emb.weight, self.feats, True, self.row_img, self.row_zero, None, R,
                                self.X, 0.0, 0)
        else:
            ops.gather_pack_fwd(self.dummy_cap, emb.weight, None, False, self.row_img, self.row_zero, st.prev_word, R,
                                self.X, 0.0, 0)
        X = self.X
        for l in range(self.L):
            self.ctx.layer = l
            if self.groups is not None:
                # the chain per group on its rows of XP.  Only S is the group's: the V stage (and, in bf16 mode, the V / U
                # weight shadows) is recomputed per group -- G - 1 redundant V GEMMs per step; sharing it would need a
                # split of _input_projection into its stages
                for g, style in enumerate(self.groups.styles):
                    r0, r1 = self.row_off[g], self.row_off[g + 1]
                    dec._input_projection(self.gctx[l][g], X[r0:r1], style, 0, r1 - r0)
            else:
                if self.L > 1:
                    self.ctx.w16 = self.__dict__.setdefault("_w16_layers", {}).setdefault(l, {})
                dec._input_projection(self.ctx, X, self.mode, 0, R)
            Whh, bhh = _rw(dec, l)
            ops.recur_fwd(dec.cell, H, R, self.bs1, self.off1, 0, 1, self.ctx.XP, Whh, bhh, self.h[l], self.h_new[l], None,
                          None, None, self.c[l])
            X = self.h_new[l]
        if draw:
            _vocab_step(dec, self.h_new[self.L - 1], self.logits, self.cache)
            st.step(self.logits, step, self.end_token, device_step=device_step)
        if st.reorders:
            idx = st.src_row.long()
            for l in range(self.L):
                torch.index_select(self.h_new[l], 0, idx, out=self.h[l])
                c_new = self.c[l].index_select(0, idx)
                self.c[l].copy_(c_new)
        else:
            self.h.copy_(self.h_new)              # (recur_fwd updated c in place)
        if draw:
            st.step_dev.add_(1)

    def step_skinny(self, step, feed_image, device_step, draw=True):
        dec, st = self._dec(), self.st
        emb, out = dec._emb(), dec._out()
        R = st.R
        fold = hasattr(dec, "factored_size")          # factored decoders: the lookup is folded into the V stage
        if feed_image and step == 1:
            X, rows = self.feats, self.row_img             # row r reads the feature row of its image
        else:
            X, rows = emb.weight, st.prev_word             # row r reads the embedding of its previous word
        if not fold:
            ops.gather_pack_fwd(self.dummy_cap, emb.weight, self.feats if (feed_image and step == 1) else None,
                                feed_image and step == 1, self.row_img, self.row_zero,
                                None if (feed_image and step == 1) else st.prev_word, R, self.X, 0.0, 0)
            X, rows = self.X, None
        src = (self.h, self.c) if self.flip == 0 else (self.hB, self.cB)
        dst = (self.hB, self.cB) if self.flip == 0 else (self.h, self.c)
        for l in range(self.L):
            if self.groups is not None:
                # every style group in one launch, each with the collapsed chain of its style (_collapse_styles)
                ent = self.ctx.collapsed_groups[l]
                Whh, bhh = _rw(dec, l)
                ops.decode_cell_groups(dec.cell, dec.hidden_size, self.row_off_dev, self.rows_max, ent["Wc"], X.shape[1],
                                       X, 0, ent["bc"], Whh, bhh, src[0][l], src[1][l], st.src_row, dst[0][l],
                                       dst[1][l], x_rows=rows if l == 0 else None)
                X = dst[0][l]
                continue
            kw = {"layer": l} if l else {}
            if l == 0 and rows is not None:
                kw["x_rows"] = rows
            dec._small_step(self.ctx, X, self.mode, R, src[0][l], src[1][l], st.src_row, dst[0][l], dst[1][l], **kw)
            X = dst[0][l]
        if draw:
            ops.skinny_linear(out.weight, dst[0][self.L - 1], self.logits, R, bias=out.bias)
            if not st.step(self.logits, step, self.end_token, device_step=device_step, advance=True):
                st.step_dev.add_(1)
        self.flip ^= 1

    STEPS_PER_GRAPH = 4

    def capture_skinny(self):
        """One graph = STEPS_PER_GRAPH consecutive steps (an even number: the state ends in the buffer it started in).
        Captured right after a restart: replays read the state from the buffer a restart leaves it in."""
        assert self.STEPS_PER_GRAPH % 2 == 0
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                self.step_skinny(2, False, True)      # warm-up on the capture side stream
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with ops.no_gc_during_capture(), torch.cuda.graph(g):
            for _ in range(self.STEPS_PER_GRAPH):
                self.step_skinny(2, False, True)
        self.graph = g

    def capture(self):
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self.step(2, False, True)            # warm-up on the capture side stream (allocator, lazy state)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        with ops.no_gc_during_capture(), torch.cuda.graph(g):
            self.step(2, False, True)
        self.graph = g


COLLAPSE_CHAIN = [True]       # few-row decode: collapse the factored chain once per call (DecoderFactoredLSTM._collapse_chain)
# mixed-style decode (sample_batch with a style list): up to this many rows (images x k) on the matrix-vector kernels
# (sn_decode_cell_groups + the row-chunked vocabulary projection), above it on the GEMM path.  Set from bench_styles.py
# (profiles/styles_bench_N1.jsonl, one B200 at 1000 W): the few-row path led at every size swept, 20 / 40 / 80 / 120 rows
# (2.4 / 5.3 / 8.4 / 18.6 ms per request vs 4.7 / 8.3 / 11.8 / 20.8 on the GEMM path), its lead shrinking to 11 % at
# 120 rows; the cap is the largest size measured -- where the two paths cross above it is not measured
STYLES_SKINNY_MAX_ROWS = [120]


def _session(dec, n_img, k, mode, start_token, end_token):
    cache = dec.__dict__.setdefault("_decode_sessions", {})
    key = (n_img, k, mode, start_token, end_token, dec.precision)
    sess = cache.get(key)
    if sess is None or sess.arena_version != dec.arena().version:
        if len(cache) > 8:
            cache.clear()
        sess = _DecodeSession(dec, n_img, k, mode, start_token, end_token)
        cache[key] = sess
    return sess


@torch.no_grad()
def beam_sample(dec, features, start_token, end_token, k, mode, feed_image, sync_every=4, use_graph=None):
    """Returns a list of LongTensor [1, L_i] (one per image; the reference handles one image per call).
    ``features``: [n_img, E] (or [n_img, 1, E]); rows are independent images.
    ``use_graph`` (default: fp32 mode): steps >= 2 replay one captured CUDA graph of the decode step.
    ``mode`` a list / tuple of n_img style names (factored decoders): image i in style mode[i], one beam search over
    the images grouped by style, results in input order."""
    emb = dec._emb()
    E = emb.weight.shape[1]
    dev = emb.weight.device
    if isinstance(mode, (list, tuple)) and not isinstance(mode, StyleGroups):
        from .decoders import STYLES
        groups, order = group_styles(mode, features.numel() // E, STYLES)
        feats = features.detach().to(dev).float().reshape(-1, E)
        feats = feats.index_select(0, torch.tensor(order, dtype=torch.long, device=dev))
        res = beam_sample(dec, feats, start_token, end_token, k, groups, feed_image, sync_every, use_graph)
        return ungroup(res, order)
    ops.lib()
    dec.arena()
    feats = features.detach().to(dev).float().reshape(-1, E)
    n_img = feats.shape[0]
    sess = _session(dec, n_img, k, mode, start_token, end_token)
    st = sess.st
    sess.calls += 1
    if sess.skinny:
        # few rows: matrix-vector kernels on the fp32 weights (both precision modes), steps 2.. replayed 4 at a time
        if use_graph is None:
            use_graph = True

        def restart_eager():
            st.reset()
            sess.h.zero_()
            sess.c.zero_()
            sess.flip = 0
            sess.step_skinny(1, feed_image, device_step=True)       # step 1 is special (image feed, one live row)

        def restart():
            # reset + step 1 are ~15 small launches: replayed as one graph per feed_image once the session is warm
            g0 = sess.__dict__.setdefault("graph0", {}).get(bool(feed_image))
            if g0 is None and use_graph and sess.graph is not None:
                s0 = torch.cuda.Stream()
                s0.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(s0):
                    restart_eager()
                torch.cuda.current_stream().wait_stream(s0)
                torch.cuda.synchronize()
                g0 = torch.cuda.CUDAGraph()
                with ops.no_gc_during_capture(), torch.cuda.graph(g0):
                    restart_eager()
                sess.graph0[bool(feed_image)] = g0
            if g0 is not None:
                g0.replay()
                sess.flip = 1
            else:
                restart_eager()
        sess.feats.copy_(feats)
        if sess.groups is not None:
            for l in range(sess.L):
                dec._collapse_styles(sess.ctx, sess.groups.styles, l)    # one Wc / bc per style, this call's weights
        elif COLLAPSE_CHAIN[0] and hasattr(dec, "_collapse_chain"):
            # inference: U_g S_g V_g of this mode as one matrix per gate, refreshed once per call (the weights may have
            # been trained since the last one) -- a decode step is then ONE kernel in front of the vocabulary projection
            for l in range(sess.L):
                dec._collapse_chain(sess.ctx, mode, l)
        restart()
        if use_graph and sess.graph is None and sess.calls >= 2:
            sess.capture_skinny()                                    # (runs throw-away steps: start over)
            restart()
        step = 2
        while step <= dec.max_seq_length + 1:
            if use_graph and sess.graph is not None:
                sess.graph.replay()
                step += sess.STEPS_PER_GRAPH
            else:
                for _ in range(sess.STEPS_PER_GRAPH):
                    sess.step_skinny(step, False, device_step=True)
                    step += 1
            if int(st.n_unfinished.item()) == 0:
                break
        return st.results()
    if use_graph is None:
        use_graph = not dec.bf16           # bf16 mode refreshes weight shadows per call: stays eager
    if use_graph and sess.graph is None and sess.calls >= 2:
        sess.capture()                      # first call runs eagerly (and warms everything up)
    st.reset()
    sess.h.zero_()
    sess.c.zero_()
    sess.feats.copy_(feats)
    sess.cache.clear()
    sess.ctx.w16 = {}
    sess.__dict__.pop("_w16_layers", None)
    for gcs in sess.__dict__.get("gctx", ()):
        for gc in gcs:
            gc.w16 = {}
    graph = sess.graph if use_graph else None
    for step in range(1, dec.max_seq_length + 2):
        if graph is not None and step >= 2:
            graph.replay()
        else:
            sess.step(step, feed_image, device_step=True)
        if sync_every and step % sync_every == 0 and int(st.n_unfinished.item()) == 0:
            break
    return st.results()


@torch.no_grad()
def sample_decode(dec, features, start_token, end_token, n, mode, temperature, seed, greedy, sync_every=4):
    """Sampling decode (``sample_captions``): n samples per row of ``features [n_img, E]`` on a ``_DecodeSession`` with a
    ``SampleState``.  Step 0 feeds the image and discards its output, step 1 feeds <start>, step t the token drawn at
    step t - 1 -- the conditioning of the teacher-forced ``forward_loss(captions, lengths, features)``.  Returns the
    device tensors (seqs int64 [R, max_len + 2], lengths int64 [R], logprob float32 [R, max_len + 1])."""
    emb = dec._emb()
    E = emb.weight.shape[1]
    dev = emb.weight.device
    ops.lib()
    dec.arena()
    feats = features.detach().to(dev).float().reshape(-1, E)
    n_img = feats.shape[0]
    cache = dec.__dict__.setdefault("_decode_sessions", {})
    key = ("sample", n_img, n, mode, start_token, end_token, dec.precision, float(temperature), bool(greedy))
    sess = cache.get(key)
    if sess is None or sess.arena_version != dec.arena().version:
        if len(cache) > 8:
            cache.clear()
        st = SampleState(n_img, n, dec.max_seq_length, start_token, temperature, greedy, dev)
        sess = cache[key] = _DecodeSession(dec, n_img, n, mode, start_token, end_token, state=st)
    st = sess.st
    sess.calls += 1
    st.seed_dev.fill_(seed)
    sess.feats.copy_(feats)
    last = dec.max_seq_length + 1
    if sess.skinny:
        if COLLAPSE_CHAIN[0] and hasattr(dec, "_collapse_chain"):
            for l in range(sess.L):
                dec._collapse_chain(sess.ctx, mode, l)

        def restart_eager():
            st.reset()
            sess.h.zero_()
            sess.c.zero_()
            sess.flip = 0
            sess.step_skinny(1, True, True, draw=False)             # step 0: the image, output discarded
            sess.step_skinny(1, False, True)                        # step 1: <start>, the first draw

        def restart():
            g0 = sess.__dict__.get("graph0_sample")
            if g0 is None and sess.graph is not None:
                s0 = torch.cuda.Stream()
                s0.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(s0):
                    restart_eager()
                torch.cuda.current_stream().wait_stream(s0)
                torch.cuda.synchronize()
                g0 = torch.cuda.CUDAGraph()
                with ops.no_gc_during_capture(), torch.cuda.graph(g0):
                    restart_eager()
                sess.graph0_sample = g0
            if g0 is not None:
                g0.replay()
                sess.flip = 0
            else:
                restart_eager()
        restart()
        if sess.graph is None and sess.calls >= 2:
            sess.capture_skinny()                                    # (runs throw-away steps: start over)
            restart()
        step = 2
        while step <= last:
            if sess.graph is not None:
                sess.graph.replay()
                step += sess.STEPS_PER_GRAPH
            else:
                for _ in range(sess.STEPS_PER_GRAPH):
                    sess.step_skinny(step, False, device_step=True)
                    step += 1
            if int(st.n_unfinished.item()) == 0:
                break
        return st.results()
    use_graph = not dec.bf16           # bf16 mode refreshes weight shadows per call: stays eager
    if use_graph and sess.graph is None and sess.calls >= 2:
        sess.capture()
    st.reset()
    sess.h.zero_()
    sess.c.zero_()
    sess.cache.clear()
    sess.ctx.w16 = {}
    sess.__dict__.pop("_w16_layers", None)
    sess.step(1, True, True, draw=False)                             # step 0: the image, output discarded
    graph = sess.graph if use_graph else None
    for step in range(1, last + 1):
        if graph is not None and step >= 2:
            graph.replay()
        else:
            sess.step(step, False, device_step=True)
        if sync_every and step % sync_every == 0 and int(st.n_unfinished.item()) == 0:
            break
    return st.results()


@torch.no_grad()
def beam_sample_att(dec, features, start_token, end_token, k, mode, sync_every=4):
    """Attention beam search (stylenet/model_att.py:307-426) for n_img images: features
    [n_img, S, S, D] (or [n_img, P, D]).  The feature map and the hoisted att1 are stored once per image;
    live beams index them through ``row_img`` instead of expanding them k times.
    ``mode`` a list / tuple of n_img style names: image i in style mode[i].  The images are grouped by style; per group
    the hoisted att1 comes from that style's encoder_att, and each step runs its decoder_att, the attention step and
    the style's input projection on the group's rows, while f_beta, the recurrence and C run once over all rows."""
    emb = dec._emb()
    E = emb.weight.shape[1]
    dev = emb.weight.device
    D, A, H = dec.feature_size, dec.attention_size, dec.hidden_size
    order = None
    if isinstance(mode, (list, tuple)):
        from .decoders import STYLES
        n_in = features.shape[0] if features.dim() >= 3 else 1
        groups, order = group_styles(mode, n_in, STYLES)
        styles, counts = groups.styles, groups.counts
    ops.lib()
    dec.arena()
    feats = features.detach().to(dev).float()
    n_img = feats.shape[0] if feats.dim() >= 3 else 1
    feats = feats.reshape(n_img, -1, D).contiguous()
    if order is not None:
        feats = feats.index_select(0, torch.tensor(order, dtype=torch.long, device=dev))
    else:
        styles, counts = (mode,), (n_img,)
    G = len(styles)
    # group g: images [img_off[g], img_off[g+1]), rows [k * img_off[g], k * img_off[g+1])
    img_off = [0]
    for n in counts:
        img_off.append(img_off[-1] + n)
    P = feats.shape[1]
    atts = [dec._att_module(s) for s in styles]
    st = BeamState(n_img, k, dec.max_seq_length, start_token, dev)
    R = st.R
    f32 = dict(dtype=torch.float32, device=dev)
    h0, c0 = dec.init_hidden_state(feats)
    h = h0.repeat_interleave(k, 0).contiguous()
    c = c0.repeat_interleave(k, 0).contiguous()
    att1 = torch.empty(n_img * P, A, **f32)
    for g, att in enumerate(atts):
        i0, i1 = img_off[g], img_off[g + 1]
        ops.linear_nt(feats[i0:i1].view((i1 - i0) * P, D), att.encoder_att.weight, att.encoder_att.bias,
                      out=att1[i0 * P:i1 * P])
    # per-row views of the per-image tensors (beams of one image share its rows)
    feats_r = feats.repeat_interleave(k, 0).contiguous()
    att1_r = att1.view(n_img, P, A).repeat_interleave(k, 0).contiguous()
    h_new = torch.empty_like(h)
    out = dec._out()
    V = out.weight.shape[0]
    logits = torch.empty(R, V, **f32)
    X = torch.empty(R, E + D, **f32)
    att2 = torch.empty(R, A, **f32)
    gate_pre = torch.empty(R, D, **f32)
    alpha = torch.empty(R, P, **f32)
    ctx = _StepCtx()
    ctx.XP = torch.empty(R, 4 * H, **f32)
    gctx = []
    for g in range(G):
        gc = _StepCtx()
        gc.XP = ctx.XP[k * img_off[g]:k * img_off[g + 1]]
        gctx.append(gc)
    row_img = torch.zeros(R, dtype=torch.int32, device=dev)
    dummy_cap = torch.zeros(1, 1, dtype=torch.int64, device=dev)
    bs1, off1 = _i32(dev, [R]), _i32(dev, [0])
    Whh, bhh = dec._recurrent_weights()
    wfull = [att.full_att.weight.view(-1) for att in atts]
    for step in range(1, dec.max_seq_length + 2):
        ops.gather_pack_fwd(dummy_cap, emb.weight, None, False, row_img, row_img, st.prev_word, R, X, 0.0, 0)
        for g, att in enumerate(atts):
            r0, r1 = k * img_off[g], k * img_off[g + 1]
            ops.gemm(ops.OP_NT, h[r0:r1], att.decoder_att.weight, att2[r0:r1], r1 - r0, A, H, H, H, A,
                     bias=att.decoder_att.bias)
        ops.gemm(ops.OP_NT, h, dec.f_beta.weight, gate_pre, R, D, H, H, H, D, bias=dec.f_beta.bias)
        for g in range(G):
            r0, r1 = k * img_off[g], k * img_off[g + 1]
            ops.att_step_fwd(att1_r[r0:r1], att2[r0:r1], feats_r[r0:r1], wfull[g], 0.0, gate_pre[r0:r1], r1 - r0, P, A,
                             D, alpha[r0:r1], P, X[r0:r1, E:], E + D)
        if G == 1:
            dec._input_projection(ctx, X, styles[0], 0, R)
        else:
            for g in range(G):
                r0, r1 = k * img_off[g], k * img_off[g + 1]
                dec._input_projection(gctx[g], X[r0:r1], styles[g], 0, r1 - r0)
        ops.recur_fwd(dec.cell, H, R, bs1, off1, 0, 1, ctx.XP, Whh, bhh, h, h_new, None, None, None, c)
        ops.gemm(ops.OP_NT, h_new, out.weight, logits, R, V, H, H, H, V, bias=out.bias)
        st.step(logits, step, end_token)
        idx = st.src_row.long()
        h = h_new.index_select(0, idx)
        c = c.index_select(0, idx)
        if sync_every and step % sync_every == 0 and int(st.n_unfinished.item()) == 0:
            break
    res = st.results()
    return res if order is None else ungroup(res, order)
