"""Fused clamp + Adam (K7): utils.clip_gradient (stylenet/utils.py:51-60) followed by
torch.optim.Adam.step (stylenet/train_multitask.py:388-389) as ONE kernel over the flat arena ranges that
received a gradient this step.  Several optimizer objects may share the same parameters, each with its own
moments and step counts (the reference keeps ``optimizer`` and ``lang_optimizer`` over the same decoder,
train_multitask.py:163-167); parameters whose grad is None are skipped exactly like torch.optim.Adam.

Per-parameter step counters and the learning rate live in DEVICE memory (a prologue kernel bumps the counters
and derives the bias corrections in double precision), so ``step()`` has no host-dependent kernel arguments
and a whole training step can be captured in / replayed from a CUDA graph."""
import torch

from . import ops


class FusedClampAdam:
    def __init__(self, decoder, lr=2e-4, betas=(0.9, 0.999), eps=1e-8, grad_clip=0.5, extra_params=()):
        self.decoder = decoder
        self.betas, self.eps, self.grad_clip = betas, float(eps), float(grad_clip)
        self.param_groups = [{"lr": float(lr), "params": list(decoder.parameters()) + list(extra_params)}]
        self._arena_version = -1
        self.m = self.v = None
        self.extra = list(extra_params)       # e.g. encoder.linear / encoder.bn parameters
        self.extra_state = {}
        self._lr_on_device = None

    # -- state -----------------------------------------------------------------------------------------
    def _state(self):
        a = self.decoder.arena()
        if self._arena_version != a.version or self.m is None:
            dev = a.flat.device
            names = list(a.named)
            if self.m is not None and self.m.numel() == a.total and getattr(self, "names", None) == names:
                # the arena was re-bound (.to() / .cuda(), an un-pickled checkpoint, a replaced Parameter): the layout
                # is a pure function of the parameter shapes, so moments and step counters carry over
                self.m, self.v = self.m.to(dev), self.v.to(dev)
                self.steps_dev = self.steps_dev.to(dev)
            else:
                self.m = torch.zeros_like(a.flat)
                self.v = torch.zeros_like(a.flat)
                self.steps_dev = torch.zeros(len(names), dtype=torch.int32, device=dev)
            self.names = names
            self.index = {n: i for i, n in enumerate(self.names)}
            self.lr_dev = torch.zeros(1, dtype=torch.float32, device=dev)
            self.coef_ws = torch.zeros(2 * len(self.names) + 2, dtype=torch.float32, device=dev)
            self._lr_on_device = None
            self._arena_version = a.version
        return a

    def _sync_lr(self):
        lr = float(self.param_groups[0]["lr"])
        if self._lr_on_device != lr:       # adjust_learning_rate (utils.py:116-124) mutates param_groups
            self.lr_dev.fill_(lr)
            self._lr_on_device = lr

    def step_counts(self):
        """{parameter name: number of Adam steps taken} (device counters, copied to the host)."""
        self._state()
        return dict(zip(self.names, self.steps_dev.tolist()))

    def zero_grad(self):
        for p in self.param_groups[0]["params"]:
            p.grad = None

    # -- checkpointing -----------------------------------------------------------------------------------
    def __getstate__(self):
        """Whole-object pickling (the reference's save_checkpoint pickles optimizers, stylenet/utils.py:62-90)."""
        st = self.__dict__.copy()
        st["_lr_on_device"] = None
        return st

    def state_dict(self):
        """torch.optim.Adam's schema: {"state": {i: {"step", "exp_avg", "exp_avg_sq"}}, "param_groups": [...]} with i
        the position in ``param_groups[0]["params"]``; only parameters that took at least one step have state.
        Under the peer-fused data-parallel step each rank holds the moments of the chunks it owns only (ZeRO-1
        style, ownership = (arena offset / 4096) % world): all-reduce ``m`` / ``v`` (SUM) before saving there."""
        a = self._state()
        params = self.param_groups[0]["params"]
        by_id = {id(p): n for n, p in a.named.items()}
        steps = self.steps_dev.tolist()
        state = {}
        for i, p in enumerate(params):
            n = by_id.get(id(p))
            if n is not None:
                st = self.extra_state.get(("arena", n))
                if st is not None and int(st["step"].item()) > 0:      # stepped through a foreign gradient tensor
                    state[i] = {"step": st["step"].float().reshape(()).clone(), "exp_avg": st["m"].clone(),
                                "exp_avg_sq": st["v"].clone()}
                elif steps[self.index[n]] > 0:
                    o, k = a.offset[n], a.numel[n]
                    state[i] = {"step": torch.tensor(float(steps[self.index[n]])),
                                "exp_avg": self.m[o:o + k].view(p.shape).clone(),
                                "exp_avg_sq": self.v[o:o + k].view(p.shape).clone()}
        for j, p in enumerate(self.extra):
            st = self.extra_state.get(("extra", j))
            if st is not None and int(st["step"].item()) > 0:
                state[len(params) - len(self.extra) + j] = {
                    "step": st["step"].float().reshape(()).clone(), "exp_avg": st["m"].clone(), "exp_avg_sq": st["v"].clone()}
        group = {"lr": self.param_groups[0]["lr"], "betas": tuple(self.betas), "eps": self.eps, "weight_decay": 0,
                 "amsgrad": False, "grad_clip": self.grad_clip, "params": list(range(len(params)))}
        return {"state": state, "param_groups": [group]}

    def load_state_dict(self, sd):
        a = self._state()
        params = self.param_groups[0]["params"]
        group = sd["param_groups"][0]
        if len(group["params"]) != len(params):
            raise ValueError("loaded state dict has a different number of parameters")
        self.param_groups[0]["lr"] = float(group["lr"])
        self.betas, self.eps = tuple(group.get("betas", self.betas)), float(group.get("eps", self.eps))
        by_id = {id(p): n for n, p in a.named.items()}
        self.m.zero_(); self.v.zero_(); self.steps_dev.zero_()
        self.extra_state = {}
        steps = [0] * len(self.names)
        for i, st in sd["state"].items():
            p = params[int(i)]
            n = by_id.get(id(p))
            if n is not None:
                o, k = a.offset[n], a.numel[n]
                self.m[o:o + k].copy_(st["exp_avg"].reshape(-1))
                self.v[o:o + k].copy_(st["exp_avg_sq"].reshape(-1))
                steps[self.index[n]] = int(float(st["step"]))
            else:
                j = int(i) - (len(params) - len(self.extra))
                self.extra_state[("extra", j)] = {
                    "m": st["exp_avg"].to(p.device).clone(), "v": st["exp_avg_sq"].to(p.device).clone(),
                    "step": torch.full((1,), int(float(st["step"])), dtype=torch.int32, device=p.device),
                    "coef": torch.zeros(2, dtype=torch.float32, device=p.device)}
        self.steps_dev.copy_(torch.tensor(steps, dtype=torch.int32))
        self._lr_on_device = None

    # -- step ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def step(self, only=None, skip=None, max_ctas=0):
        """``only`` / ``skip``: parameter names to restrict the step to / leave out.  A training step may update the
        vocabulary projection (43 % of the Adam traffic at configs[1]) on a side stream as soon as its gradient is
        final, under the reverse recurrence, and finish with ``step(skip=...)`` -- per-parameter step counters make
        the two calls equivalent to one.  ``max_ctas`` > 0 caps the grid of the arena ranges' kernel (a bucket updated
        next to the critical chain); it changes no result."""
        a = self._state()
        self._sync_lr()
        items, foreign = a.grad_ranges()
        if only is not None:
            keep = set(only)
            items = [it for it in items if it[2] in keep]
            foreign = [n for n in foreign if n in keep]
        if skip is not None:
            drop = set(skip)
            items = [it for it in items if it[2] not in drop]
            foreign = [n for n in foreign if n not in drop]
        b1, b2 = self.betas
        ranges = [(off, n) for off, n, _ in items]
        idx = [self.index[name] for _, _, name in items]
        a.kernel_epoch += 1
        ops.adam_clamp_dev(a.flat, a.gflat, self.m, self.v, ranges, idx, self.steps_dev, self.lr_dev, self.coef_ws,
                           b1, b2, self.eps, self.grad_clip, max_ctas=max_ctas)
        # parameters outside the arena (foreign gradient tensors, extra params): same kernel, one range each
        for name in foreign:
            self._step_tensor(a.named[name], ("arena", name))
        if only is None:
            for i, p in enumerate(self.extra):
                if p.grad is not None:
                    self._step_tensor(p, ("extra", i))

    @torch.no_grad()
    def step_peer(self, peers, only=None, skip=None, bucket=0):
        """Data-parallel step: gradient reduce-scatter + clamp/Adam on the owned shard + parameter all-gather in
        one kernel over NVLink peer memory.  Every rank must call it with the same set of gradients (``only`` /
        ``skip`` as in ``step``: the vocabulary projection's exchange can run early, under the reverse recurrence)."""
        a = self._state()
        self._sync_lr()
        items, foreign = a.grad_ranges()
        if only is not None:
            keep = set(only)
            items = [it for it in items if it[2] in keep]
        if skip is not None:
            drop = set(skip)
            items = [it for it in items if it[2] not in drop]
        if foreign or any(p.grad is not None for p in self.extra):
            raise RuntimeError("peer-fused step needs every gradient in the arena")
        ranges = [(off, n) for off, n, _ in items]
        idx = [self.index[name] for _, _, name in items]
        if not ranges:
            return          # every bucket was exchanged early (the same on every rank): no empty barrier-only call
        a.kernel_epoch += 1
        ops.dp_adam_fused(peers.world, peers.rank, peers.grad_ptrs, peers.param_ptrs, peers.pads(bucket), self.m, self.v,
                          ranges, idx, self.steps_dev, self.lr_dev, self.coef_ws, self.betas[0], self.betas[1],
                          self.eps, self.grad_clip)

    def _peer_items(self, only, skip):
        a = self._state()
        items, foreign = a.grad_ranges()
        if only is not None:
            keep = set(only)
            items = [it for it in items if it[2] in keep]
        if skip is not None:
            drop = set(skip)
            items = [it for it in items if it[2] not in drop]
        if foreign or any(p.grad is not None for p in self.extra):
            raise RuntimeError("peer-fused step needs every gradient in the arena")
        return a, items

    @torch.no_grad()
    def push_peer(self, peers, only=None, skip=None, bucket=0, max_ctas=0):
        """Push form, part 1: send this rank's gradients of ``only`` (minus ``skip``) to the chunk owners' receive buffers
        (non-blocking, on the current stream) and raise this bucket's ARRIVE flags.  Returns False when there was nothing
        to send (no call was made -- the same on every rank)."""
        a, items = self._peer_items(only, skip)
        if not items:
            return False
        ops.dp_push(peers.world, peers.rank, a.gflat, peers.recv_ptrs, peers.slot_elems, peers.elem_size,
                    peers.pads(bucket), [(off, n) for off, n, _ in items], max_ctas=max_ctas)
        return True

    @torch.no_grad()
    def step_peer_recv(self, peers, buckets, only=None, skip=None, max_ctas=0):
        """Push form, part 2: wait for the pushes of ``buckets`` (1..4 bucket ids whose gradients are exactly ``only`` minus
        ``skip``), reduce, clamp + Adam on the owned chunks, parameter all-gather, exit barrier.  As with ``step_peer``,
        ``p.grad`` keeps this rank's LOCAL, unclamped gradient afterwards (the reference's clip_gradient clamps in place,
        stylenet/utils.py:60; the summed, clamped gradient only ever exists in the owner's registers)."""
        a, items = self._peer_items(only, skip)
        self._sync_lr()
        if not items:
            if buckets:
                raise RuntimeError("step_peer_recv: pushed buckets without gradients")
            return
        ranges = [(off, n) for off, n, _ in items]
        idx = [self.index[name] for _, _, name in items]
        mine = [peers.pads(b)[peers.rank] for b in buckets]
        a.kernel_epoch += 1
        ops.dp_adam_recv(peers.world, peers.rank, a.gflat, peers.param_ptrs, peers.recv, peers.slot_elems,
                         peers.elem_size, peers.pads(buckets[0]), mine, self.m, self.v, ranges, idx, self.steps_dev,
                         self.lr_dev, self.coef_ws, self.betas[0], self.betas[1], self.eps, self.grad_clip,
                         max_ctas=max_ctas)

    def _step_tensor(self, p, key):
        st = self.extra_state.get(key)
        if st is None:
            st = {"m": torch.zeros_like(p.data), "v": torch.zeros_like(p.data),
                  "step": torch.zeros(1, dtype=torch.int32, device=p.device),
                  "coef": torch.zeros(2, dtype=torch.float32, device=p.device)}
            self.extra_state[key] = st
        if not p.data.is_contiguous():
            raise RuntimeError("non-contiguous parameter")
        g = p.grad.contiguous()
        ops.adam_clamp_dev(p.data.view(-1), g.view(-1), st["m"].view(-1), st["v"].view(-1), [(0, p.numel())], [0],
                           st["step"], self.lr_dev, st["coef"], self.betas[0], self.betas[1], self.eps,
                           self.grad_clip)
        if g.data_ptr() != p.grad.data_ptr():
            p.grad.copy_(g.view_as(p.grad))
