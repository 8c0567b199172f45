"""Batch-sharded data parallelism over the GPUs of one box (SURVEY.md section 8e): one process per GPU,
weights / Adam states / teacher-forcing coins replicated, samples sharded after the length sort, and ONE
exchange step -- a SUM all-reduce (NCCL over NVLink/NVSwitch) of the flat gradient-arena ranges that
received a gradient this step, issued in two buckets as backward produces them so the first (the
vocabulary projection, 1/3 of the bytes) overlaps the reverse-time recurrence:
    bucket 0: C.weight, C.bias          ready right after the vocab-projection backward
    bucket 1: everything else active    ready after the sequence backward
Each rank scales its gradients by 1/N_global tokens (not 1/N_local) so the SUM equals the single-GPU
gradient of the token-mean loss even with ragged shards.  The reference has no distributed code at all.
"""
import os
import re

import torch
import torch.distributed as dist

from . import ops


def merged_ranges(arena, names, max_gap=64):
    """Flat (offset, length) ranges covering ``names`` in the arena, merged across alignment padding."""
    spans = sorted((arena.offset[n], arena.numel[n]) for n in names)
    out = []
    for o, n in spans:
        if out and o - (out[-1][0] + out[-1][1]) < max_gap:
            out[-1] = (out[-1][0], o + n - out[-1][0])
        else:
            out.append((o, n))
    return out


class GradSync:
    """Asynchronous SUM all-reduce of flat ranges of one buffer; ``wait()`` joins the current stream."""

    def __init__(self, group=None):
        self.group = group
        self.pending = []
        self.bytes = 0

    def launch(self, flat, ranges):
        if not dist.is_initialized() or dist.get_world_size(self.group) == 1:
            return                      # single process: nothing to exchange
        for o, n in ranges:
            w = dist.all_reduce(flat[o:o + n], op=dist.ReduceOp.SUM, group=self.group, async_op=True)
            self.pending.append(w)
            self.bytes += 4 * n

    def wait(self):
        for w in self.pending:
            w.wait()
        self.pending = []


class PeerExchange:
    """NVLink peer-memory view of every rank's parameter arena, gradient arena and signal pad: each rank exports
    CUDA IPC handles of the three buffers (exchanged once through torch.distributed), and opens its peers' with
    its own device current, which yields peer mappings its kernels can load from / store to over NVLink.
    Feeds sn_dp_adam_fused: ONE kernel per step does reduce-scatter + clamp/Adam + all-gather, no NCCL."""

    _opened = {}        # handle bytes -> mapped base address (an allocation can be opened once per process)
    N_PADS = 16         # exchange calls of one step that may be in flight at the same time (one pad each)

    def pads(self, bucket):
        """Signal-pad pointers (one per rank) of bucket ``bucket``: concurrent exchange kernels on different streams
        must not share flags."""
        if not 0 <= bucket < self.N_PADS:
            raise RuntimeError("too many exchange buckets in one step")
        return [p + 128 * bucket for p in self.pad_ptrs]

    def __init__(self, arena, group=None, grad_dtype=None):
        from . import ops
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        if self.world > 8:
            raise RuntimeError("peer exchange supports one NVSwitch box (<= 8 ranks)")
        dev = arena.flat.device
        self.pad = torch.zeros(32 * self.N_PADS, dtype=torch.int32, device=dev)   # one signal pad per concurrent bucket
        # push form: receive buffer = `world` slots (one per sender) of this rank's share of the arena
        grad_dtype = grad_dtype or torch.float32
        self.elem_size = 2 if grad_dtype == torch.bfloat16 else 4
        self.slot_elems = ops.dp_slot_elems(arena.flat.numel(), self.world)
        self.recv = torch.zeros(self.world * self.slot_elems, dtype=grad_dtype, device=dev)
        torch.cuda.synchronize()
        mine = [ops.ipc_export(t) for t in (arena.flat, arena.gflat, self.pad, self.recv)]
        gathered = [None] * self.world
        dist.all_gather_object(gathered, (self.rank, dev.index, mine), group=group)
        self.param_ptrs, self.grad_ptrs, self.pad_ptrs = [0] * self.world, [0] * self.world, [0] * self.world
        self.recv_ptrs = [0] * self.world
        for r, dev_index, exports in gathered:
            if r == self.rank:
                ptrs = [t.data_ptr() for t in (arena.flat, arena.gflat, self.pad, self.recv)]
            else:
                ops.enable_peer_access(dev_index)
                ptrs = []
                for handle, offset in exports:
                    base = PeerExchange._opened.get(handle)
                    if base is None:
                        base = ops.ipc_open(handle)
                        PeerExchange._opened[handle] = base
                    ptrs.append(base + offset)
            self.param_ptrs[r], self.grad_ptrs[r], self.pad_ptrs[r], self.recv_ptrs[r] = ptrs
        self.arena_version = arena.version
        self.keep = (arena.flat, arena.gflat, self.pad, self.recv)      # exported memory must stay allocated
        torch.cuda.synchronize()
        dist.barrier(group=group)


EARLY_PEER_EXCHANGE = [True]     # split the peer-fused exchange+Adam: vocabulary projection early, the rest at the end
PEER_FORM = [os.environ.get("SN_DP_FORM", "push")]     # "push": sn_dp_push + sn_dp_adam_recv; "pull": sn_dp_adam_fused (peer loads)
BG_PUSH_SMS = [int(os.environ.get("SN_DP_BG_PUSH_SMS", "16"))]     # grid cap of a push that runs under the backward (0 = whole GPU)
BG_RECV_CTAS = [int(os.environ.get("SN_DP_BG_RECV_CTAS", "0"))]    # same for its receive side (512-thread CTAs)
BG_WU = [os.environ.get("SN_DP_BG_WU", "0") == "1"]              # exchange the W_hh / U bucket in the background too
PEER_BUCKETS = [False]           # also exchange the W_hh/U, S/V and embedding buckets as soon as they are final (slower: see step())


def tail_schedule(world, bucketed):
    """Whether a training step takes the tail schedule of ops.TAIL_SCHEDULE: single GPU, bucketed (bf16, no attention)
    step, and the switch on.  The data-parallel exchange paths keep theirs."""
    return bool(ops.TAIL_SCHEDULE[0]) and world == 1 and bool(bucketed)


class DataParallelTrainer:
    """forward -> loss -> backward -> gradient exchange -> fused clamp+Adam, one rank per GPU.

    comm="peer" (default when world > 1 on CUDA): the exchange and the optimizer are ONE kernel over NVLink peer
    memory (sn_dp_adam_fused: reduce-scatter by peer loads, Adam on the owned shard, all-gather by peer stores).
    comm="nccl": bucketed NCCL SUM all-reduce (bucket 0 overlapped with the recurrence backward) + local Adam."""

    def __init__(self, decoder, optimizer, group=None, comm=None):
        self.decoder, self.optimizer = decoder, optimizer
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.sync = GradSync(group)
        if comm is None:
            comm = "peer" if (self.world > 1 and dist.get_backend(group) == "nccl") else "nccl"
        self.comm = comm
        self.peers = None

    def _peers(self):
        a = self.decoder.arena()
        # gradient transport of the push form: fp32 (the N-GPU step then differs from the 1-GPU step by the summation
        # order only).  SN_DP_GRAD_BF16=1 sends bf16 and accumulates in fp32 at the owner -- half the bytes, but Adam's
        # normalisation turns the rounding of near-zero gradients into full-size steps: 2.5e-2 relative parameter
        # difference vs 1 GPU after 3 steps in bf16 mode instead of 4e-4 (bench.py dp_parity, N=2), so it is opt-in
        dt = torch.bfloat16 if os.environ.get("SN_DP_GRAD_BF16") == "1" else torch.float32
        if self.peers is None or self.peers.arena_version != a.version or self.peers.recv.dtype != dt:
            self.peers = PeerExchange(a, self.group, grad_dtype=dt)
        return self.peers

    def _step_push(self, captions, lengths, features, n_global, b_global, bucketed, kw):
        """Peer exchange, push form: every gradient bucket is SENT to the chunk owners (sn_dp_push: posted NVLink stores,
        nothing waits) on the stream that produced it as soon as it is final, so only the last bucket's transfer is left
        at the end of the step; the vocabulary projection's reduce + Adam + parameter all-gather (sn_dp_adam_recv) also
        runs early, under the reverse recurrence, the other buckets' in ONE call at the end."""
        peers = self._peers()
        opt = self.optimizer
        done = []            # names whose parameters are already updated
        if bucketed:
            out_names = set(self.decoder._out_names())
            calls = [0]

            def early_step(names):
                # buckets that are final well before the end of the backward -- the vocabulary projection (41 % of the
                # arena at configs[1]; final before the reverse recurrence) and, optionally, W_hh / U (final right after
                # it) -- are exchanged in the BACKGROUND on their own side stream (the producing streams go on with the
                # weight-gradient GEMMs).  The push is bound by the link, not by the SMs: it gets BG_PUSH_SMS CTAs so
                # that the projection-backward GEMMs keep theirs; the receive side is Adam traffic (36 B per element) and
                # runs full width.  S / V and the embedding become final within the last ~20 us: they travel together in
                # one full-width exchange at the end.
                is_out = out_names.issuperset(names)
                is_wu = BG_WU[0] and bool(names) and all(re.match(r"(l\d+_)?[WU]_", n) for n in names)
                if not (is_out or is_wu) or calls[0] >= PeerExchange.N_PADS - 1:
                    return
                b = calls[0]
                bg = self.decoder._side(3)
                bg.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(bg):
                    if opt.push_peer(peers, only=names, bucket=b, max_ctas=BG_PUSH_SMS[0]):
                        opt.step_peer_recv(peers, [b], only=names, max_ctas=BG_RECV_CTAS[0])
                        calls[0] += 1
                        done.extend(names)
            kw = dict(kw, early_step=early_step)
        loss, stats = self.forward_backward(captions, lengths, features, n_global=n_global, b_global=b_global, **kw)
        last = PeerExchange.N_PADS - 1
        if opt.push_peer(peers, skip=done or None, bucket=last):
            opt.step_peer_recv(peers, [last], skip=done or None)
        return loss, stats

    def forward_backward(self, captions, lengths, features, n_global=None, b_global=None, grad_hook=None, **kw):
        """zero_grad + forward + loss + backward with gradients scaled by 1/N_global; ``grad_hook(names)`` is
        called when a bucket of gradients is final."""
        dec = self.decoder
        a = dec.arena()
        N_local = sum(int(l) for l in lengths)
        if n_global is None:
            n_global = N_local * self.world
        for p in a.named.values():
            p.grad = None
        extra = {}
        if b_global is not None or hasattr(dec, "attention"):
            extra["b_global"] = b_global if b_global is not None else len(lengths) * self.world
        return dec.forward_loss(captions, lengths, features, n_global=n_global, grad_hook=grad_hook, **extra, **kw)

    def step(self, captions, lengths, features, n_global=None, b_global=None, **kw):
        a = self.decoder.arena()
        bucketed = getattr(self.decoder, "bf16", False) and not hasattr(self.decoder, "attention") and EARLY_PEER_EXCHANGE[0]
        if self.world > 1 and self.comm == "peer" and PEER_FORM[0] == "push":
            return self._step_push(captions, lengths, features, n_global, b_global, bucketed, kw)
        if self.world > 1 and self.comm == "peer":
            peers = self._peers()
            early = []
            if bucketed:
                # gradient buckets are exchanged (reduce-scatter + Adam + all-gather, one kernel) on the side stream that
                # produced them AS SOON AS THEY ARE FINAL: the vocabulary projection under the reverse recurrence, W_hh / U
                # and S / V under the rest of the projection backward; only the embedding is left for the end of the step.
                # Every bucket has its own signal pad (the kernels overlap each other).
                calls = [0]
                out_names = set(self.decoder._out_names())

                def early_step(names):
                    # every exchange kernel costs two cross-GPU barriers plus the skew between the ranks (~50 us measured
                    # at N=2, profiles/r2_timeline_N2.txt): only the large vocabulary bucket, which has the whole reverse
                    # recurrence + projection backward to hide under, goes early; everything else is ONE call at the end
                    if not PEER_BUCKETS[0] and not out_names.issuperset(names):
                        return
                    self.optimizer.step_peer(peers, only=names, bucket=calls[0])
                    calls[0] += 1
                    early.extend(names)
                kw = dict(kw, early_step=early_step)
            loss, stats = self.forward_backward(captions, lengths, features, n_global=n_global, b_global=b_global, **kw)
            self.optimizer.step_peer(peers, skip=early or None, bucket=PeerExchange.N_PADS - 1)
            return loss, stats
        hook = None
        if self.world > 1:
            def hook(names):
                self.sync.launch(a.gflat, merged_ranges(a, names))
        early = []
        if self.world == 1 and bucketed:
            # single GPU: Adam of each bucket runs on the side stream that produced it (under the reverse recurrence /
            # the projection backward); the rest follows at the end
            tail = tail_schedule(self.world, bucketed)
            emb = getattr(self.decoder, "_emb_name", lambda: None)()

            def early_step(names):
                # the vocabulary, W_hh / U and S / V buckets run next to the dZ -> dA2 -> dA1 -> dX chain: their grid can
                # be capped (ops.ADAM_BG_CTAS; full width measured fastest).  The embedding bucket ends the step: full width
                cap = ops.ADAM_BG_CTAS[0] if (tail and list(names) != [emb]) else 0
                self.optimizer.step(only=names, max_ctas=cap)
                early.extend(names)
            kw = dict(kw, early_step=early_step, early_embed=tail)
        loss, stats = self.forward_backward(captions, lengths, features, n_global=n_global, b_global=b_global,
                                            grad_hook=hook, **kw)
        if self.world > 1:
            self.sync.wait()
        self.optimizer.step(skip=early or None)
        return loss, stats
