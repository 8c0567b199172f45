"""The tail schedule of the single-GPU bf16 training step (ops.TAIL_SCHEDULE) computes the same bits as the previous
one: the split embedding backward, the 16-byte column sums, the capped Adam grid, and whole training steps."""
import random

import pytest
import torch

pytestmark = pytest.mark.gpu


def _sn():
    import icei_b200 as sn
    from icei_b200 import ops
    return sn, ops


def _captions(B, T, V, seed, ragged):
    g = torch.Generator().manual_seed(seed)
    cap = torch.randint(4, V, (B, T), generator=g)
    cap[:, 0] = 1                     # <start>: a group of B rows, several 32-row chunks
    cap[: B // 2, 3] = 5              # a second multi-chunk group
    if ragged:
        lens = sorted((int(x) for x in torch.randint(2, T + 1, (B,), generator=g)), reverse=True)
        lens[0] = T
    else:
        lens = [T] * B
    return cap, lens


@pytest.mark.parametrize("p_drop", [0.0, 0.5])
@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("has_feat", [False, True])
@pytest.mark.parametrize("E", [300, 40])
def test_embed_plan_grad_equals_gather_pack_bwd(p_drop, ragged, has_feat, E):
    sn, ops = _sn()
    from icei_b200.packing import get_plan
    dev = torch.device("cuda", 0)
    B, T, V = 80, 12, 997
    cap, lens = _captions(B, T, V, 7, ragged)
    cap = cap.to(dev)
    plan = get_plan([l + 1 for l in lens] if has_feat else lens)
    d = plan.dev(dev)
    N = plan.N
    dX = torch.randn(N, E, device=dev)
    ref, new = torch.zeros(V, E, device=dev), torch.zeros(V, E, device=dev)
    fr = torch.empty(B, E, device=dev) if has_feat else None
    fn = torch.empty(B, E, device=dev) if has_feat else None
    seed_dev = torch.tensor([3], dtype=torch.int64, device=dev)
    ops.gather_pack_bwd(cap, ref, fr, has_feat, d["row_b"], d["row_t"], None, N, dX, p_drop, 11, seed_dev=seed_dev)
    ws = ops.embed_plan_ws(V, N, dev)
    ops.embed_plan(cap, has_feat, d["row_b"], d["row_t"], None, N, V, ws)
    ops.embed_grad(new, fn, has_feat, d["row_b"], d["row_t"], None, N, dX, p_drop, 11, ws, seed_dev=seed_dev, wide=True)
    torch.cuda.synchronize()
    assert torch.equal(ref, new)
    if has_feat:
        assert torch.equal(fr, fn)


def test_embed_grad_wide_with_override():
    """Fed-back tokens (tok_override >= 0) take no dropout: the wide group sums keep that too."""
    sn, ops = _sn()
    from icei_b200.packing import get_plan
    dev = torch.device("cuda", 0)
    B, T, V, E = 64, 10, 500, 300
    cap, lens = _captions(B, T, V, 3, False)
    cap = cap.to(dev)
    plan = get_plan(lens)
    d = plan.dev(dev)
    N = plan.N
    ov = torch.full((N,), -1, dtype=torch.int32, device=dev)
    ov[N // 2:] = torch.randint(0, 8, (N - N // 2,), dtype=torch.int32, device=dev)
    dX = torch.randn(N, E, device=dev)
    ref, new = torch.zeros(V, E, device=dev), torch.zeros(V, E, device=dev)
    ops.gather_pack_bwd(cap, ref, None, False, d["row_b"], d["row_t"], ov, N, dX, 0.5, 5)
    ws = ops.embed_plan_ws(V, N, dev)
    ops.embed_plan(cap, False, d["row_b"], d["row_t"], ov, N, V, ws)
    ops.embed_grad(new, None, False, d["row_b"], d["row_t"], ov, N, dX, 0.5, 5, ws, wide=True)
    torch.cuda.synchronize()
    assert torch.equal(ref, new)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("N", [10000, 2048, 300, 7])
@pytest.mark.parametrize("M", [1921, 37, 5])
def test_colsum_wide_equals_scalar(dtype, N, M):
    sn, ops = _sn()
    dev = torch.device("cuda", 0)
    ld = (N + 7) // 8 * 8
    X = (torch.randn(M, ld, device=dev) * 3).to(dtype)
    f = ops.colsum if dtype == torch.float32 else ops.colsum_bf16
    for beta in (0.0, 0.5):
        a = torch.randn(N, device=dev)
        b = a.clone()
        f(X, M, N, ld, a, beta=beta)
        f(X, M, N, ld, b, beta=beta, wide=True)
        torch.cuda.synchronize()
        assert torch.equal(a, b)


def test_adam_capped_grid_equal():
    sn, ops = _sn()
    dev = torch.device("cuda", 0)
    n = 3_000_000 + 37
    p0, g0 = torch.randn(n, device=dev), torch.randn(n, device=dev)
    m0, v0 = torch.randn(n, device=dev) * 0.1, torch.rand(n, device=dev) * 0.01
    outs = []
    for cap in (0, 17):
        p, g, m, v = p0.clone(), g0.clone(), m0.clone(), v0.clone()
        steps = torch.zeros(2, dtype=torch.int32, device=dev)
        lr = torch.full((1,), 1e-3, device=dev)
        coef = torch.zeros(6, device=dev)
        ops.adam_clamp_dev(p, g, m, v, [(0, 1_000_003), (1_000_003, n - 1_000_003)], [0, 1], steps, lr, coef,
                           0.9, 0.999, 1e-8, 0.5, max_ctas=cap)
        outs.append((p, g, m, v))
    torch.cuda.synchronize()
    for x, y in zip(*outs):
        assert torch.equal(x, y)


def _train(schedule, graph, steps, ragged=False):
    sn, ops = _sn()
    import bench
    old = ops.TAIL_SCHEDULE[0]
    ops.TAIL_SCHEDULE[0] = schedule
    try:
        dev = torch.device("cuda", 0)
        E, H, F, V, T, B = 300, 512, 512, 10000, 20, 96
        torch.manual_seed(0)
        dec = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.5).to(dev)
        dec.train()
        dec.set_precision("bf16")
        opt = sn.FusedClampAdam(dec, lr=5e-4, grad_clip=0.5)
        tr = sn.DataParallelTrainer(dec, opt)
        cap, lens, feat = bench.synthetic_batch(B, T, V, E, seed=0)
        if ragged:
            lens = sorted((int(x) for x in torch.randint(4, T + 1, (B,), generator=torch.Generator().manual_seed(1))),
                          reverse=True)
            lens[0] = T
        cap, feat = cap.to(dev), feat.to(dev)
        random.seed(0)
        losses = []
        if graph:
            g = sn.GraphedTrainStep(tr, cap, lens, feat, warmup=2, teacher_forcing_ratio=1.0, mode="happy")
            for _ in range(steps):
                g()
                losses.append(g.loss.clone())
        else:
            for _ in range(steps):
                loss, _ = tr.step(cap, lens, feat, teacher_forcing_ratio=1.0, mode="happy")
                losses.append(loss.clone())
        torch.cuda.synchronize()
        a = dec.arena()
        return (torch.stack(losses), a.flat.clone(), a.gflat.clone(), opt.m.clone(), opt.v.clone(),
                opt.steps_dev.clone())
    finally:
        ops.TAIL_SCHEDULE[0] = old


@pytest.mark.parametrize("graph,steps,ragged", [(False, 3, False), (False, 3, True), (True, 2, False)])
def test_training_step_tail_schedule_bitwise(graph, steps, ragged):
    new = _train(1, graph, steps, ragged)
    old = _train(0, graph, steps, ragged)
    for name, x, y in zip(("loss", "params", "grads", "m", "v", "steps"), new, old):
        assert torch.equal(x, y), name
