"""Self-critical training on the GPU: the K12 sampler against the numpy Gumbel-max (oracle/scst.py) and a chi-square
test, ``sample_captions`` against the teacher-forced oracle and the training forward, the reward-weighted K5 loss in
both precisions, ``CiderD.score_samples`` against ``compute_score`` and the external-df oracle, and ``scst_step``
against the oracle step given the same samples."""
import random

import numpy as np
import pytest
import torch

from golden_util import rel_l2

pytestmark = pytest.mark.gpu

START, END = 1, 2


def _state(R, V, max_len=6, temperature=1.0, greedy=False, seed=0):
    from icei_b200.decode import SampleState
    st = SampleState(R, 1, max_len, START, temperature, greedy, torch.device("cuda"))
    st.seed_dev.fill_(seed)
    return st


@pytest.mark.parametrize("temperature", [1.0, 0.5, 2.0])
def test_sampler_kernel_vs_numpy_gumbel_max(temperature):
    from oracle import scst as so
    R, V, seed, step = 7, 1000, 11, 3
    g = torch.Generator().manual_seed(0)
    logits = torch.randn(R, V, generator=g) * 3
    st = _state(R, V, temperature=temperature, seed=seed)
    st.step_dev.fill_(step)
    st.step(logits.cuda(), step, END)
    torch.cuda.synchronize()
    lsm = torch.log_softmax(logits.double(), 1)
    for r in range(R):
        p = so.perturbed(logits[r].numpy(), seed, step, r, temperature)
        top2 = np.sort(p)[-2:]
        tok = int(st.seqs[r, step])
        if top2[1] - top2[0] > 1e-5:
            assert tok == int(np.argmax(p))
        assert p[tok] >= top2[1] - 1e-5
        assert int(st.prev_word[r]) == tok
        assert abs(float(st.logprob[r, step - 1]) - float(lsm[r, tok])) < 1e-5
    # greedy: the plain arg-max, lowest index on ties
    logits[:, 5] = 50.0
    logits[:, 9] = 50.0
    st = _state(R, V, greedy=True)
    st.step(logits.cuda(), 1, END)
    assert torch.equal(st.seqs[:, 1].cpu(), torch.full((R,), 5, dtype=torch.int64))


@pytest.mark.parametrize("temperature", [1.0, 0.5])
def test_sampler_chi_square(temperature):
    from scipy.stats import chisquare
    R, V = 200_000, 16
    row = torch.linspace(-2.0, 1.5, V)
    st = _state(R, V, temperature=temperature, seed=1234)
    st.step(row.expand(R, V).contiguous().cuda(), 1, END + 100)
    counts = torch.bincount(st.seqs[:, 1], minlength=V).cpu().double().numpy()
    expect = torch.softmax(row.double() / temperature, 0).numpy() * R
    stat, p = chisquare(counts, expect)
    assert p > 1e-3, (stat, p)


def _port_pair(kind, seed=3, sharpen=True, precision="fp32", V=97, E=24, H=32, F=24, max_len=8):
    import icei_b200 as sn
    from oracle import port
    torch.manual_seed(seed)
    if kind == "factored":
        ref = port.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0, max_seq_length=max_len)
        dec = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0, max_seq_length=max_len)
    else:
        ref = port.DecoderRNN(E, H, V, 1, dropout=0.0, max_seq_length=max_len)
        dec = sn.DecoderRNN(E, H, V, 1, dropout=0.0, max_seq_length=max_len)
    port.lively_weights(ref, gain=1.5, out_gain=4.0, end_bias=1.0, end_token=END)
    if sharpen:
        port.sharpen_for_decode(ref, end_token=END, scale=3.0, end_bias=1.0)
    dec.load_state_dict(ref.state_dict())
    dec = dec.cuda().set_precision(precision)
    dec.eval()
    return ref, dec


def _step_fn(ref, kind, mode):
    if kind == "factored":
        return ref.B, ref.C, (lambda x, s: ref.forward_step(x, s, mode))
    return ref.embed, ref.linear, (lambda x, s: ref.forward_step(x, s))


@pytest.mark.parametrize("kind", ["factored", "rnn"])
@pytest.mark.parametrize("n_img,n", [(3, 4), (10, 4)])          # 12 rows: few-row kernels; 40 rows: the GEMM path
def test_sample_captions_vs_teacher_forced_oracle(kind, n_img, n):
    from oracle import scst as so
    ref, dec = _port_pair(kind)
    ref = ref.double()
    mode = "happy"
    feats = torch.randn(n_img, 24, generator=torch.Generator().manual_seed(4))
    emb, out, step = _step_fn(ref, kind, mode)
    for temperature, greedy in ((1.0, False), (0.7, False), (1.0, True)):
        seqs, lens, lp = dec.sample_captions(feats.cuda(), START, END, n=n, temperature=temperature, seed=5, mode=mode,
                                             greedy=greedy)
        seqs, lens, lp = seqs.cpu(), lens.cpu(), lp.cpu()
        assert seqs.shape == (n_img * n, dec.max_seq_length + 2) and lp.shape == (n_img * n, dec.max_seq_length + 1)
        for r in range(n_img * n):
            L = int(lens[r])
            assert 2 <= L <= dec.max_seq_length + 2 and int(seqs[r, 0]) == START
            assert (L == dec.max_seq_length + 2) or int(seqs[r, L - 1]) == END
            assert not (seqs[r, 1:L - 1] == END).any() and not seqs[r, L:].any() and not lp[r, L - 1:].any()
            with torch.no_grad():
                lg = so.teacher_forced_logits(step, emb, out, feats[r // n], seqs[r], L)
            lsm = torch.log_softmax(lg, 1)
            for t in range(1, L):
                tok = int(seqs[r, t])
                assert abs(float(lp[r, t - 1]) - float(lsm[t - 1, tok])) < 1e-5
                if greedy:
                    assert tok == int(torch.argmax(lg[t - 1]))
                else:
                    p = so.perturbed(lg[t - 1].float().numpy(), 5, t, r, temperature)
                    assert p[tok] >= p.max() - 1e-4, (r, t)


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("bf16", 2e-2)])
@pytest.mark.parametrize("kind", ["factored", "rnn"])
def test_sample_logprob_equals_training_forward(precision, tol, kind):
    """The sampler's log-probabilities equal -NLL of forward_loss on the same sequences (steps t >= 1): the sampler
    conditions exactly as the teacher-forced training forward.  Per sequence, and over a whole length-sorted batch of
    samples (in bf16 mode the fused vocabulary-NLL path)."""
    import icei_b200 as sn
    _, dec = _port_pair(kind, precision=precision, sharpen=False)
    n_img, n = 16, 4
    feats = torch.randn(n_img, 24, generator=torch.Generator().manual_seed(7)).cuda()
    seqs, lens, lp = dec.sample_captions(feats, START, END, n=n, seed=9, mode="sad")
    lens_h = lens.cpu().tolist()
    if precision == "fp32":
        for r in range(8):
            L = lens_h[r]
            w = torch.ones(L, dtype=torch.float32, device="cuda")
            w[0] = 0.0                                   # the image step (target <start>) is not a draw
            loss, _ = dec.forward_loss(seqs[r:r + 1], [L], feats[r // n:r // n + 1], mode="sad", backward=False,
                                       token_weights=w, n_global=1)
            want = -float(lp[r, :L - 1].double().sum())
            assert abs(float(loss) - want) <= tol * max(1.0, abs(want)), (r, float(loss), want)
    order = sn.scst.sort_by_length(lens_h)
    idx = torch.tensor(order, device="cuda")
    lens_s = [lens_h[r] for r in order]
    plan = sn.PackPlan(lens_s)
    w = sn.scst.token_weights(torch.ones(len(order), dtype=torch.float64, device="cuda"), plan)
    loss, _ = dec.forward_loss(seqs.index_select(0, idx), lens_s, feats.index_select(0, idx // n), mode="sad",
                               backward=False, token_weights=w, n_global=1)
    want = -float(lp.double().sum())
    assert abs(float(loss) - want) <= tol * max(1.0, abs(want)), (float(loss), want)


@pytest.mark.parametrize("kind", ["factored", "rnn"])
@pytest.mark.parametrize("n_img,n", [(3, 4), (10, 4)])
def test_sample_seed_determinism_eager_and_graph(kind, n_img, n):
    _, dec = _port_pair(kind)
    feats = torch.randn(n_img, 24, generator=torch.Generator().manual_seed(1)).cuda()
    runs = [dec.sample_captions(feats, START, END, n=n, seed=7, mode="angry") for _ in range(3)]   # eager, then graphs
    for s, l, p in runs[1:]:
        assert torch.equal(s, runs[0][0]) and torch.equal(l, runs[0][1]) and torch.equal(p, runs[0][2])
    other = dec.sample_captions(feats, START, END, n=n, seed=8, mode="angry")
    assert not torch.equal(other[0], runs[0][0])


def _train_inputs(V, E, B, T, seed):
    from oracle import port
    return port.synthetic_batch(B, T, V, E=E, ragged=True, seed=seed)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_token_weights_ones_bitwise_equal_unweighted(precision):
    import icei_b200 as sn
    V, E, H, F, B, T = 517, 40, 64, 64, 56, 8
    cap, lens, feats = _train_inputs(V, E, B, T, 3)
    res = []
    for weighted in (False, True):
        torch.manual_seed(5)
        dec = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0).cuda().set_precision(precision)
        w = torch.ones(sum(lens), dtype=torch.float32, device="cuda") if weighted else None
        loss, _ = dec.forward_loss(cap.cuda(), lens, feats.cuda(), mode="sad", token_weights=w)
        torch.cuda.synchronize()
        res.append((loss.clone(), {k: p.grad.clone() for k, p in dec.named_parameters() if p.grad is not None}))
    assert torch.equal(res[0][0], res[1][0])
    assert res[0][1].keys() == res[1][1].keys()
    for k in res[0][1]:
        assert torch.equal(res[0][1][k], res[1][1][k]), k


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("bf16", 2e-2)])
@pytest.mark.parametrize("kind", ["factored", "rnn"])
def test_token_weights_mixed_sign_vs_oracle(precision, tol, kind):
    import icei_b200 as sn
    from oracle import port, scst as so
    V, E, H, F, B, T = 517, 40, 64, 64, 56, 8
    cap, lens, feats = _train_inputs(V, E, B, T, 4)
    torch.manual_seed(6)
    if kind == "factored":
        ref = port.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0)
        dec = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0)
        kw = {"mode": "angry"}
    else:
        ref = port.DecoderRNN(E, H, V, 1, dropout=0.0)
        dec = sn.DecoderRNN(E, H, V, 1, dropout=0.0)
        kw = {}
    dec.load_state_dict(ref.state_dict())
    dec = dec.cuda().set_precision(precision)
    N = sum(lens)
    w = torch.randn(N, generator=torch.Generator().manual_seed(8)) * 2
    w[::7] = 0.0
    denom = 123.0
    random.seed(0)
    out = ref(cap, lens, feats, teacher_forcing_ratio=1.0, **kw)
    loss_ref = so.weighted_loss(out, port.pack_targets(cap, lens), w, denom)
    loss_ref.backward()
    random.seed(0)
    loss, _ = dec.forward_loss(cap.cuda(), lens, feats.cuda(), token_weights=w.cuda(), n_global=denom, **kw)
    torch.cuda.synchronize()
    assert abs(float(loss) - float(loss_ref)) <= tol * max(1.0, abs(float(loss_ref)))
    mine = dict(dec.named_parameters())
    for n_, q in ref.named_parameters():
        if q.grad is not None:
            assert rel_l2(mine[n_].grad.cpu(), q.grad) < tol, n_


def _random_refs(n_img, V, seed):
    rng = np.random.default_rng(seed)
    return [[[int(x) for x in rng.integers(3, V, rng.integers(2, 9))] for _ in range(rng.integers(1, 5))]
            for _ in range(n_img)]


def test_score_samples_vs_compute_score_and_oracle():
    import icei_b200 as sn
    from oracle import scst as so
    V, n_img, ld = 20, 12, 11
    refs = _random_refs(n_img, V, 0)
    cd = sn.cider.CiderD(refs)
    rng = np.random.default_rng(1)
    R = 40
    seqs = torch.zeros(R, ld, dtype=torch.int64)
    lens = torch.zeros(R, dtype=torch.int64)
    hyps = []
    for r in range(R):
        L = int(rng.integers(1, ld + 1))
        body = [int(x) for x in rng.integers(3, V, max(0, L - 1))]
        if L >= 2 and rng.random() < 0.7:
            body[-1] = END
        seqs[r, 0] = START
        seqs[r, 1:L] = torch.tensor(body, dtype=torch.int64)
        lens[r] = L
        hyps.append(body[:-1] if body and body[-1] == END else body)
    # identity ids: bitwise equal to compute_score on the same hypotheses
    got = cd.score_samples(seqs[:n_img].cuda(), lens[:n_img].cuda(), list(range(n_img)), START, END)
    _, want = cd.compute_score(hyps[:n_img])
    assert got.dtype == torch.float64 and np.array_equal(got.cpu().numpy(), want)
    # repeated, shuffled ids: the external-df oracle
    ids = [int(x) for x in rng.integers(0, n_img, R)]
    got = cd.score_samples(seqs.cuda(), lens.cuda(), ids, START, END).cpu().numpy()
    want = so.sample_scores(refs, ids, hyps)
    assert np.all(np.abs(got - want) <= 1e-12 * np.maximum(1.0, np.abs(want)))


def _oracle_stack(E, H, F, V, L):
    from oracle import port
    layers = [port.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0)]
    layers += [port.DecoderFactoredLSTM(H, H, F, V, 1, dropout=0.0) for _ in range(L - 1)]
    return layers


@pytest.mark.parametrize("baseline", ["mean", "greedy"])
@pytest.mark.parametrize("kind", ["factored", "rnn", "stack3"])
def test_scst_step_vs_oracle_step(kind, baseline):
    import icei_b200 as sn
    from oracle import port, scst as so
    from oracle.stack import stack_forward, stack_parameters
    V, E, H, F, max_len = 40, 24, 32, 24, 7
    torch.manual_seed(2)
    mode = "happy"
    if kind == "factored":
        ref = port.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0, max_seq_length=max_len)
        dec = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0, max_seq_length=max_len)
        port.lively_weights(ref, out_gain=3.0, end_bias=1.0)
        dec.load_state_dict(ref.state_dict())
        params = list(ref.parameters())
        fwd = lambda c, l, f: ref(c, l, f, teacher_forcing_ratio=1.0, mode=mode)
    elif kind == "rnn":
        ref = port.DecoderRNN(E, H, V, 1, dropout=0.0, max_seq_length=max_len)
        dec = sn.DecoderRNN(E, H, V, 1, dropout=0.0, max_seq_length=max_len)
        port.lively_weights(ref, out_gain=3.0, end_bias=1.0)
        dec.load_state_dict(ref.state_dict())
        params = list(ref.parameters())
        fwd = lambda c, l, f: ref(c, l, f, teacher_forcing_ratio=1.0)
    else:
        layers = _oracle_stack(E, H, F, V, 3)
        for l in layers:
            port.lively_weights(l, out_gain=3.0, end_bias=1.0)
        dec = sn.DecoderFactoredLSTMStack(E, H, F, V, 3, dropout=0.0, max_seq_length=max_len)
        dec.load_layer_state_dicts([l.state_dict() for l in layers])
        params = stack_parameters(layers)
        fwd = lambda c, l, f: stack_forward(layers, c, l, f, teacher_forcing_ratio=1.0, mode=mode)
    dec = dec.cuda()
    dec.train()
    n_img, n = 6, 4
    refs = _random_refs(10, V, 3)
    ids = [7, 2, 2, 9, 0, 4]
    feats = torch.randn(n_img, E, generator=torch.Generator().manual_seed(5))
    cd = sn.cider.CiderD(refs)
    opt = sn.FusedClampAdam(dec, lr=1e-3, grad_clip=0.5)
    ropt = torch.optim.Adam(params, lr=1e-3)
    seed = 17
    # the samples the step will draw (the same seed and weights): the oracle step is given these
    with torch.no_grad():
        seqs, lens, _ = dec.sample_captions(feats.cuda(), START, END, n=n, seed=seed, mode=mode)
        gs = gl = None
        if baseline == "greedy":
            gs, gl, _ = dec.sample_captions(feats.cuda(), START, END, n=1, seed=seed, mode=mode, greedy=True)
    loss, rmean, bmean = sn.scst.scst_step(dec, opt, cd, feats.cuda(), ids, START, END, mode=mode, n=n,
                                           baseline=baseline, seed=seed)
    rl, rr, rb = so.reference_step(fwd, params, ropt, refs, feats, ids, seqs.cpu(), lens.cpu(), n, baseline, END,
                                   None if gs is None else gs.cpu(), None if gl is None else gl.cpu())
    assert abs(float(rmean) - rr) <= 1e-12 * max(1.0, abs(rr)) and abs(float(bmean) - rb) <= 1e-12 * max(1.0, abs(rb))
    assert abs(float(loss) - rl) <= 1e-5 * max(1.0, abs(rl))
    if kind == "stack3":
        want = {}
        for l, layer in enumerate(layers):
            for k, v in layer.state_dict().items():
                want[("" if l == 0 else "l%d_" % l) + k] = v
    else:
        want = ref.state_dict()
    for k, v in dec.state_dict().items():
        assert rel_l2(v.cpu(), want[k]) <= 1e-5, k


def test_scst_learns_a_tiny_memorisation_task():
    """Four images, one reference each: SCST from random weights raises the mean greedy CIDEr-D on these images."""
    import icei_b200 as sn
    V, E, H, F, max_len = 24, 16, 32, 16, 6
    torch.manual_seed(0)
    dec = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0, max_seq_length=max_len).cuda()
    refs = [[[5, 6, 7, 8]], [[9, 10, 11]], [[12, 13, 14, 15, 16]], [[17, 18]]]
    ids = [0, 1, 2, 3]
    feats = torch.randn(4, E, generator=torch.Generator().manual_seed(1)).cuda()
    cd = sn.cider.CiderD(refs)
    opt = sn.FusedClampAdam(dec, lr=1e-2, grad_clip=0.5)

    def greedy_score():
        s, l, _ = dec.sample_captions(feats, START, END, n=1, greedy=True)
        return float(cd.score_samples(s, l, ids, START, END).mean())

    curve = [greedy_score()]
    for it in range(200):
        sn.scst.scst_step(dec, opt, cd, feats, ids, START, END, n=8, seed=it)
        if (it + 1) % 25 == 0:
            curve.append(greedy_score())
    print("SCST greedy CIDEr-D every 25 steps:", " ".join("%.3f" % c for c in curve))
    assert curve[-1] > curve[0]
