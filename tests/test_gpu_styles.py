"""Several styles in one beam search on the GPU: the grouped decode cell (sn_decode_cell_groups) and the >16-row
vocabulary projection against the single-group kernels bit for bit, and ``sample_batch(..., mode=[...])`` of the
factored decoder, the 3-layer stack and the attention decoder against the float64 oracle and the single-style calls."""
import pytest
import torch

pytestmark = pytest.mark.gpu

STYLE_ORDER = ("factual", "happy", "sad", "angry")


class _f64:
    """The oracle creates its zero states with the default dtype (like the reference, model.py:176-177)."""

    def __enter__(self):
        self.old = torch.get_default_dtype()
        torch.set_default_dtype(torch.float64)

    def __exit__(self, *a):
        torch.set_default_dtype(self.old)


# ---- kernels --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sizes", [(5,), (1, 16), (5, 1, 16), (16, 5, 5, 1), (5, 5, 5, 5)])
@pytest.mark.parametrize("gather", [False, True])
@pytest.mark.parametrize("Kx", [300, 30])
def test_decode_cell_groups_equals_per_group_decode_cell(sizes, gather, Kx):
    from icei_b200 import ops
    torch.manual_seed(len(sizes) * 7 + Kx)
    H, G = 512, len(sizes)
    R = sum(sizes)
    dev = "cuda"
    row_off = [0]
    for n in sizes:
        row_off.append(row_off[-1] + n)
    perm = torch.randperm(4)[:G]                        # groups in an arbitrary style order
    Wx_all = torch.randn(4, 4 * H, Kx, device=dev) * 0.05
    bx_all = torch.randn(4, 4 * H, device=dev) * 0.1
    Wx, bx = Wx_all[perm].contiguous(), bx_all[perm].contiguous()
    Wh = torch.randn(4 * H, H, device=dev) * 0.05
    bh = torch.randn(4 * H, device=dev) * 0.1
    h_prev = torch.randn(R, H, device=dev)
    c_prev = torch.randn(R, H, device=dev)
    if gather:
        table = torch.randn(50, Kx, device=dev)
        x_rows = torch.randint(0, 50, (R,), device=dev, dtype=torch.int32)
        src_row = torch.randint(0, R, (R,), device=dev, dtype=torch.int32)
        X = table
    else:
        X = torch.randn(R, Kx, device=dev)
        x_rows = src_row = None
    for cell in (ops.CELL_FACTORED, ops.CELL_LSTM):
        h_out = torch.full((R, H), float("nan"), device=dev)
        c_out = torch.full((R, H), float("nan"), device=dev)
        ops.decode_cell_groups(cell, H, torch.tensor(row_off, dtype=torch.int32, device=dev), max(sizes), Wx, Kx, X, 0,
                               bx, Wh, bh, h_prev, c_prev, src_row, h_out, c_out, x_rows=x_rows)
        h_ref = torch.empty(R, H, device=dev)
        c_ref = torch.empty(R, H, device=dev)
        for g in range(G):
            r0, r1 = row_off[g], row_off[g + 1]
            if gather:
                ops.decode_cell(cell, H, r1 - r0, Wx[g], Kx, X, 0, bx[g], Wh, bh, h_prev, c_prev, src_row[r0:r1],
                                h_ref[r0:r1], c_ref[r0:r1], x_rows=x_rows[r0:r1])
            else:
                ops.decode_cell(cell, H, r1 - r0, Wx[g], Kx, X[r0:r1], 0, bx[g], Wh, bh, h_prev[r0:r1], c_prev[r0:r1],
                                None, h_ref[r0:r1], c_ref[r0:r1])
        torch.cuda.synchronize()
        assert torch.equal(h_out, h_ref) and torch.equal(c_out, c_ref), (sizes, gather, Kx, cell)


@pytest.mark.parametrize("R", [17, 20, 37, 64, 128, 240])
@pytest.mark.parametrize("gather", [False, True])
def test_skinny_linear_over_16_rows_equals_row_chunks(R, gather):
    from icei_b200 import ops
    torch.manual_seed(R)
    V, K = 10000, 512
    W = torch.randn(V, K, device="cuda") * 0.05
    b = torch.randn(V, device="cuda")
    if gather:
        X = torch.randn(300, K, device="cuda")
        x_rows = torch.randint(0, 300, (R,), device="cuda", dtype=torch.int32)
    else:
        X, x_rows = torch.randn(R, K, device="cuda"), None
    out = torch.full((R, V), float("nan"), device="cuda")
    ops.skinny_linear(W, X, out, R, bias=b, x_rows=x_rows)
    ref = torch.empty(R, V, device="cuda")
    for r0 in range(0, R, 16):
        n = min(16, R - r0)
        if gather:
            ops.skinny_linear(W, X, ref[r0:r0 + n], n, bias=b, x_rows=x_rows[r0:r0 + n])
        else:
            ops.skinny_linear(W, X[r0:r0 + n], ref[r0:r0 + n], n, bias=b)
    torch.cuda.synchronize()
    assert torch.equal(out, ref)


# ---- end to end: DecoderFactoredLSTM at V = 10000 / H = 512 ------------------------------------------------------------
def _factored_pair(seed=4, max_seq_length=20):
    import icei_b200 as sn
    from oracle import port
    E, H, F, V = 300, 512, 512, 10000
    torch.manual_seed(seed)
    with _f64():
        ref = port.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0, max_seq_length=max_seq_length)
    port.sharpen_for_decode(ref)
    dec = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0, max_seq_length=max_seq_length)
    dec.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    return ref, dec.cuda().eval()


def _check_mixed(dec, ref, feats, modes, k, feed, oracle=True):
    """Mixed call == per-(image, style) oracle sample() == single-style sample_batch; a second call (graph replay) too."""
    x = feats.float().cuda()
    got = dec.sample_batch(x, 1, 2, k=k, mode=list(modes), feed_image=feed)
    again = dec.sample_batch(x, 1, 2, k=k, mode=list(modes), feed_image=feed)
    assert len(got) == len(modes)
    for i, m in enumerate(modes):
        single = dec.sample_batch(x[i:i + 1], 1, 2, k=k, mode=m, feed_image=feed)[0]
        assert got[i].dtype == torch.int64 and got[i].shape[0] == 1
        assert torch.equal(got[i], single), (i, m, k, feed, got[i].tolist(), single.tolist())
        assert torch.equal(again[i], got[i]), (i, m, k, feed)
        if oracle:
            with torch.no_grad(), _f64():
                want = ref.sample(feats[i:i + 1], 1, 2, k=k, mode=m, feed_image=feed)
            assert torch.equal(got[i].cpu(), want), (i, m, k, feed, got[i].tolist(), want.tolist())
    return got


def test_factored_styles_few_rows_and_gemm_path_vs_oracle():
    from icei_b200 import decode
    ref, dec = _factored_pair()
    g = torch.Generator().manual_seed(9)
    feats = torch.randn(16, 300, generator=g, dtype=torch.float64)
    lens = set()
    for feed in (True, False):
        for k in (1, 5):
            # one image in every style: the demo request (4 x k rows, matrix-vector kernels)
            got = _check_mixed(dec, ref, feats[:1].expand(4, -1), STYLE_ORDER, k, feed)
            lens |= {t.shape[1] for t in got}
            # a few images, styles out of order and repeated
            _check_mixed(dec, ref, feats[1:4], ["sad", "factual", "sad"], k, feed)
    # 16 images x 4 styles: 64 rows at k = 1 (few-row kernels, 4 row chunks), 320 at k = 5 (above the cap: GEMM path)
    modes = [STYLE_ORDER[(i + i // 4) % 4] for i in range(64)]
    rep = feats.repeat_interleave(4, 0)
    assert 64 * 5 > decode.STYLES_SKINNY_MAX_ROWS[0]
    for feed in (True, False):
        for k in (1, 5):
            # (without the image every caption of a style is the same: the oracle runs on the image-fed k = 5 case)
            _check_mixed(dec, ref, rep, modes, k, feed, oracle=(k == 5 and feed))
    assert len(lens) >= 2, lens


def test_factored_styles_follow_training_and_bf16_few_rows():
    import icei_b200 as sn
    from oracle import port
    _, dec = _factored_pair(seed=6, max_seq_length=12)
    g = torch.Generator().manual_seed(2)
    feats = torch.randn(2, 300, generator=g).cuda()
    x = feats[:1].expand(4, -1)
    modes = list(STYLE_ORDER)
    before = [t.clone() for t in dec.sample_batch(x, 1, 2, k=5, mode=modes, feed_image=True)]
    dec.sample_batch(x, 1, 2, k=5, mode=modes, feed_image=True)           # captured graphs from here on
    # an optimizer step on every style: the next call must see the new weights (collapsed chains refreshed)
    dec.train()
    opt = sn.FusedClampAdam(dec, lr=5e-2)
    tr = sn.DataParallelTrainer(dec, opt)
    cap, lens, f = port.synthetic_batch(8, 6, 10000, E=300, ragged=True, seed=3)
    for m in modes:
        tr.step(cap.cuda(), lens, f.cuda(), mode=m)
    dec.eval()
    after = dec.sample_batch(x, 1, 2, k=5, mode=modes, feed_image=True)
    for i, m in enumerate(modes):
        assert torch.equal(after[i], dec.sample_batch(x[i:i + 1], 1, 2, k=5, mode=m, feed_image=True)[0]), m
    assert any(not torch.equal(a, b) for a, b in zip(after, before))
    # bf16 mode: the few-row path keeps fp32 weights and arithmetic -> identical to the single-style calls
    dec.set_precision("bf16")
    mixed = ["angry", "factual", "happy", "angry"]
    xb = feats.repeat_interleave(2, 0)
    got = dec.sample_batch(xb, 1, 2, k=5, mode=mixed, feed_image=True)
    for i, m in enumerate(mixed):
        assert torch.equal(got[i], dec.sample_batch(xb[i:i + 1], 1, 2, k=5, mode=m, feed_image=True)[0]), (i, m)


def test_stack_styles_vs_oracle_composition():
    import icei_b200 as sn
    from oracle import port
    from oracle.stack import stack_sample
    E, H, F, V, L = 44, 64, 96, 517, 3
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        torch.manual_seed(5)
        layers = [port.DecoderFactoredLSTM(E if l == 0 else H, H, F, V, 1, dropout=0.0, max_seq_length=14)
                  for l in range(L)]
        for l, layer in enumerate(layers):
            port.lively_weights(layer, end_bias=2.0, seed=5 + l)
        torch.set_default_dtype(torch.float32)
        dec = sn.DecoderFactoredLSTMStack(E, H, F, V, L, dropout=0.0, max_seq_length=14)
        torch.set_default_dtype(torch.float64)
        dec.load_layer_state_dicts([{k: v.float() for k, v in l.state_dict().items()} for l in layers])
        dec = dec.cuda().eval()
        g = torch.Generator().manual_seed(1)
        feats = torch.randn(30, E, generator=g)
        for n_img, k in ((4, 5), (12, 1), (30, 5)):         # 20 / 12 rows (few-row kernels), 150 rows (GEMM path)
            modes = [STYLE_ORDER[(3 * i + 1) % 4] for i in range(n_img)]
            with torch.no_grad():
                want = [stack_sample(layers, feats[i:i + 1], 1, 2, k=k, mode=modes[i], feed_image=True)
                        for i in range(n_img)]
            for _ in range(2):
                got = dec.sample_batch(feats[:n_img].float().cuda(), 1, 2, k=k, mode=modes, feed_image=True)
                for i in range(n_img):
                    assert torch.equal(got[i].cpu(), want[i]), (n_img, k, i)
    finally:
        torch.set_default_dtype(old)


def test_attention_styles_vs_per_image_oracle():
    """DecoderFactoredLSTMAtt, 3 images in mixed styles, at the widths of the single-style batched attention test."""
    from icei_b200.decoders_att import DecoderFactoredLSTMAtt
    from oracle import port
    A, E, H, F, V, D = 512, 300, 512, 512, 2000, 2048
    torch.manual_seed(5)
    with _f64():
        ref = port.DecoderFactoredLSTMAtt(A, E, H, F, V, 1, feature_size=D, dropout=0.0, max_seq_length=16)
    port.sharpen_for_decode(ref)
    dec = DecoderFactoredLSTMAtt(A, E, H, F, V, 1, feature_size=D, dropout=0.0, max_seq_length=16)
    dec.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    dec = dec.cuda().eval()
    g = torch.Generator().manual_seed(10)
    feats = torch.randn(3, 7, 7, D, generator=g, dtype=torch.float64)
    modes = ["angry", "factual", "angry"]
    for k in (1, 3, 5):
        with torch.no_grad(), _f64():
            want = [ref.sample(feats[i:i + 1], 1, 2, k=k, mode=modes[i]) for i in range(3)]
        got = dec.sample_batch(feats.float().cuda(), 1, 2, k=k, mode=modes)
        for i in range(3):
            assert torch.equal(got[i].cpu(), want[i]), (k, i, got[i].tolist(), want[i].tolist())
            single = dec.sample_batch(feats[i:i + 1].float().cuda(), 1, 2, k=k, mode=modes[i])[0]
            assert torch.equal(got[i], single), (k, i)


def test_generate_styles_equals_per_style_generate():
    import icei_b200 as sn
    from icei_b200 import evaluate
    from oracle import port
    torch.manual_seed(3)
    dec = sn.DecoderFactoredLSTM(64, 128, 96, 700, 1, dropout=0.0, max_seq_length=12).cuda()
    port.sharpen_for_decode(dec, scale=20.0)
    g = torch.Generator().manual_seed(4)
    batches = [torch.randn(n, 64, generator=g).cuda() for n in (3, 1, 5)]
    got = evaluate.generate(dec, batches, 1, 2, k=3, styles=sn.STYLES, feed_image=True)
    assert list(got) == list(sn.STYLES)
    for s in sn.STYLES:
        assert got[s] == evaluate.generate(dec, batches, 1, 2, k=3, mode=s, feed_image=True), s
