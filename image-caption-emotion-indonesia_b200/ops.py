"""Thin tensor-level wrappers over the C ABI (include/sn100.h).  Tensors are only carriers of device
pointers; every op launches hand-written sm_100a kernels on torch's current CUDA stream."""
import ctypes

import torch

from . import _lib
from ._lib import OP_NN, OP_NT, OP_TN, CELL_FACTORED, CELL_LSTM  # noqa: F401
from ._lib import check as _check


def check(rc, what=""):
    _check(rc, what)
    if what != "sn_device_info":
        LAUNCHES[0] += 1


# number of libsn100 kernels launched (bench.py's gpu_launches); one per call unless noted
LAUNCHES = [0]


class no_gc_during_capture:
    """CUDA-graph capture runs in the global capture mode: if Python's cyclic garbage collector happens to free an
    OLDER torch.cuda.CUDAGraph while a capture is in progress, its cudaGraphExecDestroy invalidates the capture
    ("operation not permitted when stream is capturing (function reset)").  Collect first, then keep the collector off
    for the duration of the capture."""

    def __enter__(self):
        import gc
        gc.collect()
        self.was = gc.isenabled()
        gc.disable()

    def __exit__(self, *a):
        import gc
        if self.was:
            gc.enable()


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _req(t, dtype=torch.float32):
    if not t.is_cuda:
        raise _lib.SnError("libsn100 ops need CUDA tensors (no CPU fallback); got %s" % t.device)
    if t.dtype != dtype:
        raise _lib.SnError("expected %s, got %s" % (dtype, t.dtype))
    return t


def lib():
    l = _lib.load()
    _lib.require_device(torch.cuda.current_device())
    return l


# fp32 GEMMs: "split" = large ones run on the bf16 tensor cores with 3-limb operands (SN_PREC_BF16X6, fp32-grade
# accuracy: dropped terms <= 2^-24), small / TMA-illegal ones on the fp32 FFMA kernel; "simt" = always FFMA.
FP32_GEMM = ["split"]
SPLIT_MIN_MACS = 1 << 22
SPLIT_MAX_ACC_K = 768        # longest contraction accumulated in one TMEM accumulator in fp32 mode (see _gemm_split)


def _pad8(n):
    return (n + 7) // 8 * 8


def _split_cols(X, off, rows, K, ld, batch, s, pattern):
    """Limb-expand an operand whose contraction dimension runs along the columns.  Returns (tensor, ld', s') or None
    when the group layout is not one of {column blocks of width K, row-stacked contiguous groups}."""
    Kp = _pad8(K)
    if batch > 1 and s < ld:
        if s != K or ld < batch * K:
            return None
        G, R = batch, rows
    elif batch > 1:
        if s != rows * ld:
            return None
        G, R = 1, rows * batch
    else:
        G, R = 1, rows
    out = torch.empty(R, G * 6 * Kp, dtype=torch.bfloat16, device=X.device)
    check(lib().sn_split_limbs_cols(ctypes.c_void_p(X.data_ptr() + 4 * off), R, G, K, ld, _ptr(out), Kp, pattern,
                                    _stream()), "sn_split_limbs_cols")
    return out, G * 6 * Kp, (6 * Kp if G > 1 else rows * 6 * Kp)


def _split_rows(X, off, K, cols, ld, batch, s, pattern):
    """Limb-expand an operand whose contraction dimension runs along the rows ([K, cols] per group)."""
    Kp, ldp = _pad8(K), _pad8(ld)
    if batch > 1 and s < ld:
        if s % 8 != 0:
            return None
        G = 1                                    # column groups: the rows are shared, expand the whole matrix once
    elif batch > 1:
        if s != K * ld:
            return None
        G = batch
    else:
        G = 1
    out = torch.empty(G * 6 * Kp, ldp, dtype=torch.bfloat16, device=X.device)
    check(lib().sn_split_limbs_rows(ctypes.c_void_p(X.data_ptr() + 4 * off), G, K, ld, ld, _ptr(out), Kp, ldp, pattern,
                                    _stream()), "sn_split_limbs_rows")
    return out, ldp, (s if (batch > 1 and s < ld) else 6 * Kp * ldp)


def _gemm_split(op, A, B, C, M, N, K, lda, ldb, ldc, bias, beta, batch, sA, sB, sC, sBias, a_off, b_off, c_off,
                bias_off):
    if K > 10900:               # 6*Kp must stay a sane contraction length / fit the row-split launch
        return False
    # The tensor core aligns every MMA's products to its running fp32 accumulator and truncates (~2^-24 of the
    # accumulator per 16-deep MMA, one-sided): a contraction of thousands of terms in ONE accumulator drifts past the
    # fp32 mode's budget (measured: 1.2e-5 on dW_hh with K = 1920 tokens).  Long contractions are therefore cut into
    # pieces of <= 768 accumulated in separate accumulators (the CTA-pair kernel's deterministic work-space split-K) and
    # summed in fp32 with round-to-nearest; the single-CTA kernel (M < 256) has no such path -> FFMA there.
    Kp6 = 6 * _pad8(K)
    splits = 1
    if K > SPLIT_MAX_ACC_K:
        if M < 256 or N % 4 != 0:
            return False
        splits = -(-Kp6 // SPLIT_MAX_ACC_K)
        while splits > 1 and M * N * batch * splits * 4 > (1 << 30):
            splits -= 1
    ea = _split_cols(A, a_off, M, K, lda, batch, sA, 0) if op in (OP_NT, OP_NN) else _split_rows(A, a_off, K, M, lda, batch, sA, 0)
    if ea is None:
        return False
    eb = _split_cols(B, b_off, N, K, ldb, batch, sB, 1) if op == OP_NT else _split_rows(B, b_off, K, N, ldb, batch, sB, 1)
    if eb is None:
        return False
    LAUNCHES[0] += 2
    gemm_bf16(op, ea[0], eb[0], M, N, Kp6, ea[1], eb[1], C=C, ldc=ldc, bias=bias, beta=beta, batch=batch,
              sA=ea[2] if batch > 1 else 0, sB=eb[2] if batch > 1 else 0, sC=sC, sBias=sBias, c_off=c_off,
              bias_off=bias_off, splits=splits if splits > 1 else 1, impl="pair" if splits > 1 else None)
    return True


def gemm(op, A, B, C, M, N, K, lda, ldb, ldc, bias=None, beta=0.0, batch=1, sA=0, sB=0, sC=0, sBias=0,
         a_off=0, b_off=0, c_off=0, bias_off=0):
    """C = op(A) op(B) + bias + beta*C.  Offsets are in elements (pointer arithmetic on the base)."""
    _req(A); _req(B); _req(C)
    # (M >= 256: the time-batched GEMMs.  Per-step GEMMs on <= 96 rows would re-expand their weight operand every step.)
    if (FP32_GEMM[0] == "split" and M * N * K * batch >= SPLIT_MIN_MACS and M >= 256 and N >= 16 and K >= 16
            and batch <= 4 and ldc % 4 == 0 and c_off % 4 == 0 and (batch == 1 or sC % 4 == 0)
            and _gemm_split(op, A, B, C, M, N, K, lda, ldb, ldc, bias, beta, batch, sA, sB, sC, sBias, a_off, b_off,
                            c_off, bias_off)):
        return C
    pa = ctypes.c_void_p(A.data_ptr() + 4 * a_off)
    pb = ctypes.c_void_p(B.data_ptr() + 4 * b_off)
    pc = ctypes.c_void_p(C.data_ptr() + 4 * c_off)
    pbias = ctypes.c_void_p(bias.data_ptr() + 4 * bias_off) if bias is not None else None
    check(lib().sn_gemm(op, M, N, K, pa, lda, pb, ldb, pc, ldc, pbias, float(beta), batch, sA, sB, sC, sBias,
                        _stream()), "sn_gemm")
    return C


def linear_nt(x, w, bias=None, out=None):
    """out[M,N] = x[M,K] @ w[N,K]^T + bias  (nn.Linear forward) for contiguous 2-D tensors."""
    M, K = x.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty(M, N, device=x.device, dtype=torch.float32)
    return gemm(OP_NT, x, w, out, M, N, K, x.stride(0), w.stride(0), out.stride(0), bias=bias)


def colsum(X, M, N, ldx, out, beta=0.0, x_off=0, out_off=0, wide=False):
    """``wide``: 16-byte loads where X and ldx allow (the same bits as the scalar kernel)."""
    _req(X); _req(out)
    check(lib().sn_colsum_ex(ctypes.c_void_p(X.data_ptr() + 4 * x_off), M, N, ldx,
                             ctypes.c_void_p(out.data_ptr() + 4 * out_off), float(beta), 1 if wide else 0, _stream()),
          "sn_colsum")
    return out


def gather_pack_fwd(captions, table, features, has_feat, row_b, row_t, tok_override, N, X, p_drop, seed,
                    row_off=0, seed_dev=None, Xb=None):
    """X (fp32, may be None) and/or Xb (bf16, K-padded) receive the packed input rows."""
    E = table.shape[1]
    cap = _req(captions, torch.int64)
    ro4 = 4 * row_off
    check(lib().sn_gather_pack_fwd(
        _ptr(cap), cap.stride(0), _ptr(_req(table)), E,
        _ptr(features) if features is not None else None, features.stride(0) if features is not None else 0,
        1 if has_feat else 0,
        ctypes.c_void_p(row_b.data_ptr() + ro4), ctypes.c_void_p(row_t.data_ptr() + ro4),
        ctypes.c_void_p(tok_override.data_ptr() + ro4) if tok_override is not None else None,
        N, ctypes.c_void_p(X.data_ptr() + 4 * row_off * X.stride(0)) if X is not None else None,
        X.stride(0) if X is not None else 0, float(p_drop), ctypes.c_uint64(seed), _ptr(seed_dev),
        ctypes.c_void_p(Xb.data_ptr() + 2 * row_off * Xb.stride(0)) if Xb is not None else None,
        Xb.stride(0) if Xb is not None else 0, _stream()), "sn_gather_pack_fwd")


def colsum_bf16(X, M, N, ldx, out, beta=0.0, wide=False):
    _req(X, torch.bfloat16); _req(out)
    check(lib().sn_colsum_bf16_ex(_ptr(X), M, N, ldx, _ptr(out), float(beta), 1 if wide else 0, _stream()),
          "sn_colsum_bf16")
    return out


def gather_pack_bwd(captions, dtable, dfeatures, has_feat, row_b, row_t, tok_override, N, dX, p_drop, seed,
                    seed_dev=None):
    V, E = dtable.shape
    cap = _req(captions, torch.int64)
    # work space of the token grouping (layout: include/sn100.h); allocated per call so that concurrent calls on
    # different streams never share it
    ws_int = torch.empty(4 * V + 1 + 3 * N, dtype=torch.int32, device=dX.device)
    ws_part = torch.empty((N // 16 + 1) * E, dtype=torch.float32, device=dX.device)
    check(lib().sn_gather_pack_bwd(
        _ptr(cap), cap.stride(0), _ptr(_req(dtable)), E,
        _ptr(dfeatures) if dfeatures is not None else None,
        dfeatures.stride(0) if dfeatures is not None else 0, 1 if has_feat else 0,
        _ptr(row_b), _ptr(row_t), _ptr(tok_override) if tok_override is not None else None,
        N, _ptr(_req(dX)), dX.stride(0), float(p_drop), ctypes.c_uint64(seed), _ptr(seed_dev),
        V, _ptr(ws_int), _ptr(ws_part), _stream()),
          "sn_gather_pack_bwd")


def embed_plan_ws(V, N, device):
    """Work space of the token grouping of sn_embed_plan / sn_embed_grad (layout: include/sn100.h)."""
    return torch.empty(4 * V + 1 + 3 * N, dtype=torch.int32, device=device)


def embed_plan(captions, has_feat, row_b, row_t, tok_override, N, V, ws_int):
    """Plan part of the embedding backward (sn_embed_plan): groups the token rows by token into ``ws_int``."""
    cap = _req(captions, torch.int64)
    check(lib().sn_embed_plan(_ptr(cap), cap.stride(0), 1 if has_feat else 0, _ptr(row_b), _ptr(row_t),
                              _ptr(tok_override) if tok_override is not None else None, N, V, _ptr(_req(ws_int, torch.int32)),
                              _stream()), "sn_embed_plan")


def embed_grad(dtable, dfeatures, has_feat, row_b, row_t, tok_override, N, dX, p_drop, seed, ws_int, seed_dev=None,
               wide=True):
    """Gradient part (sn_embed_grad): group sums of dX into the zeroed ``dtable`` by the plan in ``ws_int``."""
    V, E = dtable.shape
    ws_part = torch.empty((N // 16 + 1) * E, dtype=torch.float32, device=dX.device)
    check(lib().sn_embed_grad(
        _ptr(_req(dtable)), E, _ptr(dfeatures) if dfeatures is not None else None,
        dfeatures.stride(0) if dfeatures is not None else 0, 1 if has_feat else 0, _ptr(row_b), _ptr(row_t),
        _ptr(tok_override) if tok_override is not None else None, N, _ptr(_req(dX)), dX.stride(0), float(p_drop),
        ctypes.c_uint64(seed), _ptr(seed_dev), V, _ptr(_req(ws_int, torch.int32)), _ptr(ws_part), 1 if wide else 0, _stream()),
          "sn_embed_grad")


_ws_cache = {}


def _recur_ws(device, T):
    key = (device, T)
    ws = _ws_cache.get(key)
    if ws is None:
        nbytes = lib().sn_recur_ws_bytes(1, T)
        ws = torch.empty(nbytes // 4 + 1, dtype=torch.int32, device=device)
        _ws_cache[key] = ws
    return ws


def recur_fwd(cell, H, B, bs, off, t0, t1, XP, Whh, bhh, h_init, Hall, Call, Hprev, gates, c_state):
    ws = _recur_ws(XP.device, t1 + 1)
    check(lib().sn_recur_fwd(cell, H, B, _ptr(bs), _ptr(off), t0, t1, _ptr(_req(XP)), _ptr(_req(Whh)),
                             _ptr(h_init), _ptr(bhh), _ptr(Hall), _ptr(Call), _ptr(Hprev), _ptr(gates),
                             _ptr(c_state), _ptr(ws), _stream()), "sn_recur_fwd")


def recur_bwd(cell, H, B, bs, off, t0, t1, Whh, c_init, Call, gates, dHall, dZ, dh_carry, dc_carry):
    ws = _recur_ws(dZ.device, t1 + 1)
    check(lib().sn_recur_bwd(cell, H, B, _ptr(bs), _ptr(off), t0, t1, _ptr(_req(Whh)), _ptr(c_init),
                             _ptr(Call), _ptr(gates), _ptr(_req(dHall)), _ptr(dZ), _ptr(dh_carry),
                             _ptr(dc_carry), _ptr(ws), _stream()), "sn_recur_bwd")


def softmax_nll(logits, N, V, targets=None, row_loss=None, dlogits=None, grad_scale=1.0, argmax=None,
                top5hit=None, row_off=0, dlogits_bf16=None, row_weight=None):
    ld = logits.stride(0)
    check(lib().sn_softmax_nll(
        ctypes.c_void_p(logits.data_ptr() + 4 * row_off * ld), N, V, ld, _ptr(targets), _ptr(row_loss),
        _ptr(dlogits), dlogits.stride(0) if dlogits is not None else 0, float(grad_scale),
        _ptr(None if row_weight is None else _req(row_weight)), _ptr(argmax),
        _ptr(top5hit), _ptr(dlogits_bf16), dlogits_bf16.stride(0) if dlogits_bf16 is not None else 0,
        _stream()), "sn_softmax_nll")


def reduce_sum(x, N, scale, out, accumulate=False, row_weight=None):
    """out = scale * sum(x[:N] * row_weight[:N]) (row_weight None: weight 1)."""
    check(lib().sn_reduce_sum(_ptr(_req(x)), N, float(scale), _ptr(None if row_weight is None else _req(row_weight)),
                              _ptr(out), 1 if accumulate else 0, _stream()), "sn_reduce_sum")


def adam_clamp(p, g, m, v, ranges, step_sizes, bc2_sqrts, beta1, beta2, eps, clip):
    n = len(ranges)
    if n == 0:
        return
    R = (ctypes.c_int64 * (2 * n))()
    S = (ctypes.c_float * n)()
    C = (ctypes.c_float * n)()
    for i, (o, l) in enumerate(ranges):
        R[2 * i], R[2 * i + 1] = o, l
        S[i], C[i] = step_sizes[i], bc2_sqrts[i]
    check(lib().sn_adam_clamp(_ptr(_req(p)), _ptr(_req(g)), _ptr(_req(m)), _ptr(_req(v)), n,
                              ctypes.cast(R, ctypes.c_void_p), ctypes.cast(S, ctypes.c_void_p),
                              ctypes.cast(C, ctypes.c_void_p), beta1, beta2, eps, clip, _stream()),
          "sn_adam_clamp")


def mean_pixels(feat, B, P, D, out):
    check(lib().sn_mean_pixels(_ptr(_req(feat)), B, P, D, _ptr(out), _stream()), "sn_mean_pixels")


def _att_b16_ok(feat_b16, att1, A, D):
    return (feat_b16 is not None and D == 2048 and A % 4 == 0 and feat_b16.data_ptr() % 16 == 0
            and att1.data_ptr() % 16 == 0)


def att_step_fwd(att1, att2, feat, wfull, bfull, gate_pre, nb, P, A, D, alpha, ld_alpha, ctx, ldc, feat_b16=None):
    """``feat_b16``: bf16 copy of the feature map (bf16 mode) -> the 16-byte-load kernel reading half the bytes."""
    if _att_b16_ok(feat_b16, att1, A, D) and ldc % 2 == 0:
        check(lib().sn_att_step_fwd_b16(_ptr(_req(att1)), _ptr(_req(att2)), _ptr(_req(feat_b16, torch.bfloat16)),
                                        _ptr(_req(wfull)), float(bfull), _ptr(_req(gate_pre)), nb, P, A, D, _ptr(alpha),
                                        ld_alpha, _ptr(ctx), ldc, _stream()), "sn_att_step_fwd_b16")
        return
    check(lib().sn_att_step_fwd(_ptr(_req(att1)), _ptr(_req(att2)), _ptr(_req(feat)), _ptr(_req(wfull)),
                                float(bfull), _ptr(_req(gate_pre)), nb, P, A, D, _ptr(alpha), ld_alpha,
                                _ptr(ctx), ldc, _stream()), "sn_att_step_fwd")


def att_step_bwd(att1, att2, feat, wfull, bfull, gate_pre, alpha, ld_alpha, dctx, ldc, dalpha_extra, ld_da,
                 nb, P, A, D, datt2, dgate_pre, datt1, dwfull, dfeat, feat_b16=None):
    if dfeat is None and _att_b16_ok(feat_b16, att1, A, D) and datt1.data_ptr() % 16 == 0:
        check(lib().sn_att_step_bwd_b16(_ptr(_req(att1)), _ptr(_req(att2)), _ptr(_req(feat_b16, torch.bfloat16)),
                                        _ptr(_req(wfull)), _ptr(_req(gate_pre)), _ptr(alpha), ld_alpha, _ptr(_req(dctx)),
                                        ldc, _ptr(dalpha_extra), ld_da, nb, P, A, D, _ptr(datt2), _ptr(dgate_pre),
                                        _ptr(datt1), _ptr(dwfull), _stream()), "sn_att_step_bwd_b16")
        LAUNCHES[0] += 1
        return
    check(lib().sn_att_step_bwd(_ptr(_req(att1)), _ptr(_req(att2)), _ptr(_req(feat)), _ptr(_req(wfull)),
                                float(bfull), _ptr(_req(gate_pre)), _ptr(alpha), ld_alpha, _ptr(_req(dctx)), ldc,
                                _ptr(dalpha_extra), ld_da, nb, P, A, D, _ptr(datt2), _ptr(dgate_pre),
                                _ptr(datt1), _ptr(dwfull), _ptr(dfeat), _stream()), "sn_att_step_bwd")


def _bptr(t, off_elems, elem_size):
    return ctypes.c_void_p(t.data_ptr() + elem_size * off_elems) if t is not None else None


# GEMM kernel selection for gemm_bf16: "auto" = CTA-pair kernel (sn_gemm2.cu) when the problem has at least one
# full 256-row tile, else the single-CTA 128x128 kernel (sn_gemm_tc.cu); "tc" / "pair" force one of them.
GEMM_IMPL = ["auto"]
_SM_PAIRS = 74


def _pick_splits(M, N, K, batch):
    """Split-K factor for the pair kernel: fill the 74 SM pairs when the tile count alone cannot."""
    tiles = ((M + 255) // 256) * ((N + 255) // 256) * batch
    kb = (K + 63) // 64
    # only long-K problems (dH = dL C, K = vocabulary): for the K = tokens weight-gradient GEMMs (30 k-blocks at
    # configs[1]) the partial GEMM + reduction launches cost more than the 16 unsplit tiles (timeline, profiles/r1_l)
    if tiles * 2 > _SM_PAIRS or kb < 64:
        return 1
    return max(1, min(_SM_PAIRS // tiles, kb // 8, 16))


_g2_ws = {}


def _gemm2_ws(device, nbytes):
    """Split-K work space, one per (device, stream): sized up on demand, reused across calls."""
    key = (device, torch.cuda.current_stream().cuda_stream)
    ws = _g2_ws.get(key)
    if ws is None or ws.numel() * 4 < nbytes:
        ws = torch.empty(nbytes // 4 + 4, dtype=torch.float32, device=device)
        _g2_ws[key] = ws
    return ws


def gemm_bf16(op, A, B, M, N, K, lda, ldb, C=None, ldc=0, Cb=None, ldcb=0, bias=None, beta=0.0, batch=1,
              sA=0, sB=0, sC=0, sCb=0, sBias=0, a_off=0, b_off=0, c_off=0, cb_off=0, bias_off=0, splits=1,
              impl=None, max_pairs=0):
    """tcgen05 GEMM: A, B bf16; C fp32 and/or Cb bf16.  Offsets in elements of the respective tensor.
    Pair kernel: splits=1 -> automatic split-K (deterministic work-space reduction) for few-tile / long-K shapes.
    Single-CTA kernel: splits: 1 = off, 0 = automatic, n = forced (fp32 atomics).
    max_pairs (pair kernel): cap the grid at that many SM pairs (side-stream GEMMs)."""
    _req(A, torch.bfloat16); _req(B, torch.bfloat16)
    impl = impl or GEMM_IMPL[0]
    if impl == "pair" or (impl == "auto" and M >= 256):
        sp = _pick_splits(M, N, K, batch) if splits in (0, 1) else splits
        if sp > 1 and N % 4 != 0:
            sp = 1
        ws, wsb = None, 0
        if sp > 1:
            wsb = lib().sn_gemm2_ws_bytes(M, N, batch, sp)
            ws = _gemm2_ws(A.device, wsb)
            LAUNCHES[0] += batch
        check(lib().sn_gemm2_bf16(op, M, N, K, _bptr(A, a_off, 2), lda, _bptr(B, b_off, 2), ldb,
                                  _bptr(C, c_off, 4), ldc, _bptr(Cb, cb_off, 2), ldcb, _bptr(bias, bias_off, 4),
                                  float(beta), batch, sA, sB, sC, sCb, sBias, sp, _ptr(ws), wsb, int(max_pairs),
                                  _stream()), "sn_gemm2_bf16")
        return
    check(lib().sn_gemm_bf16_splitk(op, M, N, K, _bptr(A, a_off, 2), lda, _bptr(B, b_off, 2), ldb,
                                    _bptr(C, c_off, 4), ldc, _bptr(Cb, cb_off, 2), ldcb, _bptr(bias, bias_off, 4),
                                    float(beta), batch, sA, sB, sC, sCb, sBias, splits, _stream()), "sn_gemm_bf16")


def vocab_nll_fwd(Hb, Wb, bias, targets, N, V, H, tlogit, lse, row_loss=None, argmax=None, above=None):
    """Vocabulary projection fused with log-softmax / NLL statistics (no logits in HBM)."""
    _req(Hb, torch.bfloat16); _req(Wb, torch.bfloat16); _req(targets, torch.int64)
    nbytes = lib().sn_vocab_ws_bytes(N, V)
    ws = _gemm2_ws(Hb.device, nbytes)
    check(lib().sn_vocab_nll_fwd(N, V, H, _ptr(Hb), Hb.stride(0), _ptr(Wb), Wb.stride(0), _ptr(_req(bias)),
                                 _ptr(targets), _ptr(ws), nbytes, _ptr(tlogit), _ptr(lse), _ptr(row_loss),
                                 _ptr(argmax), _ptr(above), _stream()), "sn_vocab_nll_fwd")
    LAUNCHES[0] += 1


def vocab_nll_bwd(Hb, Wb, bias, targets, N, V, H, tlogit, lse, grad_scale, dLb=None, above=None, top5hit=None,
                  row_weight=None):
    """Recompute the logits tiles; write (softmax - onehot) * grad_scale (* row_weight[row]) as bf16 [N, ld]; rank of
    the target."""
    _req(Hb, torch.bfloat16); _req(Wb, torch.bfloat16); _req(targets, torch.int64)
    check(lib().sn_vocab_nll_bwd(N, V, H, _ptr(Hb), Hb.stride(0), _ptr(Wb), Wb.stride(0), _ptr(_req(bias)),
                                 _ptr(targets), _ptr(tlogit), _ptr(lse), float(grad_scale),
                                 _ptr(None if row_weight is None else _req(row_weight)), _ptr(dLb),
                                 dLb.stride(0) if dLb is not None else 0, _ptr(above), _ptr(top5hit), _stream()),
          "sn_vocab_nll_bwd")
    if top5hit is not None:
        LAUNCHES[0] += 1


def cast_bf16(src, R, C, lds, dst, Cp, ldd, src_off=0, dst_off=0, max_blocks=0):
    """max_blocks > 0 caps the grid (side-stream casts: a cast block on an SM keeps a CTA-pair GEMM off it)."""
    check(lib().sn_cast_bf16_ex(_bptr(_req(src), src_off, 4), R, C, lds, _bptr(dst, dst_off, 2), Cp, ldd, max_blocks,
                                _stream()), "sn_cast_bf16")


def to_bf16_padded(x, pad_to=8):
    """bf16 copy of a contiguous fp32 [R,C] matrix with C padded up to a multiple of ``pad_to`` (zeros)."""
    R, C = x.shape
    Cp = (C + pad_to - 1) // pad_to * pad_to
    out = torch.empty(R, Cp, dtype=torch.bfloat16, device=x.device)
    cast_bf16(x, R, C, x.stride(0), out, Cp, Cp)
    return out


# Scheduling of the vocabulary projection's weight gradient (dC) against the reverse recurrence (decoders._vocab_backward):
# 0 = launch it immediately on the side stream; 1 = make it runnable together with the recurrence but LAUNCH it after it
# (the cluster-form recurrence needs whole free SMs, 16 per cluster); 2 = start it only after the recurrence finished.
import os as _os
DC_SCHEDULE = [int(_os.environ.get("SN_DC_SCHEDULE", "0"))]     # measured: 0 is the fastest (profiles/README.md, r2)
DC_MAX_PAIRS = [int(_os.environ.get("SN_DC_MAX_PAIRS", "37"))]     # half of the 74 SM pairs (measured best, profiles/README.md r2)

# schedule of the tail of a single-GPU bf16 training step (DESIGN.md section 4).  1 (default): the embedding's token
# grouping and gradient zeroing run on a side stream at the start of a teacher-forced forward, the group sums use the
# one-thread-per-column kernel, d b_hh / d b_U are one column sum plus a copy, and the column sums use 16-byte loads.
# 0: the previous schedule.  Both compute the same bits.
TAIL_SCHEDULE = [int(_os.environ.get("SN_TAIL_SCHEDULE", "1"))]
# grid cap (CTAs of 256 threads) of the Adam buckets that run next to the projection-backward chain under the tail
# schedule; 0 = full width.  Measured on a B200 at configs[1]: 74 CTAs 0.492 ms/step, 148 0.453, 296 0.426, full width
# 0.421 (profiles/README.md, r4) -- a capped Adam only stretches out under the chain, so the default is no cap
ADAM_BG_CTAS = [int(_os.environ.get("SN_ADAM_BG_CTAS", "0"))]

# hold the side-stream work of the vocabulary backward behind sn_gate_wait (experiment, OFF: no gain on one GPU --
# the step is bound by total work, not by the delayed clusters -- and a 2-GPU run with the peer exchange behind the
# gate did not finish; profiles/README.md r2)
GATE_DC = [int(_os.environ.get("SN_GATE_DC", "0"))]

# K3 implementation in bf16 mode: "auto" = the cluster form (sn_recur_cl.cu) whenever the hidden size supports it and all
# sample slices fit the device at once, else the flag-synchronised persistent kernel; "cluster" / "flags" force one.
RECUR_IMPL = ["auto"]
_cl_max = {}


def recur_cluster_ok(H, B):
    impl = RECUR_IMPL[0]
    if impl == "flags" or H not in (128, 256, 512):
        return False
    key = (torch.cuda.current_device(), H)
    n = _cl_max.get(key)
    if n is None:
        n = _cl_max[key] = int(lib().sn_recur_cl_max_clusters(H))
    if impl == "cluster":
        if n < 1:
            raise _lib.SnError("cluster form of the recurrence is not available for H=%d on this device" % H)
        return True
    return n >= 1 and (B + 15) // 16 <= n


def recur_fwd_bf16(cell, H, B, bs, off, t0, t1, XP, Whh_b, bhh, h_init, Hall, Hb, Hprevb, Call, gates, c_state):
    if recur_cluster_ok(H, B):
        check(lib().sn_recur_fwd_cl(cell, H, B, _ptr(bs), _ptr(off), t0, t1, _ptr(_req(XP)),
                                    _ptr(_req(Whh_b, torch.bfloat16)), _ptr(bhh), _ptr(h_init), _ptr(Hall),
                                    _ptr(_req(Hb, torch.bfloat16)), _ptr(Hprevb), _ptr(Call), _ptr(gates),
                                    _ptr(c_state), _stream()), "sn_recur_fwd_cl")
        return
    ws = _recur_ws(XP.device, t1 + 1)
    check(lib().sn_recur_fwd_bf16(cell, H, B, _ptr(bs), _ptr(off), t0, t1, _ptr(_req(XP)),
                                  _ptr(_req(Whh_b, torch.bfloat16)), _ptr(bhh), _ptr(h_init), _ptr(Hall),
                                  _ptr(_req(Hb, torch.bfloat16)), _ptr(Hprevb), _ptr(Call), _ptr(gates),
                                  _ptr(c_state), _ptr(ws), _stream()), "sn_recur_fwd_bf16")


def recur_bwd_bf16(cell, H, B, bs, off, t0, t1, Whh_b, c_init, Call, gates, dHall, dZ, dZb, dh_carry, dc_carry,
                   start_flag=None):
    if recur_cluster_ok(H, B):
        check(lib().sn_recur_bwd_cl(cell, H, B, _ptr(bs), _ptr(off), t0, t1, _ptr(_req(Whh_b, torch.bfloat16)),
                                    _ptr(c_init), _ptr(Call), _ptr(gates), _ptr(_req(dHall)), _ptr(dZ),
                                    _ptr(_req(dZb, torch.bfloat16)), _ptr(dh_carry), _ptr(dc_carry), _ptr(start_flag),
                                    _stream()), "sn_recur_bwd_cl")
        return
    ws = _recur_ws(dZb.device, t1 + 1)
    check(lib().sn_recur_bwd_bf16(cell, H, B, _ptr(bs), _ptr(off), t0, t1, _ptr(_req(Whh_b, torch.bfloat16)),
                                  _ptr(c_init), _ptr(Call), _ptr(gates), _ptr(_req(dHall)), _ptr(dZ),
                                  _ptr(_req(dZb, torch.bfloat16)), _ptr(dh_carry), _ptr(dc_carry), _ptr(ws),
                                  _stream()), "sn_recur_bwd_bf16")


# ---- K3, large-batch form (one tcgen05 GEMM per step, cell fused into the epilogue) -----------------------------
RECUR_GEMM_MIN_BATCH = [1024]      # samples per GPU from which the per-step GEMM form replaces the persistent kernel


def _host_steps(plan):
    hs = plan.__dict__.get("_host_steps")
    if hs is None:
        T = plan.T
        hs = ((ctypes.c_int32 * T)(*[int(x) for x in plan.bs]), (ctypes.c_int32 * T)(*[int(x) for x in plan.off[:T]]))
        plan.__dict__["_host_steps"] = hs
    return hs


_zeros_b16 = {}


def _zeros_bf16(device, n):
    z = _zeros_b16.get(device)
    if z is None or z.numel() < n:
        z = torch.zeros(n, dtype=torch.bfloat16, device=device)
        _zeros_b16[device] = z
    return z


def cast_gate_interleave(W):
    """bf16 copy of W_hh [4H, H] with the rows of the four gate blocks interleaved 64 units at a time."""
    H4, K = W.shape
    H = H4 // 4
    Kp = (K + 7) // 8 * 8
    out = torch.empty(H4, Kp, dtype=torch.bfloat16, device=W.device)
    check(lib().sn_cast_bf16_gate_interleave(_ptr(_req(W)), H, K, W.stride(0), _ptr(out), Kp, _stream()),
          "sn_cast_bf16_gate_interleave")
    return out


def recur_fwd_gemm(cell, H, B, plan, XP, Wp, bhh, Hall, Hb, Call, gates):
    bs_h, off_h = _host_steps(plan)
    z = _zeros_bf16(XP.device, max(B * H, 4 * H))
    check(lib().sn_recur_fwd_gemm(cell, H, B, ctypes.cast(bs_h, ctypes.c_void_p), ctypes.cast(off_h, ctypes.c_void_p),
                                  plan.T, _ptr(_req(XP)), _ptr(_req(Wp, torch.bfloat16)), _ptr(bhh), _ptr(Hall),
                                  _ptr(_req(Hb, torch.bfloat16)), _ptr(_req(Call)), _ptr(gates), _ptr(z), _stream()),
          "sn_recur_fwd_gemm")
    LAUNCHES[0] += plan.T - 1


def recur_hprev(Hb, d, N, H, Hprevb):
    check(lib().sn_recur_hprev(_ptr(_req(Hb, torch.bfloat16)), _ptr(d["row_b"]), _ptr(d["row_t"]), _ptr(d["off"]), N, H,
                               _ptr(_req(Hprevb, torch.bfloat16)), _stream()), "sn_recur_hprev")


def recur_bwd_gemm(cell, H, B, plan, Whh_b, Call, gates, dHall, dZ, dZb, dc_carry):
    bs_h, off_h = _host_steps(plan)
    z = _zeros_bf16(dZb.device, max(B * H, 4 * H))
    check(lib().sn_recur_bwd_gemm(cell, H, B, ctypes.cast(bs_h, ctypes.c_void_p), ctypes.cast(off_h, ctypes.c_void_p),
                                  plan.T, _ptr(_req(Whh_b, torch.bfloat16)), _ptr(_req(Call)), _ptr(_req(gates)),
                                  _ptr(_req(dHall)), _ptr(dZ), _ptr(_req(dZb, torch.bfloat16)), _ptr(_req(dc_carry)),
                                  _ptr(z), _stream()), "sn_recur_bwd_gemm")
    LAUNCHES[0] += plan.T


def adam_clamp_dev(p, g, m, v, ranges, step_idx, steps_dev, lr_dev, coef_ws, beta1, beta2, eps, clip, max_ctas=0):
    """Clamp + Adam with step counters / learning rate in device memory (CUDA-graph replayable).  ``max_ctas`` > 0 caps
    the grid (a bucket updated next to the critical chain); it changes no result."""
    n = len(ranges)
    for i0 in range(0, n, 48):
        k = min(48, n - i0)
        R = (ctypes.c_int64 * (2 * k))()
        S = (ctypes.c_int32 * k)()
        for i in range(k):
            R[2 * i], R[2 * i + 1] = ranges[i0 + i]
            S[i] = step_idx[i0 + i]
        # (coefficient slots are indexed by step_idx: one work space serves every call, also concurrent ones)
        check(lib().sn_adam_clamp_dev_ex(_ptr(_req(p)), _ptr(_req(g)), _ptr(_req(m)), _ptr(_req(v)), k,
                                         ctypes.cast(R, ctypes.c_void_p), ctypes.cast(S, ctypes.c_void_p),
                                         _ptr(steps_dev), _ptr(lr_dev), _ptr(coef_ws), beta1, beta2, eps, clip,
                                         int(max_ctas), _stream()), "sn_adam_clamp_dev")


def enable_peer_access(peer_device):
    _check(lib().sn_enable_peer_access(int(peer_device)), "sn_enable_peer_access")


def dp_adam_fused(world, rank, grad_ptrs, param_ptrs, pad_ptrs, m, v, ranges, step_idx, steps_dev, lr_dev, coef_ws,
                  beta1, beta2, eps, clip):
    """Fused reduce-scatter + clamp/Adam + all-gather over peer memory (sn_dp_adam_fused)."""
    if len(ranges) > 48:            # each call is also a cross-GPU barrier; batches of <= 48 ranges
        for i0 in range(0, len(ranges), 48):
            dp_adam_fused(world, rank, grad_ptrs, param_ptrs, pad_ptrs, m, v, ranges[i0:i0 + 48],
                          step_idx[i0:i0 + 48], steps_dev, lr_dev, coef_ws, beta1, beta2, eps, clip)
        return
    n = len(ranges)
    G = (ctypes.c_void_p * world)(*grad_ptrs)
    Pp = (ctypes.c_void_p * world)(*param_ptrs)
    D = (ctypes.c_void_p * world)(*pad_ptrs)
    R = (ctypes.c_int64 * (2 * max(n, 1)))()
    S = (ctypes.c_int32 * max(n, 1))()
    for i in range(n):
        R[2 * i], R[2 * i + 1] = ranges[i]
        S[i] = step_idx[i]
    check(lib().sn_dp_adam_fused(world, rank, ctypes.cast(G, ctypes.c_void_p), ctypes.cast(Pp, ctypes.c_void_p),
                                 ctypes.cast(D, ctypes.c_void_p), _ptr(_req(m)), _ptr(_req(v)), n,
                                 ctypes.cast(R, ctypes.c_void_p), ctypes.cast(S, ctypes.c_void_p), _ptr(steps_dev),
                                 _ptr(lr_dev), _ptr(coef_ws), beta1, beta2, eps, clip, _stream()), "sn_dp_adam_fused")


DP_MAX_RANGES = 128      # AdamRanges::MAX (sn_elementwise.cu)


def merge_adjacent(ranges):
    """[(offset, length)] sorted with touching neighbours merged."""
    merged = []
    for off, n in sorted(ranges):
        if merged and merged[-1][0] + merged[-1][1] == off:
            merged[-1] = (merged[-1][0], merged[-1][1] + n)
        else:
            merged.append((off, n))
    return merged


def dp_slot_elems(arena_elems, world):
    return int(_lib.load().sn_dp_slot_elems(int(arena_elems), int(world)))      # host arithmetic: no device needed


def _ranges_c(ranges, step_idx=None):
    n = len(ranges)
    R = (ctypes.c_int64 * (2 * max(n, 1)))()
    S = (ctypes.c_int32 * max(n, 1))()
    for i in range(n):
        R[2 * i], R[2 * i + 1] = ranges[i]
        if step_idx is not None:
            S[i] = step_idx[i]
    return R, S


def dp_push(world, rank, grad, recv_ptrs, slot_elems, elem_size, pad_ptrs, ranges, max_ctas=0):
    """Push-form exchange, part 1 (sn_dp_push): non-blocking send of my gradients of foreign chunks + ARRIVE flags."""
    merged = merge_adjacent(ranges)      # adjacent ranges travel as one (the push has no per-parameter state)
    if len(merged) > DP_MAX_RANGES:
        raise RuntimeError("dp_push: more than %d ranges in one bucket (each call raises the bucket's flags once)" % DP_MAX_RANGES)
    R, _ = _ranges_c(merged)
    Rv = (ctypes.c_void_p * world)(*recv_ptrs)
    D = (ctypes.c_void_p * world)(*pad_ptrs)
    check(lib().sn_dp_push(world, rank, _ptr(_req(grad)), ctypes.cast(Rv, ctypes.c_void_p), int(slot_elems),
                           int(elem_size), ctypes.cast(D, ctypes.c_void_p), len(merged),
                           ctypes.cast(R, ctypes.c_void_p), int(max_ctas), _stream()), "sn_dp_push")


def dp_adam_recv(world, rank, grad, param_ptrs, recv, slot_elems, elem_size, pad_ptrs, wait_pads, m, v, ranges, step_idx,
                 steps_dev, lr_dev, coef_ws, beta1, beta2, eps, clip, max_ctas=0):
    """Push-form exchange, part 2 (sn_dp_adam_recv): wait for the pushes, reduce, clamp/Adam, parameter all-gather."""
    if len(ranges) > DP_MAX_RANGES:
        raise RuntimeError("dp_adam_recv: more than %d ranges in one call" % DP_MAX_RANGES)
    R, S = _ranges_c(ranges, step_idx)
    Pp = (ctypes.c_void_p * world)(*param_ptrs)
    D = (ctypes.c_void_p * world)(*pad_ptrs)
    Wp = (ctypes.c_void_p * len(wait_pads))(*wait_pads)
    check(lib().sn_dp_adam_recv(world, rank, _ptr(_req(grad)), ctypes.cast(Pp, ctypes.c_void_p), ctypes.c_void_p(recv.data_ptr()),
                                int(slot_elems), int(elem_size), ctypes.cast(D, ctypes.c_void_p),
                                ctypes.cast(Wp, ctypes.c_void_p), len(wait_pads), _ptr(_req(m)), _ptr(_req(v)),
                                len(ranges), ctypes.cast(R, ctypes.c_void_p), ctypes.cast(S, ctypes.c_void_p),
                                _ptr(steps_dev), _ptr(lr_dev), _ptr(coef_ws), beta1, beta2, eps, clip, int(max_ctas),
                                _stream()), "sn_dp_adam_recv")


def ipc_export(t):
    """(handle bytes, byte offset) describing tensor ``t``'s device memory for another process."""
    h = (ctypes.c_uint8 * 64)()
    off = ctypes.c_int64(0)
    _check(lib().sn_ipc_export(ctypes.c_void_p(t.data_ptr()), ctypes.cast(h, ctypes.c_void_p), ctypes.byref(off)),
           "sn_ipc_export")
    return bytes(h), off.value


def ipc_open(handle):
    """Map an exported allocation into this process (peer mapping of the current device); returns its base."""
    h = (ctypes.c_uint8 * 64).from_buffer_copy(handle)
    base = ctypes.c_void_p(0)
    _check(lib().sn_ipc_open(ctypes.cast(h, ctypes.c_void_p), ctypes.byref(base)), "sn_ipc_open")
    return base.value


# ---- encoder tail -> decoder hand-off (SURVEY.md section 8 f1) -----------------------------------------------------
def pool_nhwc_fwd(x, S, out, out_bf16=None, mean=None):
    """AdaptiveAvgPool2d((S,S)) + permute(0,2,3,1) of an NCHW map in one pass (stylenet/model_att.py:24-28)."""
    B, D, h, w = x.shape
    check(lib().sn_pool_nhwc_fwd(_ptr(_req(x)), B, D, h, w, S, _ptr(_req(out)), _ptr(out_bf16), _ptr(mean), _stream()),
          "sn_pool_nhwc_fwd")
    return out


def pool_nhwc_bwd(dout, h, w, dx):
    B, S, _, D = dout.shape
    check(lib().sn_pool_nhwc_bwd(_ptr(_req(dout)), B, D, h, w, S, _ptr(_req(dx)), _stream()), "sn_pool_nhwc_bwd")
    return dx


def bn1d_fwd(x, gamma, beta, running_mean, running_var, momentum, eps, training, y, save_mean, save_invstd):
    B, E = x.shape
    check(lib().sn_bn1d_fwd(_ptr(_req(x)), B, E, _ptr(gamma), _ptr(beta), _ptr(running_mean), _ptr(running_var),
                            float(momentum), float(eps), 1 if training else 0, _ptr(_req(y)), _ptr(save_mean),
                            _ptr(save_invstd), _stream()), "sn_bn1d_fwd")


def bn1d_bwd(x, dy, gamma, save_mean, save_invstd, training, dx, dgamma, dbeta):
    B, E = x.shape
    check(lib().sn_bn1d_bwd(_ptr(_req(x)), _ptr(_req(dy)), B, E, _ptr(gamma), _ptr(save_mean), _ptr(save_invstd),
                            1 if training else 0, _ptr(dx), _ptr(dgamma), _ptr(dbeta), _stream()), "sn_bn1d_bwd")


# ---- decode steps on few rows (matrix-vector kernels, sn_decode.cu) -------------------------------------------------
SKINNY_MAX_ROWS = 16


SKINNY_LINEAR_MAX_ROWS = 256       # sn_skinny_linear beyond 16 rows: chunks of <= 16 rows along grid.y


def skinny_linear(W, X, out, R, bias=None, group_n=0, group_x=0, K=None, x_rows=None):
    """out[:R] = X[:R] W^T + bias for R <= SKINNY_LINEAR_MAX_ROWS rows (more than 16 in row chunks, each as a call on
    its rows alone); W [N, K] fp32 (row pitch W.stride(0)); grouped form see sn100.h.
    ``x_rows`` (int32 [R]): gather the input rows, X[x_rows[r]] (embedding lookup folded into the stage)."""
    N = W.shape[0]
    K = K if K is not None else W.shape[1]
    check(lib().sn_skinny_linear(_ptr(_req(W)), W.stride(0), N, K, _ptr(_req(X)), X.stride(0), R, group_n, group_x,
                                 _ptr(bias), _ptr(_req(out)), out.stride(0), _ptr(x_rows), _stream()), "sn_skinny_linear")
    return out


def decode_cell(cell, H, R, Wx, Kx, X, group_x, bx, Wh, bh, h_prev, c_prev, src_row, h_out, c_out, x_rows=None):
    check(lib().sn_decode_cell(cell, H, R, _ptr(_req(Wx)), Wx.stride(0), Kx, _ptr(_req(X)), X.stride(0), group_x,
                               _ptr(bx), _ptr(_req(Wh)), _ptr(bh), _ptr(_req(h_prev)), _ptr(_req(c_prev)),
                               _ptr(src_row), _ptr(x_rows), _ptr(_req(h_out)), _ptr(_req(c_out)), _stream()),
          "sn_decode_cell")


def decode_cell_groups(cell, H, row_off, rows_max, Wx, Kx, X, group_x, bx, Wh, bh, h_prev, c_prev, src_row, h_out,
                       c_out, x_rows=None):
    """decode_cell for G = len(row_off) - 1 <= 4 row groups in one launch: group g (rows [row_off[g], row_off[g+1]),
    ``row_off`` a device int32 tensor) uses Wx[g] / bx[g] of ``Wx`` [G, 4H, Kx] and ``bx`` [G, 4H]."""
    G = row_off.numel() - 1
    if Wx.dim() != 3 or Wx.shape[0] != G or bx.shape[0] != G:
        raise ValueError("decode_cell_groups: Wx / bx need one leading entry per group (%d)" % G)
    check(lib().sn_decode_cell_groups(cell, H, G, _ptr(_req(row_off, torch.int32)), int(rows_max), _ptr(_req(Wx)),
                                      Wx.stride(1), Wx.stride(0), Kx, _ptr(_req(X)), X.stride(0), group_x, _ptr(_req(bx)),
                                      bx.stride(0), _ptr(_req(Wh)), _ptr(bh), _ptr(_req(h_prev)), _ptr(_req(c_prev)),
                                      _ptr(src_row), _ptr(x_rows), _ptr(_req(h_out)), _ptr(_req(c_out)), _stream()),
          "sn_decode_cell_groups")


def bleu_counts(hyp_tok, hyp_off, ref_tok, ref_off, ref_group, max_sentence_len, max_group_tokens):
    """Per-hypothesis BLEU statistics (sn_bleu_counts): int32 [n_hyp, 10], column layout in include/sn100.h.
    Token arrays int32, offset arrays int64, all CUDA tensors (CSR: ``hyp_off`` / ``ref_group`` have n_hyp + 1 entries,
    ``ref_off`` one more than the number of references)."""
    n_hyp = hyp_off.numel() - 1
    stats = torch.empty(n_hyp, 10, dtype=torch.int32, device=hyp_off.device)
    check(lib().sn_bleu_counts(_ptr(_req(hyp_tok, torch.int32)), _ptr(_req(hyp_off, torch.int64)), n_hyp,
                               _ptr(_req(ref_tok, torch.int32)), _ptr(_req(ref_off, torch.int64)),
                               _ptr(_req(ref_group, torch.int64)), int(max_sentence_len), int(max_group_tokens),
                               _ptr(_req(stats, torch.int32)), _stream()), "sn_bleu_counts")
    return stats


def cider_df(ref_tok, ref_off, ref_group, n, max_sentence_len, max_group_tokens, capacity, err):
    """CIDEr-D document frequencies (sn_cider_df) of orders 1..n into a new table of ``capacity`` slots (a power of two):
    returns (keys int32 [capacity, 4], counts int32 [capacity]), layout in include/sn100.h.  Inputs as for
    ``bleu_counts`` without the hypotheses.  ``err`` (int32 CUDA tensor) receives the error bits; read it on the host
    before trusting the table."""
    dev = ref_group.device
    keys = torch.empty(int(capacity), 4, dtype=torch.int32, device=dev)
    counts = torch.empty(int(capacity), dtype=torch.int32, device=dev)
    check(lib().sn_cider_df(_ptr(_req(ref_tok, torch.int32)), _ptr(_req(ref_off, torch.int64)),
                            _ptr(_req(ref_group, torch.int64)), ref_group.numel() - 1, int(n), int(max_sentence_len),
                            int(max_group_tokens), _ptr(keys), _ptr(counts), int(capacity),
                            _ptr(_req(err, torch.int32)), _stream()), "sn_cider_df")
    return keys, counts


def cider_scores(hyp_tok, hyp_off, ref_tok, ref_off, ref_group, n, sigma, max_sentence_len, max_group_tokens, keys,
                 counts, out=None):
    """CIDEr-D per image (sn_cider_scores) against the table of ``cider_df``: returns (scores float64 [n_img], per-order
    sums float64 [n_img, 4]).  ``out``: a float64 [n_img] CUDA tensor to write the scores into."""
    n_img = hyp_off.numel() - 1
    scores = out if out is not None else torch.empty(n_img, dtype=torch.float64, device=hyp_off.device)
    per_order = torch.empty(n_img, 4, dtype=torch.float64, device=hyp_off.device)
    check(lib().sn_cider_scores(_ptr(_req(hyp_tok, torch.int32)), _ptr(_req(hyp_off, torch.int64)), n_img,
                                _ptr(_req(ref_tok, torch.int32)), _ptr(_req(ref_off, torch.int64)),
                                _ptr(_req(ref_group, torch.int64)), int(n), float(sigma), int(max_sentence_len),
                                int(max_group_tokens), _ptr(_req(keys, torch.int32)), _ptr(_req(counts, torch.int32)),
                                keys.shape[0], _ptr(_req(scores, torch.float64)), _ptr(per_order), _stream()),
          "sn_cider_scores")
    return scores, per_order


def cider_scores_rows(seqs, lengths, img, end_token, n_corpus, ref_tok, ref_off, ref_group, n, sigma, max_sentence_len,
                      max_group_tokens, keys, counts):
    """CIDEr-D of sampled captions (sn_cider_scores_rows): row r = seqs[r, 1:lengths[r]] without a final end_token,
    against the references of corpus image img[r], idf from the table of ``cider_df`` and log(n_corpus).  Returns
    float64 [R]."""
    R = seqs.shape[0]
    scores = torch.empty(R, dtype=torch.float64, device=seqs.device)
    check(lib().sn_cider_scores_rows(_ptr(_req(seqs, torch.int64)), seqs.stride(0), _ptr(_req(lengths, torch.int64)), R,
                                     int(end_token), _ptr(_req(img, torch.int64)), int(n_corpus),
                                     _ptr(_req(ref_tok, torch.int32)), _ptr(_req(ref_off, torch.int64)),
                                     _ptr(_req(ref_group, torch.int64)), int(n), float(sigma), int(max_sentence_len),
                                     int(max_group_tokens), _ptr(_req(keys, torch.int32)),
                                     _ptr(_req(counts, torch.int32)), keys.shape[0], _ptr(scores), _stream()),
          "sn_cider_scores_rows")
    return scores


def rouge_l(hyp_tok, hyp_off, ref_tok, ref_off, ref_group, max_sentence_len, beta2, out=None):
    """ROUGE-L per image (sn_rouge_l): float64 [n_img].  Inputs as for ``bleu_counts``; ``beta2`` is the scorer's
    beta ** 2.  ``out``: a float64 [n_img] CUDA tensor to write the scores into."""
    n_img = hyp_off.numel() - 1
    scores = out if out is not None else torch.empty(n_img, dtype=torch.float64, device=hyp_off.device)
    check(lib().sn_rouge_l(_ptr(_req(hyp_tok, torch.int32)), _ptr(_req(hyp_off, torch.int64)), n_img,
                           _ptr(_req(ref_tok, torch.int32)), _ptr(_req(ref_off, torch.int64)),
                           _ptr(_req(ref_group, torch.int64)), int(max_sentence_len), float(beta2),
                           _ptr(_req(scores, torch.float64)), _stream()), "sn_rouge_l")
    return scores


def rouge_l_rows(seqs, lengths, img, end_token, n_corpus, ref_tok, ref_off, ref_group, max_sentence_len, beta2):
    """ROUGE-L of sampled captions (sn_rouge_l_rows): row r = seqs[r, 1:lengths[r]] without a final end_token, against
    the references of corpus image img[r].  Returns float64 [R]."""
    R = seqs.shape[0]
    scores = torch.empty(R, dtype=torch.float64, device=seqs.device)
    check(lib().sn_rouge_l_rows(_ptr(_req(seqs, torch.int64)), seqs.stride(0), _ptr(_req(lengths, torch.int64)), R,
                                int(end_token), _ptr(_req(img, torch.int64)), int(n_corpus),
                                _ptr(_req(ref_tok, torch.int32)), _ptr(_req(ref_off, torch.int64)),
                                _ptr(_req(ref_group, torch.int64)), int(max_sentence_len), float(beta2), _ptr(scores),
                                _stream()), "sn_rouge_l_rows")
    return scores


def sample_step(logits, V, R, max_len, end_token, temperature, greedy, seed_dev, step_dev, prev_word, seqs, lengths,
                logprob, done, n_unfinished):
    """K12: one sampling-decode draw per live row of ``logits`` (Gumbel-max at ``temperature``, or the arg-max), with
    the row bookkeeping on the device (include/sn100.h)."""
    check(lib().sn_sample_step(_ptr(_req(logits)), logits.stride(0), V, R, max_len, int(end_token), float(temperature),
                               1 if greedy else 0, _ptr(_req(seed_dev, torch.int64)), _ptr(_req(step_dev, torch.int32)),
                               _ptr(_req(prev_word, torch.int32)), _ptr(_req(seqs, torch.int64)),
                               _ptr(_req(lengths, torch.int64)), _ptr(_req(logprob)), _ptr(_req(done, torch.int32)),
                               _ptr(_req(n_unfinished, torch.int32)), _stream()), "sn_sample_step")
    LAUNCHES[0] += 1


def gate_wait(flag3, timeout_us=300):
    """Queue a one-thread kernel that returns once the cluster-form reverse recurrence (given the same flag) is resident."""
    check(lib().sn_gate_wait(_ptr(_req(flag3, torch.int32)), int(timeout_us), _stream()), "sn_gate_wait")
