"""Host logic of the tail schedule: which training steps take it (no GPU needed)."""
import pytest


def test_tail_schedule_selection():
    from icei_b200 import dp, ops
    old = ops.TAIL_SCHEDULE[0]
    try:
        ops.TAIL_SCHEDULE[0] = 1
        assert dp.tail_schedule(1, True)
        assert not dp.tail_schedule(1, False)        # fp32 mode / attention decoder: not bucketed
        assert not dp.tail_schedule(2, True)         # data-parallel exchange paths keep theirs
        assert not dp.tail_schedule(8, True)
        ops.TAIL_SCHEDULE[0] = 0
        assert not dp.tail_schedule(1, True)
    finally:
        ops.TAIL_SCHEDULE[0] = old


def test_early_embed_flag_only_for_teacher_forced_bf16_training():
    """forward_loss arms the early embedding plan only for a bf16 backward whose embedding holds no live gradient;
    _run_forward then takes it only when every step is teacher-forced (checked on the GPU)."""
    import torch
    import icei_b200 as sn
    dec = sn.DecoderFactoredLSTM(16, 32, 32, 50, 1)
    cap = torch.randint(4, 50, (2, 5))
    with pytest.raises(Exception):          # CPU tensors are refused before any flag is set
        dec.forward_loss(cap, [5, 5], torch.randn(2, 16), early_embed=True)
    assert not dec.__dict__.get("_emb_early", False)
