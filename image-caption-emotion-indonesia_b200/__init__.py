"""B200-native caption-decoder hot path of deryrahman/image-caption-emotion-indonesia.

The reference's PyTorch module surface (DecoderFactoredLSTM / DecoderFactoredLSTMAtt / DecoderRNN /
DecoderRNNAtt: same constructor arguments, parameter names, forward / forward_step / sample signatures)
over hand-written sm_100a CUDA in libsn100.so (C ABI: include/sn100.h).  No Triton, no multi-backend
dispatch, no CPU fallback: ops raise if the library is missing or the device is not sm_100.
"""
from .decoders import DecoderFactoredLSTM, DecoderRNN, STYLES  # noqa: F401
from .optim import FusedClampAdam  # noqa: F401
from .packing import PackPlan, batch_sizes_from_lengths, get_plan, shard_lengths  # noqa: F401
from . import ops  # noqa: F401
from .dp import DataParallelTrainer, GradSync, merged_ranges  # noqa: F401
from .graph import GraphedTrainStep  # noqa: F401
from .stack import DecoderFactoredLSTMStack, MultitaskSchedule  # noqa: F401
from .encoders import EncoderCNN, EncoderCNNAtt  # noqa: F401
from . import bleu, checkpoint, cider, evaluate, seq2seq  # noqa: F401

try:  # attention variants
    from .decoders_att import DecoderFactoredLSTMAtt, DecoderRNNAtt  # noqa: F401
except ImportError:  # pragma: no cover - during bring-up
    pass
