"""tensorized_rnn_b200 -- B200-native (sm_100a) tensor-train LSTM / GRU recurrence.

Drop-in mirror of the recurrent path of onucharles/tensorized-rnn: `TTLSTM`, `TTGRU`,
`TTLinear` keep the reference's nn.Module API and state_dict layout; the time loop, the
TT-matrix contractions and BPTT run in hand-written CUDA kernels behind the C ABI of
`include/ttrnn_b200.h`.  CUDA only, FP32 only, no fallback.
"""
from .shapes import auto_shape, tt_shape
from .tensor_train import TensorTrain, transpose
from .initializers import glorot_initializer, random_matrix, matrix_with_random_cores
from .layers import TTLinear, TTLinearSet
from .rnn_utils import ActivGradLogger, av_norm
from .rnn import TTLSTM, TTLSTMCell, TTGRU, TTGRUCell, param_count
from .ge2e import GE2EHead, embed_normalize, ge2e_loss, gather_partials, partial_windows, segment_mean_normalize
from .dense import LSTM, LSTMCell, GRU, GRUCell
from .speaker_encoder import SpeakerEncoder

__all__ = ["auto_shape", "tt_shape", "TensorTrain", "transpose", "glorot_initializer", "random_matrix",
           "matrix_with_random_cores", "TTLinear", "TTLinearSet", "ActivGradLogger", "av_norm", "TTLSTM", "TTLSTMCell", "TTGRU", "TTGRUCell", "param_count",
           "GE2EHead", "embed_normalize", "ge2e_loss", "partial_windows", "gather_partials", "segment_mean_normalize",
           "LSTM", "LSTMCell", "GRU", "GRUCell", "SpeakerEncoder"]
from . import compat  # noqa: E402,F401  (compat.patch_reference(): switch a reference checkout over)

__version__ = "0.2.0"
