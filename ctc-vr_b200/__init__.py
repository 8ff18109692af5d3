"""ctcvr_b200 — B200 (sm_100a) implementation of the transducer hot path of CentaureaHO/CTC-VR.

Host side mirrors the reference's Python call surface (SURVEY.md §8b); all arithmetic runs in the
hand-written CUDA kernels of libctcvr.so through the C ABI of include/ctcvr.h.  There is no CPU path
and no fallback: ops raise RuntimeError without the library or without a CUDA device.
"""
from . import _lib  # noqa: F401
from . import functional  # noqa: F401
from . import patch  # noqa: F401
from .ctc import CTC, OnlineCTC  # noqa: F401
from .evaluate import calculate_cer, calculate_cer_batch  # noqa: F401
from .decode import (BeamHypothesis, OnlineBeamState, basic_greedy_search, beam_chunk_online, beam_search_batch,  # noqa: F401
                     greedy_batch, greedy_chunk, prefix_beam_search, prefix_beam_search_batch)
from .functional import (ctc_forced_align, ctc_greedy_search as ctc_greedy_hyps, ctc_loss_from_logits,  # noqa: F401
                         fused_joint_rnnt_loss, joint_logits, rnnt_forced_align, rnnt_loss, rnnt_viterbi)
from .graph import BucketedJointRnntStep, GraphedJointRnntStep  # noqa: F401
from .joint import TransducerJoint  # noqa: F401
from .predictor import RNNPredictor  # noqa: F401
from .search import DecodeResult, ctc_greedy_search, ctc_prefix_beam_search  # noqa: F401
from .transducer import Transducer, add_blank, compute_rnnt_alignment  # noqa: F401

__version__ = "0.1.0"
