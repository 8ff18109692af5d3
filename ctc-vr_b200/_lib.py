"""ctypes binding of libctcvr.so (include/ctcvr.h).  There is NO fallback: if the library is
missing or a call fails, RuntimeError is raised (the reference's train loop catches RuntimeError,
rnnt_train.py:139-141)."""
import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_long, c_size_t, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libctcvr.so")
_lib = None

P, I, F, Z = c_void_p, c_int, c_float, c_size_t


class DecoderWeights(ctypes.Structure):
    """Mirror of `ctcvr_decoder_weights` (include/ctcvr.h)."""
    _fields_ = [(n, c_void_p) for n in ("gate_tok", "w_hh_t", "w_ih_t", "b_gate", "proj_t", "proj_b",
                                        "pred_ffn_t", "pred_ffn_b", "out_t", "out_b")] + \
               [(n, c_int) for n in ("V", "H", "L", "P", "D", "activation")]   # activation: CTCVR_ACT_*, 0 = tanh


_SIGS = {
    "ctcvr_last_error": (c_char_p, []),
    "ctcvr_version": (I, []),
    "ctcvr_launch_count": (ctypes.c_ulonglong, []),
    "ctcvr_debug_tc_error": (ctypes.c_uint, []),
    "ctcvr_debug_set_prof": (None, [P]),
    "ctcvr_debug_set_mode": (None, [I]),
    "ctcvr_joint_logits": (I, [P, P, P, P, P, I, I, I, I, I, P]),
    "ctcvr_joint_rnnt_fwd_ws_bytes": (Z, [I, I, I, I, I, I]),
    "ctcvr_joint_rnnt_fwd": (I, [P, P, P, P, P, P, P, P, P, P, I, I, I, I, I, I, I, P, Z, P]),
    "ctcvr_rnnt_lattice": (I, [P, P, P, P, P, P, P, I, I, I, P]),
    "ctcvr_joint_rnnt_bwd_ws_bytes": (Z, [I, I, I, I, I, I]),
    "ctcvr_joint_rnnt_bwd": (I, [P] * 14 + [F] + [P] * 4 + [I] * 7 + [P, Z, P]),
    "ctcvr_joint_tc_supported": (I, [I, I, I]),
    "ctcvr_joint_rnnt_fwd_bf16in": (I, [P, P, P, P, P, P, P, P, P, P, I, I, I, I, I, I, P, Z, P]),
    "ctcvr_joint_rnnt_bwd_bf16in": (I, [P] * 14 + [F] + [P] * 4 + [I] * 6 + [P, Z, P]),
    "ctcvr_rnnt_prologue": (I, [P, P, I, P, I, I, I, I, P, P, P, P, P]),
    "ctcvr_loss_combine": (I, [P, I, P, F, F, P, P]),
    "ctcvr_cer_ws_bytes": (Z, [I, I, I]),
    "ctcvr_cer_batch": (I, [P, P, I, P, P, I, I, P, Z, P, P]),
    "ctcvr_lstm_seq_supported": (I, [I, I]),
    "ctcvr_lstm_seq_ws_bytes": (Z, [I, I]),
    "ctcvr_lstm_seq_fwd": (I, [P] * 9 + [I, I, I, P, Z, P]),
    "ctcvr_lstm_seq_bwd": (I, [P] * 10 + [I, I, I, P, Z, P]),
    "ctcvr_split_tf32": (I, [P, P, c_long, c_long, I, I, P]),
    "ctcvr_peer_create": (I, [I, I, Z, P, P]),
    "ctcvr_peer_connect": (I, [P, P, P]),
    "ctcvr_peer_local_buffer": (P, [P]),
    "ctcvr_peer_set_timeout_ms": (I, [P, c_long]),
    "ctcvr_peer_allreduce": (I, [P, P, P, I, I, P]),
    "ctcvr_peer_destroy": (I, [P]),
    "ctcvr_rnnt_loss_dense_ws_bytes": (Z, [I, I, I]),
    "ctcvr_rnnt_loss_dense": (I, [P, P, P, P, P, P, I, I, I, I, I, F, P, Z, P]),
    "ctcvr_log_softmax": (I, [P, P, c_long, I, P]),
    "ctcvr_ctc_loss_ws_bytes": (Z, [I, I, I]),
    "ctcvr_ctc_loss": (I, [P, P, P, P, P, P, P, I, I, I, I, I, I, P, Z, P]),
    "ctcvr_ctc_greedy": (I, [P, P, P, P, I, I, I, I, P]),
    "ctcvr_rnnt_viterbi_ws_bytes": (Z, [I, I, I]),
    "ctcvr_rnnt_viterbi": (I, [P, P, P, P, P, P, P, I, I, I, P, Z, P]),
    "ctcvr_ctc_viterbi_ws_bytes": (Z, [I, I, I]),
    "ctcvr_ctc_viterbi": (I, [P, P, P, P, P, P, P, P, I, I, I, I, I, P, Z, P]),
    "ctcvr_rnnt_greedy_ws_bytes": (Z, [P, I]),
    "ctcvr_rnnt_greedy": (I, [P, P, P, P, P, P, P, P, I, I, I, I, I, P, Z, P]),
    "ctcvr_rnnt_beam_state_bytes": (Z, [P, I, I, I]),
    "ctcvr_rnnt_beam_reset": (I, [P, P, I, I, I, P]),
    "ctcvr_rnnt_beam_chunk": (I, [P, P, I, P, I, I, I, I, P, P, P, P, P, P, P]),
    "ctcvr_rnnt_beam_reset_batch": (I, [P, P, I, I, I, I, P]),
    "ctcvr_rnnt_beam_chunk_batch": (I, [P, P, P, I, I, P, I, I, I, I, P, P, P, P, P, P, P]),
    "ctcvr_rnnt_prefix_beam_ws_bytes": (Z, [P, I, I]),
    "ctcvr_rnnt_prefix_beam": (I, [P, P, P, I, I, I, F, F, P, P, P, P, P, Z, P]),
    "ctcvr_rnnt_prefix_beam_batch": (I, [P, P, P, P, I, I, I, I, F, F, P, P, P, P, P, Z, P]),
    "ctcvr_ctc_prefix_beam_ws_bytes": (Z, [I, I, I, I]),
    "ctcvr_ctc_prefix_beam": (I, [P, P, I, I, I, I, I, P, P, P, P, P, P, Z, P]),
}
EXPORTS = tuple(_SIGS)


def lib():
    """Load libctcvr.so (built in-tree by `python ctc-vr_b200/build.py`)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"ctcvr_b200: {LIB_PATH} is missing - build it with `python ctc-vr_b200/build.py` "
                               "(there is no CPU / PyTorch fallback)")
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def ptr(t):
    return None if t is None else c_void_p(t.data_ptr())


def stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def call(name, *args):
    """Invoke an int-returning entry point; non-zero -> RuntimeError(ctcvr_last_error())."""
    l = lib()
    rc = getattr(l, name)(*args)
    if rc != 0:
        raise RuntimeError(f"{name}: {l.ctcvr_last_error().decode()}")


def query(name, *args):
    return getattr(lib(), name)(*args)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("ctcvr_b200 ops run on CUDA (B200) tensors only; there is no CPU path")
