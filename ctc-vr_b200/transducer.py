"""Transducer wrapper with the reference's constructor, attributes and method signatures
(model/component/transducer.py:73-189); `_compute_rnnt_loss` is the fused seam."""
from typing import Dict, List, Optional

import torch
from torch import nn

from . import decode as D


def add_blank(text: torch.Tensor, blank: int, ignore_id: int) -> torch.Tensor:
    """model/component/transducer.py:8-19: prepend blank (ignore_id is NOT remapped there)."""
    ys_in = torch.zeros((text.size(0), text.size(1) + 1), dtype=text.dtype, device=text.device)
    ys_in[:, 0] = blank
    ys_in[:, 1:] = text
    return ys_in


basic_greedy_search = D.basic_greedy_search


class Transducer(nn.Module):
    def __init__(self, vocab_size: int, blank: int, encoder: nn.Module, predictor: nn.Module, joint: nn.Module,
                 ctc: Optional[nn.Module] = None, ctc_weight: float = 0.3, ignore_id: int = -1,
                 transducer_weight: float = 0.7, precision: str = "fp32") -> None:
        super().__init__()
        assert ctc_weight + transducer_weight == 1.0
        self.vocab_size = vocab_size
        self.blank = blank
        self.ignore_id = ignore_id
        self.ctc_weight = ctc_weight
        self.transducer_weight = transducer_weight
        self.encoder = encoder
        self.predictor = predictor
        self.joint = joint
        self.ctc = ctc
        self.precision = precision

    def forward(self, batch: dict, device: torch.device) -> Dict[str, Optional[torch.Tensor]]:
        speech = batch["feats"].to(device)
        speech_lengths = batch["feats_lengths"].to(device)
        text = batch["target"].to(device)
        text_lengths = batch["target_lengths"].to(device)
        encoder_out, encoder_mask = self.encoder(speech, speech_lengths)
        encoder_out_lens = encoder_mask.squeeze(1).sum(1)
        loss_rnnt = self._compute_rnnt_loss(encoder_out, encoder_out_lens, text, text_lengths)
        loss = self.transducer_weight * loss_rnnt
        loss_ctc: Optional[torch.Tensor] = None
        if self.ctc_weight != 0.0 and self.ctc is not None:
            loss_ctc, _ = self.ctc(encoder_out, encoder_out_lens, text, text_lengths)
            loss = loss + self.ctc_weight * loss_ctc.sum()
        return {"loss": loss, "loss_ctc": loss_ctc, "loss_rnnt": loss_rnnt}

    def greedy_search(self, speech, speech_lengths, decoding_chunk_size: int = -1,
                      num_decoding_left_chunks: int = -1, n_steps: int = 64) -> List[List[int]]:
        assert speech.shape[0] == speech_lengths.shape[0]
        encoder_out, encoder_mask = self.encoder(speech, speech_lengths)
        encoder_out_lens = encoder_mask.squeeze(1).sum(1)
        return basic_greedy_search(self, encoder_out, encoder_out_lens, n_steps=n_steps)

    def _compute_rnnt_loss(self, encoder_out, encoder_out_lens, text, text_lengths) -> torch.Tensor:
        """transducer.py:161-189 with joint + log-softmax + lattice + gradients fused."""
        return compute_rnnt_loss(self, encoder_out, encoder_out_lens, text, text_lengths)


def rnnt_prologue(text, text_lengths, encoder_out_lens, blank: int, ignore_id: int):
    """add_blank + the ignore_id remap + the int32 casts of transducer.py:8-19,168,174-178 in one launch
    (`ctcvr_rnnt_prologue`): -> (ys_in int64 [B,U+1], targets int32 [B,U], logit_lengths int32, target_lengths int32)."""
    from ._lib import call, ptr, stream
    dev = text.device
    B, U = text.shape
    t64 = text if text.dtype == torch.int64 and text.is_contiguous() else text.to(torch.int64).contiguous()
    el = encoder_out_lens.to(device=dev, dtype=torch.int64).contiguous()
    tl = text_lengths.to(dev).contiguous()
    if tl.dtype not in (torch.int32, torch.int64):
        tl = tl.to(torch.int32)
    ys_in = torch.empty((B, U + 1), dtype=torch.int64, device=dev)
    targets = torch.empty((B, U), dtype=torch.int32, device=dev)
    t_len = torch.empty((B,), dtype=torch.int32, device=dev)
    u_len = torch.empty((B,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        call("ctcvr_rnnt_prologue", ptr(t64), ptr(tl), int(tl.dtype == torch.int64), ptr(el), B, U, int(blank), int(ignore_id),
             ptr(ys_in), ptr(targets), ptr(t_len), ptr(u_len), stream())
    return ys_in, targets, t_len, u_len


def compute_rnnt_loss(self, encoder_out, encoder_out_lens, text, text_lengths, clamp: float = -1.0):
    """Body shared with `patch.install()` (patch.py): works on the reference's own Transducer instance too."""
    if not text.is_cuda:
        raise RuntimeError("ctcvr_b200 ops run on CUDA (B200) tensors only; there is no CPU path")
    ys_in_pad, rnnt_text, t_len32, u_len32 = rnnt_prologue(text, text_lengths, encoder_out_lens, self.blank, self.ignore_id)
    predictor_out = self.predictor(ys_in_pad)
    joint = self.joint
    precision = getattr(self, "precision", "fp32")      # reference arithmetic unless the model opts into bf16
    from . import functional as CF
    from .joint import fused_joint_inputs, joint_activation
    act = joint_activation(joint)                       # tanh / relu / exact gelu, anything else raises
    # pre-join linears (if any), then the post-join linear folded into both sides (joint.fused_joint_inputs)
    if precision == "bf16" and encoder_out.is_cuda:
        with torch.autocast("cuda", dtype=torch.bfloat16):
            e, p = fused_joint_inputs(joint, encoder_out, predictor_out)
    else:
        e, p = fused_joint_inputs(joint, encoder_out, predictor_out)
    return CF.fused_joint_rnnt_loss(e, p, joint.ffn_out.weight, joint.ffn_out.bias, rnnt_text, t_len32, u_len32,
                                    self.blank, clamp, "mean", precision, activation=act)


@torch.no_grad()
def compute_rnnt_alignment(self, encoder_out, encoder_out_lens, text, text_lengths):
    """Forced alignment of `text` with the same prologue, predictor and joint as `compute_rnnt_loss` (works on the
    reference's own Transducer instance too).  Returns (frames [B,U] int32: the encoder frame of each token, -1 beyond
    its length; token_logprobs [B,U]; scores [B]: the best path's log-probability)."""
    if not text.is_cuda:
        raise RuntimeError("ctcvr_b200 ops run on CUDA (B200) tensors only; there is no CPU path")
    ys_in_pad, rnnt_text, t_len32, u_len32 = rnnt_prologue(text, text_lengths, encoder_out_lens, self.blank, self.ignore_id)
    predictor_out = self.predictor(ys_in_pad)
    joint = self.joint
    precision = getattr(self, "precision", "fp32")
    from . import functional as CF
    from .joint import fused_joint_inputs, joint_activation
    act = joint_activation(joint)
    if precision == "bf16" and encoder_out.is_cuda:
        with torch.autocast("cuda", dtype=torch.bfloat16):
            e, p = fused_joint_inputs(joint, encoder_out, predictor_out)
    else:
        e, p = fused_joint_inputs(joint, encoder_out, predictor_out)
    return CF.rnnt_forced_align(e, p, joint.ffn_out.weight, joint.ffn_out.bias, rnnt_text, t_len32, u_len32,
                                self.blank, precision, activation=act)
