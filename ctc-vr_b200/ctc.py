"""CTC heads with the reference's constructors / parameter names / return values.
  CTC       — model/rnnt_model.py:11-80   (reduction 'sum' then / batch)
  OnlineCTC — model/online_rnnt_model.py:14-38 (reduction 'mean')
Kept quirk: F.dropout(p) is called without `training=`, i.e. it is active in eval too
(rnnt_model.py:52, online_rnnt_model.py:27-28)."""
from typing import Tuple

import torch
import torch.nn.functional as F

from . import functional as CF


class CTC(torch.nn.Module):
    def __init__(self, odim: int, encoder_output_size: int, dropout_rate: float = 0.0, reduce: bool = True,
                 blank_id: int = 0):
        super().__init__()
        self.dropout_rate = dropout_rate
        self.ctc_lo = torch.nn.Linear(encoder_output_size, odim)
        self.reduce = reduce
        self.blank_id = blank_id

    def forward(self, hs_pad, hlens, ys_pad, ys_lens) -> Tuple[torch.Tensor, torch.Tensor]:
        logits = self.ctc_lo(F.dropout(hs_pad, p=self.dropout_rate))
        loss, ys_hat = CF.ctc_loss_from_logits(logits, ys_pad, hlens, ys_lens, self.blank_id,
                                               "sum" if self.reduce else "none", True)
        loss = loss / logits.size(0)          # "Batch-size average" (rnnt_model.py:57-58)
        return loss, ys_hat

    def log_softmax(self, hs_pad):
        return CF.log_softmax_rows(self.ctc_lo(hs_pad))

    @torch.no_grad()
    def forced_align(self, hs_pad, hlens, ys_pad, ys_lens):
        """Best CTC alignment of ys_pad [B,Umax] on log_softmax(ctc_lo(hs_pad)) (no dropout):
        functional.ctc_forced_align -> (labels [B,T], frame_logprobs [B,T], scores [B], spans [B,Umax,2])."""
        return CF.ctc_forced_align(self.log_softmax(hs_pad), ys_pad, hlens, ys_lens, self.blank_id)

    def argmax(self, hs_pad):
        return torch.argmax(self.ctc_lo(hs_pad), dim=2)


class OnlineCTC(torch.nn.Module):
    def __init__(self, vocab_size: int, encoder_output_size: int, dropout_rate: float = 0.0, blank_id: int = 0):
        super().__init__()
        self.ctc_lo = torch.nn.Linear(encoder_output_size, vocab_size)
        self.dropout_rate = dropout_rate
        self.blank_id = blank_id

    def forward(self, hs_pad, hlens, ys_pad, ys_lens) -> Tuple[torch.Tensor, torch.Tensor]:
        logits = self.ctc_lo(F.dropout(hs_pad, p=self.dropout_rate))
        return CF.ctc_loss_from_logits(logits, ys_pad, hlens, ys_lens, self.blank_id, "mean", True)

    def log_softmax(self, hs_pad):
        return CF.log_softmax_rows(self.ctc_lo(hs_pad))

    @torch.no_grad()
    def forced_align(self, hs_pad, hlens, ys_pad, ys_lens):
        """Best CTC alignment of ys_pad [B,Umax] on log_softmax(ctc_lo(hs_pad)) (no dropout):
        functional.ctc_forced_align -> (labels [B,T], frame_logprobs [B,T], scores [B], spans [B,Umax,2])."""
        return CF.ctc_forced_align(self.log_softmax(hs_pad), ys_pad, hlens, ys_lens, self.blank_id)

    def argmax(self, hs_pad):
        return torch.argmax(self.ctc_lo(hs_pad), dim=2)
