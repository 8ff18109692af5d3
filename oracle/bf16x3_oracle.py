"""Oracle (TEST INFRASTRUCTURE ONLY) for precision='bf16x3' of the fused joint + RNN-T loss.

`split_bf16_product` restates the operand split of the tcgen05 kernels (ctc-vr_b200/csrc/joint_tc*.cu[h], the split
instantiations): each fp32 operand x is hi + lo with hi = bf16_rn(x), lo = bf16_rn(x - hi), and the tensor cores
accumulate a_hi b_hi + a_hi b_lo + a_lo b_hi (lo lo dropped).  Accumulation is fp64 here: the restatement bounds the
OPERAND error, which is what the split changes (cf. `lstm_oracle.split_tf32_product`).

`fused_joint_rnnt_bf16x3_restated` is `transducer_oracle.fused_joint_rnnt_restated` with the three GEMMs of the joint
(logits = z W^T, dZ = G W, dW = G^T z) computed that way; z = tanh(e + p), the softmax, the lattice, G and the
reductions are exact (fp64), as they are fp32 in the kernels.
"""
from __future__ import annotations

import torch

from .transducer_oracle import rnnt_lattice_restated


def _split(x):
    x = x.to(torch.float32)
    hi = x.to(torch.bfloat16).to(torch.float32)
    lo = (x - hi).to(torch.bfloat16).to(torch.float32)
    return hi.double(), lo.double()


def split_bf16_product(a, b):
    """a [M,K] @ b [K,N] as hi*hi + hi*lo + lo*hi of the bf16 splits of the fp32 operands, accumulated in fp64."""
    a_hi, a_lo = _split(a)
    b_hi, b_lo = _split(b)
    return a_hi @ b_hi + a_hi @ b_lo + a_lo @ b_hi


def fused_joint_rnnt_bf16x3_restated(enc_out, pred_out, w, targets, logit_lengths, target_lengths, blank: int,
                                     clamp: float = -1.0):
    """Loss (reduction='mean') and gradients wrt enc_out / pred_out / ffn_out.* of the fused seam with pre_project=False
    (enc_out / pred_out are the enc_ffn / pred_ffn outputs the fused op takes).  Keys as in fused_joint_rnnt_restated."""
    e = enc_out.detach().to(torch.float32)
    p = pred_out.detach().to(torch.float32)
    W = w["ffn_out.weight"].detach().to(torch.float32)
    bias = w["ffn_out.bias"].detach().to(torch.float64)
    B, T, D = e.shape
    U1, V = p.shape[1], W.shape[0]
    z = torch.tanh(e.double()[:, :, None] + p.double()[:, None]).to(torch.float32)        # fp32 z, as the kernels form it
    z2 = z.reshape(-1, D)
    logits = (split_bf16_product(z2, W.t()) + bias).reshape(B, T, U1, V)
    r = rnnt_lattice_restated(logits, targets, logit_lengths, target_lengths, blank, clamp, torch.float64)
    g = (r["grads"] / B).reshape(-1, V).to(torch.float32)                                   # G in fp32, then split
    dz = split_bf16_product(g, W).reshape(B, T, U1, D)
    dh = dz * (1.0 - z.double() ** 2)
    return dict(loss=r["costs"].mean(), costs=r["costs"], d_enc_out=dh.sum(2), d_pred_out=dh.sum(1),
                **{"d_ffn_out.weight": split_bf16_product(g.t().contiguous(), z2), "d_ffn_out.bias": g.double().sum(0)})
