"""TransducerJoint — same constructor, parameter names and forward signature as
model/component/joint.py:9-69 (and wenet/transducer/joint.py:62-92), so checkpoints load unchanged
(state_dict keys enc_ffn.*, pred_ffn.*, ffn_out.*[, post_ffn.*])."""
from typing import Optional

import torch
from torch import nn
from torch.nn import functional as F

from . import functional as CF


_ONES = {}


def _ones_row(n: int, device) -> torch.Tensor:
    """[1, n] bf16 ones, cached per (n, device): the bias gradient of a pre-projection is ones @ dy."""
    key = (n, str(device))
    t = _ONES.get(key)
    if t is None:
        t = _ONES[key] = torch.ones(1, n, dtype=torch.bfloat16, device=device)
    return t


class _Bf16Linear(torch.autograd.Function):
    """`F.linear` for the two pre-projections of the bf16 path: bf16 operands, fp32 accumulation (what
    `torch.autocast` gives), but the backward writes fp32 gradients straight from the library GEMMs
    (`torch.mm(..., out_dtype=float32)`) and takes the bias gradient as a ones-row GEMM - three GEMMs instead of
    autocast's two GEMMs + a column-sum reduction + three cast kernels per layer and step."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        xb = x.reshape(-1, x.shape[-1]).to(torch.bfloat16)
        wb = weight.to(torch.bfloat16)
        y = torch.addmm(bias.to(torch.bfloat16), xb, wb.t()) if bias is not None else torch.mm(xb, wb.t())
        ctx.save_for_backward(xb, wb)
        ctx.x_shape, ctx.x_dtype, ctx.w_dtype = x.shape, x.dtype, weight.dtype
        return y.reshape(*x.shape[:-1], weight.shape[0])

    @staticmethod
    def backward(ctx, dy):
        xb, wb = ctx.saved_tensors
        dy2 = dy.reshape(-1, dy.shape[-1]).to(torch.bfloat16)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            if ctx.x_dtype == torch.bfloat16:       # bf16 inputs take bf16 gradients straight from the GEMM
                dx = torch.mm(dy2, wb).reshape(ctx.x_shape)
            else:
                dx = torch.mm(dy2, wb, out_dtype=torch.float32).reshape(ctx.x_shape).to(ctx.x_dtype)
        if ctx.needs_input_grad[1]:
            dw = torch.mm(dy2.t(), xb, out_dtype=torch.float32).to(ctx.w_dtype)
        if ctx.needs_input_grad[2]:
            db = torch.mm(_ones_row(dy2.shape[0], dy2.device), dy2, out_dtype=torch.float32).reshape(-1).to(ctx.w_dtype)
        return dx, dw, db


def joint_activation(joint) -> str:
    """'tanh', 'relu' or 'gelu': the activation module of a TransducerJoint or of the reference's joint
    (model/component/joint.py:20-27).  Anything else (e.g. the tanh approximation of GELU) raises: the fused kernels
    would otherwise compute a different function."""
    act = getattr(joint, "activation", None)
    if isinstance(act, nn.Tanh):
        return "tanh"
    if isinstance(act, nn.ReLU):
        return "relu"
    if isinstance(act, nn.GELU) and getattr(act, "approximate", "none") == "none":
        return "gelu"
    raise RuntimeError(f"ctcvr_b200: the fused joint kernels compute tanh, relu or exact gelu, not {act!r}")


def fused_joint_inputs(joint, enc_out, pred_out, linear=F.linear, pre_project: bool = True):
    """(enc_proj, pred_proj) for the fused loss of a joint_mode='add' joint: the pre-join linears (when the joint has
    them), then the post-join linear folded into both sides - it is linear, so
    post(e + p) = (W_post e + b_post) + W_post p.  `linear(x, weight, bias)` runs each product (bias may be None)."""
    if getattr(joint, "joint_mode", "add") != "add":
        raise RuntimeError("ctcvr_b200: the fused RNN-T loss needs joint_mode='add'")
    e, p = enc_out, pred_out
    if pre_project and getattr(joint, "prejoin_linear", True) and joint.enc_ffn is not None and joint.pred_ffn is not None:
        e = linear(e, joint.enc_ffn.weight, joint.enc_ffn.bias)
        p = linear(p, joint.pred_ffn.weight, joint.pred_ffn.bias)
    post = getattr(joint, "post_ffn", None)
    if getattr(joint, "postjoin_linear", False) and post is not None:
        e = linear(e, post.weight, post.bias)
        p = linear(p, post.weight, None)
    return e, p


class TransducerJoint(nn.Module):
    def __init__(self, vocab_size: int, enc_output_size: int, pred_output_size: int, join_dim: int,
                 prejoin_linear: bool = True, postjoin_linear: bool = False, joint_mode: str = "add",
                 activation: str = "tanh"):
        super().__init__()
        self.activation_name = activation if activation in ("tanh", "relu", "gelu") else "tanh"
        self.activation = {"tanh": nn.Tanh(), "relu": nn.ReLU(), "gelu": nn.GELU()}[self.activation_name]
        self.prejoin_linear = prejoin_linear
        self.postjoin_linear = postjoin_linear
        self.joint_mode = joint_mode
        if not self.prejoin_linear and not self.postjoin_linear:
            assert enc_output_size == pred_output_size == join_dim
        self.enc_ffn: Optional[nn.Linear] = None
        self.pred_ffn: Optional[nn.Linear] = None
        if self.prejoin_linear:
            self.enc_ffn = nn.Linear(enc_output_size, join_dim)
            self.pred_ffn = nn.Linear(pred_output_size, join_dim)
        self.post_ffn: Optional[nn.Linear] = None
        if self.postjoin_linear:
            self.post_ffn = nn.Linear(join_dim, join_dim)
        self.ffn_out = nn.Linear(join_dim, vocab_size)

    @property
    def fusable(self) -> bool:
        """True for the configuration both reference models build (add + tanh, no post-join linear)."""
        return self.activation_name == "tanh" and not self.postjoin_linear and self.joint_mode == "add"

    def project(self, enc_out, pred_out, pre_project: bool = True):
        """enc_ffn / pred_ffn (joint.py:52-55): two small library GEMMs."""
        if pre_project and self.prejoin_linear and self.enc_ffn is not None and self.pred_ffn is not None:
            enc_out = self.enc_ffn(enc_out)
            pred_out = self.pred_ffn(pred_out)
        return enc_out, pred_out

    def forward(self, enc_out: torch.Tensor, pred_out: torch.Tensor, pre_project: bool = True) -> torch.Tensor:
        """Dense logits [B,T,U,V] (joint.py:48-69).  The training path does not call this: it uses
        `rnnt_loss_fused`, which never materialises the logits."""
        enc_out, pred_out = self.project(enc_out, pred_out, pre_project)
        if self.fusable and enc_out.is_cuda and enc_out.dim() == 3 and pred_out.dim() == 3:
            return CF.joint_logits(enc_out, pred_out, self.ffn_out.weight, self.ffn_out.bias)
        if not enc_out.is_cuda:
            raise RuntimeError("ctcvr_b200.TransducerJoint runs on CUDA (B200) tensors only; there is no CPU path")
        # non-default configurations (relu/gelu, post-join linear) keep the reference data flow
        if enc_out.ndim != 4:
            enc_out = enc_out.unsqueeze(2)
        if pred_out.ndim != 4:
            pred_out = pred_out.unsqueeze(1)
        out = enc_out + pred_out
        if self.postjoin_linear and self.post_ffn is not None:
            out = self.post_ffn(out)
        return self.ffn_out(self.activation(out))

    def rnnt_loss_fused(self, enc_out, pred_out, targets, logit_lengths, target_lengths, blank: int,
                        clamp: float = -1.0, reduction: str = "mean", precision: str = "fp32",
                        pre_project: bool = True):
        """joint + log-softmax + RNN-T lattice loss in one op (the seam of transducer.py:172-187).
        precision='fp32' keeps the reference's arithmetic; 'bf16' opts into the tcgen05 tensor-core path; 'bf16x3'
        runs the tensor-core path at fp32 accuracy (the pre-projections then stay fp32, as with 'fp32').
        Every activation ('tanh', 'relu', 'gelu') with or without pre-join and post-join linears is fused; the post-join
        linear folds into the two inputs (`fused_joint_inputs`).  joint_mode must be 'add'."""
        if self.joint_mode != "add":
            raise RuntimeError("rnnt_loss_fused: only joint_mode='add'")
        if not self.fusable:
            lin = _Bf16Linear.apply if precision in ("bf16", CF.BF16) and enc_out.is_cuda else F.linear
            e, p = fused_joint_inputs(self, enc_out, pred_out, lin, pre_project)
            return CF.fused_joint_rnnt_loss(e, p, self.ffn_out.weight, self.ffn_out.bias, targets, logit_lengths,
                                            target_lengths, blank, clamp, reduction, precision,
                                            activation=self.activation_name)
        if precision in ("bf16", CF.BF16) and enc_out.is_cuda:
            # bf16 path: the two pre-projections are plain library GEMMs; run them on the tensor cores too
            if pre_project and self.prejoin_linear and self.enc_ffn is not None and self.pred_ffn is not None:
                e = _Bf16Linear.apply(enc_out, self.enc_ffn.weight, self.enc_ffn.bias)
                p = _Bf16Linear.apply(pred_out, self.pred_ffn.weight, self.pred_ffn.bias)
            else:
                e, p = enc_out, pred_out
        else:
            e, p = self.project(enc_out, pred_out, pre_project)
        return CF.fused_joint_rnnt_loss(e, p, self.ffn_out.weight, self.ffn_out.bias, targets, logit_lengths,
                                        target_lengths, blank, clamp, reduction, precision)

    @torch.no_grad()
    def forced_align(self, enc_out, pred_out, targets, logit_lengths, target_lengths, blank: int,
                     precision: str = "fp32", pre_project: bool = True):
        """Forced alignment of `targets` [B,U] through this joint (functional.rnnt_forced_align): the inputs go through
        the same pre-join / post-join handling as `rnnt_loss_fused` (every activation, joint_mode='add').  Returns
        (frames [B,U] int32, token_logprobs [B,U], scores [B])."""
        lin = _Bf16Linear.apply if precision in ("bf16", CF.BF16) and enc_out.is_cuda else F.linear
        e, p = fused_joint_inputs(self, enc_out, pred_out, lin, pre_project)
        return CF.rnnt_forced_align(e, p, self.ffn_out.weight, self.ffn_out.bias, targets, logit_lengths, target_lengths,
                                    blank, precision, activation=self.activation_name)
