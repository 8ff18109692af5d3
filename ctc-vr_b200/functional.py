"""Autograd ops over the C-ABI kernels.

  fused_joint_rnnt_loss  — the fused seam of SURVEY.md §8b: everything between the predictor output and
                           the per-utterance cost (model/component/transducer.py:172-187,
                           model/online_rnnt_model.py:243-255) as one op; logits never reach HBM.
  rnnt_loss              — drop-in for torchaudio.functional.rnnt_loss on dense logits
                           (site-packages/torchaudio/functional/functional.py:1747-1800).
  ctc_loss               — drop-in for F.log_softmax + nn.CTCLoss(zero_infinity=True) tails
                           (model/rnnt_model.py:55-58, model/online_rnnt_model.py:29-30).
  joint_logits           — dense TransducerJoint tail (model/component/joint.py:57-68).
  lstm_sequence          — one layer of the predictor's nn.LSTM over a whole label sequence, forward and backward
                           (model/component/predictor.py:58, SURVEY.md §8f row 2).
  rnnt_viterbi / rnnt_forced_align / ctc_forced_align
                         — batched forced alignment: the best path of a known transcript through the RNN-T lattice
                           (on the fused joint's log-probs) or the CTC trellis, with per-token frames / spans.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import call, ptr, query, stream

F32, BF16, BF16X3 = 0, 1, 2
_PREC = {"fp32": F32, "f32": F32, "bf16": BF16, "bf16x3": BF16X3, F32: F32, BF16: BF16, BF16X3: BF16X3}
_PREC_NAME = {F32: "fp32", BF16: "bf16", BF16X3: "bf16x3"}
# joint activation bits OR'ed into the precision argument (CTCVR_ACT_* of include/ctcvr.h)
ACT_TANH, ACT_RELU, ACT_GELU = 0x000, 0x100, 0x200
_ACT = {"tanh": ACT_TANH, "relu": ACT_RELU, "gelu": ACT_GELU}


def _f32c(t):
    return t.detach().to(torch.float32).contiguous()


def _i32c(t, device):
    return t.detach().to(device=device, dtype=torch.int32).contiguous()


def _ws(nbytes, device):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def _vocab_tiled(precision, V, vocab_tiling):
    """Whether a call takes the vocabulary-tile entry points (`ctcvr_joint_rnnt_*_vt`): only a tensor-core precision
    with vocab_tiling=True and pad32(V) > 416.  Every other call keeps its entry points and kernels."""
    return bool(vocab_tiling) and precision in (BF16, BF16X3) and (V + 31) // 32 * 32 > 416


def _joint_fwd(enc_proj, pred_proj, w_out, b_out, targets, t_len, u_len, blank, precision, act,
               op="fused_joint_rnnt_loss", vocab_tiling=False):
    """The fused joint forward (`ctcvr_joint_rnnt_fwd` / `_bf16in` / `_vt`) with the fused loss's input handling and
    errors.  Returns the kernel inputs (e, p, w, b, tg, tl, ul), whether the bf16-input entry point ran, and lse /
    lp_blank / lp_label [B,T,U1]."""
    _lib.require_cuda(enc_proj, pred_proj, w_out, b_out)
    dev = enc_proj.device
    w, b = _f32c(w_out), _f32c(b_out)
    B, T, D = enc_proj.shape
    U1 = pred_proj.shape[1]
    V = w.shape[0]
    # bf16 activations (autocast) are consumed in place by the tensor-core path: no fp32 round trip.  The bf16-input
    # entry points are tanh only; other joints pass bf16 inputs through the fp32-input entry point, whose bf16 path
    # rounds them to bf16 again (exact), so the arithmetic is the same.
    tiled = _vocab_tiled(precision, V, vocab_tiling)
    bf16_in = precision == BF16 and act == ACT_TANH and enc_proj.dtype == torch.bfloat16 and \
        pred_proj.dtype == torch.bfloat16 and not tiled
    if bf16_in:
        e, p = enc_proj.detach().contiguous(), pred_proj.detach().contiguous()
    else:
        e, p = _f32c(enc_proj), _f32c(pred_proj)
    if p.shape[0] != B or p.shape[2] != D or w.shape[1] != D or b.shape[0] != V:
        raise RuntimeError(f"{op}: inconsistent shapes")
    tg = _i32c(targets, dev)
    if tg.dim() != 2 or tg.shape[0] != B or tg.shape[1] != U1 - 1:
        raise RuntimeError(f"{op}: targets must be [B, U] with U == pred_out.size(1) - 1")
    tl, ul = _i32c(t_len, dev), _i32c(u_len, dev)
    if tl.dim() != 1 or ul.dim() != 1 or tl.shape[0] != B or ul.shape[0] != B:
        raise RuntimeError(f"{op}: logit_lengths / target_lengths must be [B]")
    if not (0 <= blank < V):
        raise RuntimeError(f"{op}: blank must be within [0, vocab)")
    # Length / label VALUES are not read back (that would be a host sync in the training step): the kernels clamp
    # lengths to the tensor extents and treat a label outside [0, V) as blank, so bad values cannot fault the GPU.
    if tiled and not bool(query("ctcvr_joint_tc_vt_supported", U1, D, V)):
        raise RuntimeError(f"{op}: precision='{_PREC_NAME[precision]}' with vocab_tiling=True needs D % 128 == 0, "
                           f"D <= 512, V <= 32768 and U+1 <= 128 (got D={D}, V={V}, U+1={U1}); use precision='fp32' "
                           "for this shape")
    if precision in (BF16, BF16X3) and not tiled and not bool(query("ctcvr_joint_tc_supported", U1, D, V)):
        more = ", or vocab_tiling=True for V > 416" if D % 128 == 0 and D <= 512 and U1 <= 128 else ""
        raise RuntimeError(f"{op}: precision='{_PREC_NAME[precision]}' needs D % 128 == 0, D <= 512, "
                           f"V <= 416 and U+1 <= 128 (got D={D}, V={V}, U+1={U1}); use precision='fp32' for this "
                           f"shape{more}")
    lse = torch.empty((B, T, U1), dtype=torch.float32, device=dev)
    lpb, lpl = torch.empty_like(lse), torch.empty_like(lse)
    with torch.cuda.device(dev):
        vt = "_vt" if tiled else ""
        ws = _ws(query(f"ctcvr_joint_rnnt_fwd{vt}_ws_bytes", B, T, U1, D, V, precision | act), dev)
        if bf16_in:
            call("ctcvr_joint_rnnt_fwd_bf16in", ptr(e), ptr(p), ptr(w), ptr(b), ptr(tg), ptr(tl), ptr(ul), ptr(lse),
                 ptr(lpb), ptr(lpl), B, T, U1, D, V, blank, ptr(ws), ws.numel(), stream())
        else:
            call(f"ctcvr_joint_rnnt_fwd{vt}", ptr(e), ptr(p), ptr(w), ptr(b), ptr(tg), ptr(tl), ptr(ul), ptr(lse),
                 ptr(lpb), ptr(lpl), B, T, U1, D, V, blank, precision | act, ptr(ws), ws.numel(), stream())
    return (e, p, w, b, tg, tl, ul), bf16_in, lse, lpb, lpl


class _FusedJointRnnt(torch.autograd.Function):
    @staticmethod
    def forward(ctx, enc_proj, pred_proj, w_out, b_out, targets, t_len, u_len, blank, clamp, precision, act,
                vocab_tiling=False):
        (e, p, w, b, tg, tl, ul), bf16_in, lse, lpb, lpl = _joint_fwd(enc_proj, pred_proj, w_out, b_out, targets, t_len,
                                                                      u_len, blank, precision, act,
                                                                      vocab_tiling=vocab_tiling)
        B, T, U1 = lse.shape
        alpha, beta = torch.empty_like(lse), torch.empty_like(lse)
        costs = torch.empty((B,), dtype=torch.float32, device=lse.device)
        with torch.cuda.device(lse.device):
            call("ctcvr_rnnt_lattice", ptr(lpb), ptr(lpl), ptr(tl), ptr(ul), ptr(alpha), ptr(beta), ptr(costs),
                 B, T, U1, stream())
        ctx.save_for_backward(e, p, w, b, tg, tl, ul, lse, lpb, lpl, alpha, beta, costs)
        ctx.cfg = (blank, float(clamp), precision, bf16_in, act, enc_proj.dtype, pred_proj.dtype,
                   _vocab_tiled(precision, w.shape[0], vocab_tiling))
        return costs

    @staticmethod
    def backward(ctx, grad_costs):
        e, p, w, b, tg, tl, ul, lse, lpb, lpl, alpha, beta, costs = ctx.saved_tensors
        blank, clamp, precision, bf16_in, act, e_dtype, p_dtype, tiled = ctx.cfg
        B, T, D = e.shape
        U1, V = p.shape[1], w.shape[0]
        dev = e.device
        gc = _f32c(grad_costs)
        # bf16-input entry point: gradients come back in bf16 (the dtype autograd expects for bf16 inputs)
        gdt = torch.bfloat16 if bf16_in else torch.float32
        d_e = torch.empty(e.shape, dtype=gdt, device=dev)
        d_p = torch.empty(p.shape, dtype=gdt, device=dev)
        d_w, d_b = torch.empty_like(w), torch.empty_like(b)
        with torch.cuda.device(dev):
            vt = "_vt" if tiled else ""
            ws = _ws(query(f"ctcvr_joint_rnnt_bwd{vt}_ws_bytes", B, T, U1, D, V, precision | act), dev)
            if bf16_in:
                call("ctcvr_joint_rnnt_bwd_bf16in", ptr(e), ptr(p), ptr(w), ptr(b), ptr(tg), ptr(tl), ptr(ul), ptr(lse),
                     ptr(lpb), ptr(lpl), ptr(alpha), ptr(beta), ptr(costs), ptr(gc), clamp, ptr(d_e), ptr(d_p), ptr(d_w), ptr(d_b),
                     B, T, U1, D, V, blank, ptr(ws), ws.numel(), stream())
            else:
                call(f"ctcvr_joint_rnnt_bwd{vt}", ptr(e), ptr(p), ptr(w), ptr(b), ptr(tg), ptr(tl), ptr(ul), ptr(lse),
                     ptr(lpb), ptr(lpl), ptr(alpha), ptr(beta), ptr(costs), ptr(gc), clamp, ptr(d_e), ptr(d_p), ptr(d_w), ptr(d_b),
                     B, T, U1, D, V, blank, precision | act, ptr(ws), ws.numel(), stream())
        if not bf16_in:                                   # gradients in the dtype of the inputs
            d_e, d_p = d_e.to(e_dtype), d_p.to(p_dtype)
        return d_e, d_p, d_w, d_b, None, None, None, None, None, None, None, None


def fused_joint_rnnt_loss(enc_proj, pred_proj, w_out, b_out, targets, logit_lengths, target_lengths,
                          blank: int, clamp: float = -1.0, reduction: str = "mean", precision="fp32",
                          activation: str = "tanh", vocab_tiling: bool = False):
    """costs_b = RNN-T negative log-likelihood of utterance b for
    logits = ffn_out(act(enc_proj[:, :, None] + pred_proj[:, None])) without materialising them.
    enc_proj [B,T,D] / pred_proj [B,U+1,D] are the enc_ffn / pred_ffn outputs (joint.py:54-55).
    activation: 'tanh' (default), 'relu' (nn.ReLU, derivative 0 at 0) or 'gelu' (nn.GELU(), exact erf form).  A post-join
    linear folds into the two inputs: post(e + p) = (W_post e + b_post) + W_post p.  Every precision below holds for every
    activation; in 'bf16' the sum e + p is rounded to bf16 before the activation (gelu is then evaluated in fp32).  One
    exception, from relu's kink: in 'bf16' on fp32 inputs, every element whose e + p lies within the bf16 rounding error
    of 0 can land on the other side of the kink, and its derivative flips between 0 and 1.  That adds about
    sqrt(flipped fraction) to the relative error of the gradients (measured 4.6e-2 on d_enc with 0.5-scale Gaussian
    inputs at D = 384, where 4.6e-4 of the elements flip), on top of the 3e-2 below; a relu joint on bf16 inputs is within
    the 3e-2 of those inputs.

    precision='fp32' (default) is the reference's arithmetic (loss and gradients within 1e-4 of torchaudio's);
    precision='bf16' is the explicit opt-in to the tcgen05 path (bf16 operands, fp32 accumulation, softmax and
    lattice; each cost within 2e-3, or within 1e-3 nats per lattice step (T_b + U_b) where that is larger, since bf16
    rounding moves every log-probability by up to ~1e-3 and small costs (under ~0.5 nats a step) cannot meet 2e-3 of
    themselves; gradients within 3e-2 rel-L2) and raises on shapes outside its tiling.
    precision='bf16x3' runs the same tcgen05 tiling at fp32 accuracy: every fp32 GEMM operand is split into
    hi = bf16(x) and lo = bf16(x - hi) and each product is hi*hi + hi*lo + lo*hi, with tanh, d cost / d logits and the
    reductions in fp32.  Loss and gradients are within 1e-4 of the reference, like fp32; inputs are taken as fp32, and
    the shape limits and the error on other shapes are those of 'bf16'.

    vocab_tiling=True lets 'bf16' and 'bf16x3' take vocabularies up to 32768 (D % 128 == 0, D <= 512 and U+1 <= 128
    still hold): where pad32(V) > 416 the softmax runs over vocabulary tiles of at most 416 columns, each through the
    tensor-core kernels, with a running log-sum-exp; the logits still never reach HBM.  The bars are those above:
    'bf16' 2e-3 per cost (or 1e-3 nats per lattice step) and 3e-2 rel-L2 on the gradients, 'bf16x3' 1e-4.  Where
    pad32(V) <= 416 it changes nothing (the same kernels run), and with 'fp32', which takes every V, it has no effect,
    so a model can set it once whatever its precision.  Without it, V > 416 raises on the tensor-core precisions."""
    if activation not in _ACT:
        raise ValueError(f"fused_joint_rnnt_loss: activation must be one of {sorted(_ACT)}, got {activation!r}")
    costs = _FusedJointRnnt.apply(enc_proj, pred_proj, w_out, b_out, targets, logit_lengths, target_lengths,
                                  int(blank), float(clamp), _PREC[precision], _ACT[activation], bool(vocab_tiling))
    return _reduce(costs, reduction)


def _reduce(costs, reduction):
    if reduction == "mean":
        return costs.mean()
    if reduction == "sum":
        return costs.sum()
    if reduction == "none":
        return costs
    raise ValueError('reduction should be one of "none", "mean", or "sum"')


class _RnntLossDense(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, targets, t_len, u_len, blank, clamp):
        B, T, U1, V = logits.shape
        dev = logits.device
        costs = torch.empty((B,), dtype=torch.float32, device=dev)
        grads = torch.empty_like(logits) if logits.requires_grad else None
        with torch.cuda.device(dev):
            ws = _ws(query("ctcvr_rnnt_loss_dense_ws_bytes", B, T, U1), dev)
            call("ctcvr_rnnt_loss_dense", ptr(logits), ptr(targets), ptr(t_len), ptr(u_len), ptr(costs), ptr(grads),
                 B, T, U1, V, blank, clamp, ptr(ws), ws.numel(), stream())
        ctx.grads = grads
        return costs

    @staticmethod
    def backward(ctx, dy):
        g = ctx.grads
        return (g * dy.view(-1, 1, 1, 1) if g is not None else None), None, None, None, None, None


def rnnt_loss(logits, targets, logit_lengths, target_lengths, blank: int = -1, clamp: float = -1,
              reduction: str = "mean", fused_log_softmax: bool = True):
    """Same signature and checks as torchaudio.functional.rnnt_loss (functional.py:1747-1800); the
    validation errors of rnnt/cpu/compute.cpp:36-84 are raised as RuntimeError.  Those checks compare only the
    longest lengths with the shape.  Values the reference leaves undefined are defined here and cannot index outside
    the tensors: lengths are clamped to [0, T] and [0, U], so a negative length behaves exactly like 0 (no frames:
    cost 0 and zero gradient; no labels: the blank-only path), and a label outside [0, V) behaves exactly like
    `blank`, in the cost and the gradient."""
    if reduction not in ("none", "mean", "sum"):
        raise ValueError('reduction should be one of "none", "mean", or "sum"')
    _lib.require_cuda(logits)
    if not fused_log_softmax:
        raise RuntimeError("rnnt_loss: only fused_log_softmax=True is supported (the only mode the reference uses)")
    if logits.dtype != torch.float32:
        raise RuntimeError("rnnt_loss: logits must be float32")
    if targets.dtype != torch.int32 or logit_lengths.dtype != torch.int32 or target_lengths.dtype != torch.int32:
        raise RuntimeError("rnnt_loss: targets, logit_lengths and target_lengths must be int32")
    if logits.dim() != 4 or targets.dim() != 2 or logit_lengths.dim() != 1 or target_lengths.dim() != 1:
        raise RuntimeError("rnnt_loss: logits must be 4-D, targets 2-D, lengths 1-D")
    if not (logits.is_contiguous() and targets.is_contiguous()):
        raise RuntimeError("rnnt_loss: logits and targets must be contiguous")
    B, T, U1, V = logits.shape
    if blank < 0:
        blank = V + blank
    if not (0 <= blank < V):
        raise RuntimeError("rnnt_loss: blank must be within [0, logits.shape[-1])")
    if targets.shape[0] != B or logit_lengths.shape[0] != B or target_lengths.shape[0] != B:
        raise RuntimeError("rnnt_loss: batch dimension mismatch")
    # torchaudio also rejects non-max shapes (one host sync, as in the reference op)
    if int(logit_lengths.max()) != T:
        raise RuntimeError("rnnt_loss: input length mismatch")
    if int(target_lengths.max()) != U1 - 1 or targets.shape[1] != U1 - 1:
        raise RuntimeError("rnnt_loss: output length mismatch")
    dev = logits.device
    costs = _RnntLossDense.apply(logits, targets.to(dev), logit_lengths.to(dev).contiguous(),
                                 target_lengths.to(dev).contiguous(), int(blank), float(clamp))
    return _reduce(costs, reduction)


class _JointLogits(torch.autograd.Function):
    """Dense joint tail; backward through plain matmuls (not the hot path: the fused op is)."""
    @staticmethod
    def forward(ctx, enc_proj, pred_proj, w_out, b_out):
        e, p, w, b = _f32c(enc_proj), _f32c(pred_proj), _f32c(w_out), _f32c(b_out)
        B, T, D = e.shape
        U1, V = p.shape[1], w.shape[0]
        out = torch.empty((B, T, U1, V), dtype=torch.float32, device=e.device)
        with torch.cuda.device(e.device):
            call("ctcvr_joint_logits", ptr(e), ptr(p), ptr(w), ptr(b), ptr(out), B, T, U1, D, V, stream())
        ctx.save_for_backward(e, p, w)
        return out

    @staticmethod
    def backward(ctx, g):
        e, p, w = ctx.saved_tensors
        z = torch.tanh(e.unsqueeze(2) + p.unsqueeze(1))
        g2 = g.reshape(-1, g.shape[-1])
        dz = (g2 @ w).view_as(z) * (1 - z * z)
        return dz.sum(2), dz.sum(1), g2.t() @ z.reshape(-1, z.shape[-1]), g2.sum(0)


def joint_logits(enc_proj, pred_proj, w_out, b_out):
    """logits[b,t,u,:] = W_out tanh(enc_proj[b,t] + pred_proj[b,u]) + b_out (joint.py:57-68)."""
    _lib.require_cuda(enc_proj, pred_proj, w_out, b_out)
    return _JointLogits.apply(enc_proj, pred_proj, w_out, b_out)


def log_softmax_rows(x):
    """F.log_softmax(x, dim=-1) for fp32 CUDA input (forward only; used inside ctc_loss)."""
    xc = _f32c(x)
    y = torch.empty_like(xc)
    with torch.cuda.device(xc.device):
        call("ctcvr_log_softmax", ptr(xc), ptr(y), xc.numel() // xc.shape[-1], xc.shape[-1], stream())
    return y


class _CtcFromLogits(torch.autograd.Function):
    """logits [B,T,V] -> (nll [B], log_probs [B,T,V]).  As torchaudio does for rnnt_loss, the gradient
    wrt logits is produced by the same launch as the loss and scaled by dL/dnll in backward."""
    @staticmethod
    def forward(ctx, logits, targets, in_lens, tgt_lens, blank, zero_infinity):
        x = _f32c(logits)
        B, T, V = x.shape
        dev = x.device
        lp = torch.empty_like(x)
        nll = torch.empty((B,), dtype=torch.float32, device=dev)
        if targets.dim() != 2 or targets.shape[0] != B:
            raise ValueError(f"ctc_loss_from_logits: targets must be [B, Umax] = [{B}, Umax] (padded), got "
                             f"{list(targets.shape)}; concatenated 1-D targets are not supported")
        tg = targets.detach().to(device=dev, dtype=torch.int64).contiguous()
        Umax = tg.shape[1]
        il, tl = _i32c(in_lens, dev), _i32c(tgt_lens, dev)
        grad = torch.empty_like(x) if logits.requires_grad else None
        with torch.cuda.device(dev):
            call("ctcvr_log_softmax", ptr(x), ptr(lp), B * T, V, stream())
            ws = _ws(query("ctcvr_ctc_loss_ws_bytes", B, T, Umax), dev)
            call("ctcvr_ctc_loss", ptr(lp), ptr(tg), ptr(il), ptr(tl), None, ptr(nll), ptr(grad), B, T, V, Umax,
                 blank, int(zero_infinity), ptr(ws), ws.numel(), stream())
        ctx.grad = grad
        ctx.mark_non_differentiable(lp)
        return nll, lp

    @staticmethod
    def backward(ctx, g_nll, _g_lp):
        g = ctx.grad
        return (g * g_nll.view(-1, 1, 1) if g is not None else None), None, None, None, None, None


def ctc_loss_from_logits(logits, targets, input_lengths, target_lengths, blank: int, reduction: str = "sum",
                         zero_infinity: bool = True):
    """F.log_softmax(logits, -1) followed by nn.CTCLoss(blank, reduction, zero_infinity) on [B,T,V] logits.
    Returns (loss, log_probs [B,T,V]).  reduction semantics are ATen's: 'mean' divides each nll by
    clamp_min(target_length, 1) and averages over the batch.
    targets are padded [B, Umax] (ValueError otherwise); Umax <= 511.  Values the reference leaves undefined are
    defined here and cannot index outside the tensors: lengths are clamped to [0, T] and [0, Umax], so a negative
    input length behaves exactly like 0 (cost inf, 0 under zero_infinity, when the target is not empty; zero
    gradient), and a label outside [0, V) behaves exactly like `blank`."""
    _lib.require_cuda(logits)
    nll, lp = _CtcFromLogits.apply(logits, targets, input_lengths, target_lengths, int(blank), bool(zero_infinity))
    if reduction == "sum":
        loss = nll.sum()
    elif reduction == "mean":
        tl = target_lengths.to(device=nll.device, dtype=torch.float32).clamp_min(1)
        loss = (nll / tl).mean()
    elif reduction == "none":
        loss = nll
    else:
        raise ValueError(f"{reduction} is not a valid value for reduction")
    return loss, lp


class _tf32_matmul:
    """cuBLAS fp32 matmuls inside the block run on the TF32 tensor cores (torch's `fp32_precision` switch of the cuBLAS
    backend, restored on exit).  Only used on operands pre-split by `_split3`, where the result keeps fp32-level
    accuracy.  `ok` is False when the switch cannot be set (a script that drives the legacy allow_tf32 flag): the
    caller then multiplies the unsplit fp32 operands."""
    def __enter__(self):
        self.ok, self.old = True, None
        try:
            m = torch.backends.cuda.matmul
            self.old = m.fp32_precision
            m.fp32_precision = "tf32"
        except Exception:  # noqa: BLE001
            self.ok = False
        return self

    def __exit__(self, *exc):
        if self.ok:
            torch.backends.cuda.matmul.fp32_precision = self.old
        return False


def _split3(t2, stack_cols: bool, pattern: int):
    """[R,C] fp32 -> the (hi, hi|lo, lo|hi) TF32 terms stacked along the columns ([R,3C]) or the rows ([3R,C])."""
    R, Cc = t2.shape
    out = torch.empty((R, 3 * Cc) if stack_cols else (3 * R, Cc), dtype=torch.float32, device=t2.device)
    call("ctcvr_split_tf32", ptr(t2), ptr(out), R, Cc, int(stack_cols), int(pattern), stream())
    return out


def _mm3(a, b, out=None, a_t=False, b_t=False):
    """a @ b in fp32 accuracy on the tensor cores: a is [M,K] (or [K,M] with a_t), b is [K,N] (or [N,K] with b_t), both
    contiguous fp32.  Each operand is split along K into its TF32 terms (csrc/lstm_seq.cu::split_tf32_kernel) and the
    three products are one GEMM with K tripled."""
    with _tf32_matmul() as t:
        if not t.ok:
            aa, bb = (a.t() if a_t else a), (b.t() if b_t else b)
            return torch.mm(aa, bb, out=out) if out is not None else torch.mm(aa, bb)
        a3 = _split3(a, stack_cols=not a_t, pattern=0)           # K is the column index of a unless a is given transposed
        b3 = _split3(b, stack_cols=b_t, pattern=1)
        aa, bb = (a3.t() if a_t else a3), (b3.t() if b_t else b3)
        return torch.mm(aa, bb, out=out) if out is not None else torch.mm(aa, bb)


_SIDE = {}


def _side_streams(dev):
    """Two side streams per device for the independent GEMMs of the LSTM backward."""
    key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
    st = _SIDE.get(key)
    if st is None:
        st = _SIDE[key] = (torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev))
    return st


class _LstmSeq(torch.autograd.Function):
    """One LSTM layer over [B,U1,*] (batch_first, fp32).  The sequential part runs in the two persistent kernels of
    csrc/lstm_seq.cu; the input projection and the three weight / input gradient products are plain library GEMMs
    over all B*U1 rows at once."""
    @staticmethod
    def forward(ctx, x, w_ih, w_hh, b_ih, b_hh, h0, c0):
        _lib.require_cuda(x, w_ih, w_hh, h0, c0)
        dev = x.device
        B, U1, E = x.shape
        H = w_hh.shape[1]
        if w_ih.shape != (4 * H, E) or w_hh.shape != (4 * H, H) or h0.shape != (B, H) or c0.shape != (B, H):
            raise RuntimeError("lstm_sequence: inconsistent shapes")
        if U1 == 0:
            raise RuntimeError("lstm_sequence: empty sequence")
        if not bool(query("ctcvr_lstm_seq_supported", B, H)):
            raise RuntimeError(f"lstm_sequence: hidden size {H} with batch {B} does not fit the persistent kernel "
                               "(H <= 16 x SM count and the per-CTA shared memory)")
        x2 = _f32c(x).view(B * U1, E)
        wi, wh = _f32c(w_ih), _f32c(w_hh)
        bias = None
        if b_ih is not None:
            bias = _f32c(b_ih) + _f32c(b_hh)
        with torch.cuda.device(dev):
            xg = _mm3(x2, wi, b_t=True)                            # x W_ih^T
        if bias is not None:
            xg += bias
        h0c, c0c = _f32c(h0), _f32c(c0)
        keep = any(ctx.needs_input_grad)
        out = torch.empty((B, U1, H), dtype=torch.float32, device=dev)
        hn = torch.empty((B, H), dtype=torch.float32, device=dev)
        cn = torch.empty_like(hn)
        cs = torch.empty_like(out) if keep else None
        act = torch.empty((B, U1, 4 * H), dtype=torch.float32, device=dev) if keep else None
        with torch.cuda.device(dev):
            ws = _ws(query("ctcvr_lstm_seq_ws_bytes", B, H), dev)
            call("ctcvr_lstm_seq_fwd", ptr(xg), ptr(wh), ptr(h0c), ptr(c0c), ptr(out), ptr(cs), ptr(act), ptr(hn), ptr(cn),
                 B, U1, H, ptr(ws), ws.numel(), stream())
        if keep:
            ctx.save_for_backward(x2, wi, wh, h0c, c0c, out, cs, act)
        ctx.has_bias = b_ih is not None
        ctx.dims = (B, U1, E, H)
        return out, hn, cn

    @staticmethod
    def backward(ctx, d_out, d_hn, d_cn):
        x2, wi, wh, h0c, c0c, out, cs, act = ctx.saved_tensors
        B, U1, E, H = ctx.dims
        dev = x2.device
        d_out = _f32c(d_out) if d_out is not None else None
        d_hn = _f32c(d_hn) if d_hn is not None else None
        d_cn = _f32c(d_cn) if d_cn is not None else None
        dg = torch.empty((B, U1, 4 * H), dtype=torch.float32, device=dev)
        d_h0 = torch.empty((B, H), dtype=torch.float32, device=dev)
        d_c0 = torch.empty_like(d_h0)
        with torch.cuda.device(dev):
            ws = _ws(query("ctcvr_lstm_seq_ws_bytes", B, H), dev)
            call("ctcvr_lstm_seq_bwd", ptr(act), ptr(cs), ptr(c0c), ptr(wh), ptr(d_out), ptr(d_hn), ptr(d_cn), ptr(dg),
                 ptr(d_h0), ptr(d_c0), B, U1, H, ptr(ws), ws.numel(), stream())
        dg2 = dg.view(B * U1, 4 * H)
        ng = ctx.needs_input_grad
        # dx, dW_ih (+ the bias column sum) and dW_hh are independent plain GEMMs of 44 - 64 output tiles each at the
        # reference sizes - a third of the chip apiece - so they run side by side on three streams (parallel branches
        # when the step is captured in a CUDA graph).  Outputs are allocated on the calling stream.
        need_b = ctx.has_bias and (ng[3] or ng[4])
        d_wi = torch.empty((4 * H, E), dtype=torch.float32, device=dev) if ng[1] else None
        d_wh = torch.empty((4 * H, H), dtype=torch.float32, device=dev) if ng[2] else None
        db = torch.empty((4 * H,), dtype=torch.float32, device=dev) if need_b else None
        h_prev = torch.empty((B, U1, H), dtype=torch.float32, device=dev) if ng[2] else None
        cur = torch.cuda.current_stream(dev)
        s1, s2 = _side_streams(dev)
        if ng[1] or need_b:
            s1.wait_stream(cur)
            with torch.cuda.stream(s1):
                if ng[1]:
                    _mm3(dg2, x2, out=d_wi, a_t=True)              # dG^T x
                if need_b:
                    torch.sum(dg2, 0, out=db)
        if ng[2]:
            s2.wait_stream(cur)
            with torch.cuda.stream(s2):
                h_prev[:, 0].copy_(h0c)
                if U1 > 1:
                    h_prev[:, 1:].copy_(out[:, :-1])
                _mm3(dg2, h_prev.view(B * U1, H), out=d_wh, a_t=True)   # dG^T h_prev
        dx = _mm3(dg2, wi).view(B, U1, E) if ng[0] else None          # dG W_ih
        if ng[1] or need_b:
            cur.wait_stream(s1)
        if ng[2]:
            cur.wait_stream(s2)
        return dx, d_wi, d_wh, (db if ctx.has_bias and ng[3] else None), (db if ctx.has_bias and ng[4] else None), \
            (d_h0 if ng[5] else None), (d_c0 if ng[6] else None)


def lstm_sequence(x, w_ih, w_hh, b_ih, b_hh, h0, c0):
    """`out, (h_n, c_n) = nn.LSTM(batch_first=True)(x, (h0, c0))` for ONE layer: x [B,U1,E], w_ih [4H,E], w_hh [4H,H],
    biases [4H] (or both None), h0 / c0 [B,H].  Returns (out [B,U1,H], h_n [B,H], c_n [B,H]) in fp32, differentiable
    in every argument.  This is the reference predictor's recurrence (model/component/predictor.py:58)."""
    return _LstmSeq.apply(x, w_ih, w_hh, b_ih, b_hh, h0, c0)


def _len_check(op, B, *lens):
    for t in lens:
        if t.dim() != 1 or t.shape[0] != B:
            raise RuntimeError(f"{op}: lengths must be [B] = [{B}]")


@torch.no_grad()
def rnnt_viterbi(lp_blank, lp_label, logit_lengths, target_lengths):
    """Best path through the RNN-T lattice of lp_blank / lp_label [B,T,U+1] (fp32, the layout the fused forward writes):
    delta(0,0) = 0, delta(t,u) = max(delta(t-1,u) + lp_blank(t-1,u), delta(t,u-1) + lp_label(t,u-1)).
    Returns (frames [B,U] int32: the frame at which label u is emitted, non-decreasing, -1 beyond U_b;
    token_logprobs [B,U] fp32: lp_label at that cell, 0 beyond U_b; scores [B] fp32: the path's log-probability).
    An exact tie takes the blank predecessor, so a label goes to the earliest frame among equal paths.  Lengths are
    clamped to [0, T] / [0, U]; an utterance without frames (or whose best path crosses a -inf log-prob) gets score
    -inf and frames -1.  No host sync: capturable in a CUDA graph."""
    _lib.require_cuda(lp_blank, lp_label)
    lpb, lpl = _f32c(lp_blank), _f32c(lp_label)
    if lpb.dim() != 3 or lpl.shape != lpb.shape:
        raise RuntimeError("rnnt_viterbi: lp_blank and lp_label must both be [B, T, U+1]")
    B, T, U1 = lpb.shape
    dev = lpb.device
    tl, ul = _i32c(logit_lengths, dev), _i32c(target_lengths, dev)
    _len_check("rnnt_viterbi", B, tl, ul)
    frames = torch.empty((B, U1 - 1), dtype=torch.int32, device=dev)
    tok = torch.empty((B, U1 - 1), dtype=torch.float32, device=dev)
    scores = torch.empty((B,), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        ws = _ws(query("ctcvr_rnnt_viterbi_ws_bytes", B, T, U1), dev)
        call("ctcvr_rnnt_viterbi", ptr(lpb), ptr(lpl), ptr(tl), ptr(ul), ptr(frames), ptr(tok), ptr(scores), B, T, U1,
             ptr(ws), ws.numel(), stream())
    return frames, tok, scores


@torch.no_grad()
def rnnt_forced_align(enc_proj, pred_proj, w_out, b_out, targets, logit_lengths, target_lengths, blank: int,
                      precision="fp32", activation: str = "tanh", vocab_tiling: bool = False):
    """Forced alignment of `targets` [B,U] through the fused joint: the forward of `fused_joint_rnnt_loss` (same inputs,
    precisions, activations, vocab_tiling and errors; the logits never reach HBM) followed by `rnnt_viterbi` on its log-probs.
    Returns (frames [B,U] int32, token_logprobs [B,U] fp32, scores [B] fp32) as `rnnt_viterbi`; scores <= -cost of the
    loss on the same inputs (one path against the sum over all of them)."""
    if activation not in _ACT:
        raise ValueError(f"rnnt_forced_align: activation must be one of {sorted(_ACT)}, got {activation!r}")
    (_, _, _, _, _, tl, ul), _, _, lpb, lpl = _joint_fwd(enc_proj, pred_proj, w_out, b_out, targets, logit_lengths,
                                                         target_lengths, int(blank), _PREC[precision],
                                                         _ACT[activation], op="rnnt_forced_align",
                                                         vocab_tiling=vocab_tiling)
    return rnnt_viterbi(lpb, lpl, tl, ul)


@torch.no_grad()
def ctc_forced_align(log_probs, targets, input_lengths, target_lengths, blank: int):
    """Batched CTC forced alignment (torchaudio.functional.forced_align + merge_tokens for a whole padded batch).
    log_probs [B,T,V] fp32, targets [B,Umax] padded (Umax <= 511).  Returns (labels [B,T] int32: per frame the blank or
    the label of the best path, -1 for t >= T_b; frame_logprobs [B,T] fp32: its log-prob, 0 for t >= T_b; scores [B];
    spans [B,Umax,2] int32: first frame and last frame + 1 of each target token, -1 beyond U_b).  An exact tie takes
    the smaller jump, and between the two end states the final blank.  Lengths are clamped to [0, T] / [0, Umax] and a
    label outside [0, V) acts as blank, as in `ctc_loss_from_logits`.  An utterance without a path (T_b = 0, or fewer
    frames than labels plus repeated neighbours) gets score -inf and -1 everywhere.  No host sync."""
    _lib.require_cuda(log_probs)
    lp = _f32c(log_probs)
    if lp.dim() != 3:
        raise RuntimeError("ctc_forced_align: log_probs must be [B, T, V]")
    B, T, V = lp.shape
    dev = lp.device
    if targets.dim() != 2 or targets.shape[0] != B:
        raise ValueError(f"ctc_forced_align: targets must be [B, Umax] = [{B}, Umax] (padded), got {list(targets.shape)}")
    if not (0 <= blank < V):
        raise RuntimeError("ctc_forced_align: blank must be within [0, vocab)")
    tg = targets.detach().to(device=dev, dtype=torch.int64).contiguous()
    Umax = tg.shape[1]
    il, tl = _i32c(input_lengths, dev), _i32c(target_lengths, dev)
    _len_check("ctc_forced_align", B, il, tl)
    labels = torch.empty((B, T), dtype=torch.int32, device=dev)
    frame_lp = torch.empty((B, T), dtype=torch.float32, device=dev)
    scores = torch.empty((B,), dtype=torch.float32, device=dev)
    spans = torch.empty((B, Umax, 2), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        ws = _ws(query("ctcvr_ctc_viterbi_ws_bytes", B, T, Umax), dev)
        call("ctcvr_ctc_viterbi", ptr(lp), ptr(tg), ptr(il), ptr(tl), ptr(labels), ptr(frame_lp), ptr(scores), ptr(spans),
             B, T, V, Umax, int(blank), ptr(ws), ws.numel(), stream())
    return labels, frame_lp, scores, spans


def ctc_greedy_search(scores, lens, blank: int):
    """Per-frame argmax + collapse (model/rnnt_model.py:188-210).  scores [B,T,V] logits or log-probs."""
    _lib.require_cuda(scores)
    x = _f32c(scores)
    B, T, V = x.shape
    dev = x.device
    ln = _i32c(lens, dev)
    buf = torch.empty((B * T + B,), dtype=torch.int32, device=dev)      # tokens [B,T] | lengths [B]: one D2H copy
    toks, n = buf[:B * T].view(B, T), buf[B * T:]
    with torch.cuda.device(dev):
        call("ctcvr_ctc_greedy", ptr(x), ptr(ln), ptr(toks), ptr(n), B, T, V, int(blank), stream())
    host = buf.cpu().numpy()
    toks_h, n_h = host[:B * T].reshape(B, T), host[B * T:].tolist()
    return [toks_h[b, :n_h[b]].tolist() for b in range(B)]
