"""Whole-step CUDA graph of the fused seam (pre-projections -> fused joint / log-softmax forward -> lattice ->
fused backward -> pre-projection backward).  The reference's train loop launches ~40 kernels per step for this seam
(`rnnt_train.py:100-127` through `transducer.py:161-189`); here the step is captured once and replayed, so the host
cost per step is one graph launch plus the input copies.  B200-first: streams and graphs instead of a tracing compiler.
"""
from __future__ import annotations

from typing import Optional

import torch


class GraphedJointRnntStep:
    """Static-shape training step: `step(enc_out, pred_out, targets, logit_lengths, target_lengths)` copies the
    arguments into the captured buffers, replays the graph and returns the (device) loss scalar
    `sum_b cost_b / global_batch`.  Gradients land in `joint.<param>.grad`, `self.enc.grad`, `self.pred.grad`
    (static tensors, overwritten by every replay).  Passing no arguments replays on the resident inputs.

    Data parallel: with `grad_exchange=dist.PeerGradExchange(...)` the sum of the parameter gradients (and of the loss)
    over the ranks is the LAST kernel of the captured step (`csrc/peer_reduce.cu`, flags and 16-byte loads / stores over
    NVLink peer memory).  An NCCL collective cannot take that place: a replayed graph that contained it (grouped in round
    1, one flat bucket in round 2) hung the 2-GPU bench both times; with `grad_exchange=None` call
    `dist.GradAllReducer.reduce()` after `step()`.
    Construct it before (or after dropping every reference to) eager autograd graphs over the same parameters: a live
    graph pins their AccumulateGrad nodes to the stream it ran on, and the capture may not synchronise with that stream.
    `input_dtype=torch.bfloat16` keeps the captured input buffers in bf16 (the bf16 path rounds its inputs to bf16 in
    the first kernel anyway): a host pipeline then stages half the bytes per step.  `precision="bf16x3"` (tensor cores
    at fp32 accuracy) needs fp32 inputs.  `vocab_tiling=True` lets 'bf16' / 'bf16x3' take vocabularies beyond 416
    (functional.fused_joint_rnnt_loss).
    `predictor=RNNPredictor(...)` puts the label side of Transducer._compute_rnnt_loss (transducer.py:168-172) into the
    step: `ys_in = [blank, targets]` is built in the captured region, the predictor (embedding, the LSTM sequence kernels
    of csrc/lstm_seq.cu, projection) produces `pred_out`, and its parameters get their gradients (and join the gradient
    exchange: 13.2 MB with the joint at H = 512) - `pred_out` is then not an input (`step(enc_out, None, targets, ...)`)."""

    def __init__(self, joint, B: int, T: int, U: int, blank: int, global_batch: Optional[int] = None,
                 precision: str = "fp32", clamp: float = -1.0, warmup: int = 3,
                 input_dtype: torch.dtype = torch.float32, grad_exchange=None, predictor=None,
                 vocab_tiling: bool = False):
        if precision == "bf16x3" and input_dtype != torch.float32:
            raise ValueError("precision='bf16x3' keeps fp32 accuracy end to end: input_dtype must be torch.float32")
        p0 = next(joint.parameters())
        dev = p0.device
        if dev.type != "cuda":
            raise RuntimeError("ctcvr_b200.GraphedJointRnntStep needs the joint on a CUDA (B200) device")
        E = joint.enc_ffn.in_features if joint.enc_ffn is not None else joint.ffn_out.in_features
        P = joint.pred_ffn.in_features if joint.pred_ffn is not None else joint.ffn_out.in_features
        self.joint, self.blank, self.precision, self.clamp = joint, int(blank), precision, float(clamp)
        self.vocab_tiling = bool(vocab_tiling)
        self.gB = float(global_batch if global_batch is not None else B)
        self.grad_exchange = grad_exchange
        self.predictor = predictor
        self.enc = torch.zeros(B, T, E, device=dev, dtype=input_dtype, requires_grad=True)
        if predictor is None:
            self.pred = torch.zeros(B, U + 1, P, device=dev, dtype=input_dtype, requires_grad=True)
            self.ys_in = None
        else:
            if next(predictor.parameters()).device != dev:
                raise RuntimeError("ctcvr_b200.GraphedJointRnntStep: predictor and joint must live on the same device")
            self.pred = None
            self.ys_in = torch.full((B, U + 1), self.blank, dtype=torch.int64, device=dev)
        self.targets = torch.full((B, U), max(self.blank + 1, 1) % joint.ffn_out.out_features, dtype=torch.int32, device=dev)
        self.logit_lengths = torch.full((B,), T, dtype=torch.int32, device=dev)
        self.target_lengths = torch.full((B,), U, dtype=torch.int32, device=dev)
        self.loss = None
        self._seed = torch.full((B,), 1.0 / self.gB, dtype=torch.float32, device=dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):
                self._eager()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._eager()
        # the gradient tensors this graph writes: step() re-points `.grad` at them, so several graphed steps over the same
        # parameters (e.g. one per input staging buffer of a double-buffered loader) can be replayed in turn
        self._param_grads = [(p, p.grad) for p in self.parameters()]
        self._loss_buf = self.loss

    def parameters(self):
        """The parameters whose gradients the step writes: the joint's, then the predictor's (when it is in the step)."""
        ps = list(self.joint.parameters())
        if self.predictor is not None:
            ps += list(self.predictor.parameters())
        return ps

    def _eager(self):
        for p in self.parameters():
            p.grad = None
        self.enc.grad = None
        if self.predictor is None:
            self.pred.grad = None
            pred = self.pred
        else:
            # add_blank (transducer.py:8-19): column 0 stays `blank`, the labels follow (int32 -> int64 in the copy)
            self.ys_in[:, 1:].copy_(self.targets)
            pred = self.predictor(self.ys_in)
        costs = self.joint.rnnt_loss_fused(self.enc, pred, self.targets, self.logit_lengths, self.target_lengths,
                                           self.blank, clamp=self.clamp, reduction="none", precision=self.precision,
                                           vocab_tiling=self.vocab_tiling)
        # loss = sum_b cost_b / global_batch: the constant d loss / d cost_b vector seeds the backward directly (no
        # sum / div / fill / mul / expand kernels of the scalar-loss autograd chain), the value is one dot product
        torch.autograd.backward(costs, grad_tensors=self._seed)
        self.loss = torch.dot(costs.detach(), self._seed)
        if self.grad_exchange is not None:
            self.grad_exchange.reduce([p.grad for p in self.parameters() if p.grad is not None] + [self.loss.view(1)])

    @torch.no_grad()
    def load(self, enc_out, pred_out, targets, logit_lengths, target_lengths):
        """Copy one batch (host-pinned or device tensors) into the captured input buffers."""
        self.enc.copy_(enc_out, non_blocking=True)
        if self.predictor is None:
            self.pred.copy_(pred_out, non_blocking=True)
        self.targets.copy_(targets, non_blocking=True)
        self.logit_lengths.copy_(logit_lengths, non_blocking=True)
        self.target_lengths.copy_(target_lengths, non_blocking=True)

    @torch.no_grad()
    def load_padded(self, enc_out, pred_out, targets, logit_lengths, target_lengths):
        """Copy a batch whose T / U are SMALLER than the captured ones into the leading corner of the input buffers.
        The kernels only visit cells below the per-utterance lengths, so whatever an earlier batch left beyond them is
        never read (the buffers start as zeros and only ever hold finite values)."""
        T, U = enc_out.shape[1], targets.shape[1]
        U1 = pred_out.shape[1] if pred_out is not None else U + 1
        if enc_out.shape[0] != self.enc.shape[0] or T > self.enc.shape[1] or U > self.targets.shape[1] or U1 != U + 1:
            raise RuntimeError(f"load_padded: batch {tuple(enc_out.shape)} / U = {U} does not fit the captured "
                               f"{tuple(self.enc.shape)} / U = {self.targets.shape[1]}")
        self.enc[:, :T].copy_(enc_out, non_blocking=True)
        if self.predictor is None:
            self.pred[:, :U1].copy_(pred_out, non_blocking=True)
        if U:
            self.targets[:, :U].copy_(targets, non_blocking=True)
        self.logit_lengths.copy_(logit_lengths, non_blocking=True)
        self.target_lengths.copy_(target_lengths, non_blocking=True)

    def step(self, enc_out=None, pred_out=None, targets=None, logit_lengths=None, target_lengths=None):
        if enc_out is not None:
            self.load(enc_out, pred_out, targets, logit_lengths, target_lengths)
        self.graph.replay()
        for p, g in self._param_grads:
            p.grad = g
        self.loss = self._loss_buf
        return self.loss

    def input_buffers(self):
        """The captured input tensors [enc, pred, targets, logit_lengths, target_lengths]: a loader may copy the next
        batch straight into them (e.g. H2D on a copy stream) once the previous replay of THIS graph has finished."""
        return [self.enc, self.pred, self.targets, self.logit_lengths, self.target_lengths]   # pred is None with a predictor

    __call__ = step



class BucketedJointRnntStep:
    """Graph replay for a train loop whose batches change shape: (B, T, U) is rounded up to a bucket (T to a multiple of
    `t_bucket` frames, U to a multiple of `u_bucket` labels), one `GraphedJointRnntStep` is captured per bucket on first
    use and kept (least recently used evicted beyond `max_graphs`), and a batch is copied into the leading corner of its
    bucket's buffers.  The per-utterance lengths are device tensors read by the kernels, so the padding costs no tiles:
    a ragged batch runs in the time of its real cells, without the ~40 launches and workspace allocations of the eager
    path (`bench.py` prints both).

    `step()` returns the device loss scalar; parameter gradients land in `joint.<param>.grad`; the gradients of the inputs
    are `enc_grad` [B,T,E] / `pred_grad` [B,U+1,P] (views into the bucket's buffers, valid until its next replay)."""

    def __init__(self, joint, blank: int, t_bucket: int = 16, u_bucket: int = 8, max_graphs: int = 16, **graph_kwargs):
        if t_bucket < 1 or u_bucket < 1 or max_graphs < 1:
            raise ValueError("t_bucket, u_bucket and max_graphs must be positive")
        self.joint, self.blank = joint, int(blank)
        self.t_bucket, self.u_bucket, self.max_graphs = int(t_bucket), int(u_bucket), int(max_graphs)
        self.graph_kwargs = graph_kwargs
        self._graphs = {}                       # (B, Tb, Ub) -> GraphedJointRnntStep, in LRU order
        self.captures = 0
        self.enc_grad = self.pred_grad = None

    def bucket_of(self, B: int, T: int, U: int):
        up = lambda x, m: max(m, (x + m - 1) // m * m)
        return (int(B), up(T, self.t_bucket), up(U, self.u_bucket))

    def step(self, enc_out, pred_out, targets, logit_lengths, target_lengths):
        B, T = enc_out.shape[0], enc_out.shape[1]
        U = targets.shape[1]
        key = self.bucket_of(B, T, U)
        g = self._graphs.pop(key, None)
        if g is None:
            if len(self._graphs) >= self.max_graphs:
                self._graphs.pop(next(iter(self._graphs)))          # least recently used
            g = GraphedJointRnntStep(self.joint, key[0], key[1], key[2], self.blank, **self.graph_kwargs)
            self.captures += 1
        self._graphs[key] = g
        g.load_padded(enc_out, pred_out, targets, logit_lengths, target_lengths)
        loss = g.step()
        self.enc_grad = g.enc.grad[:, :T]
        self.pred_grad = g.pred.grad[:, :U + 1] if g.pred is not None else None
        return loss

    __call__ = step
