"""Oracle (TEST INFRASTRUCTURE ONLY) for the RNN-T half of the hot path.

Every function cites the reference file:line it restates (paths relative to
/root/reference; `site-packages/` = the installed torchaudio / torch wheels
which hold the arithmetic the reference delegates to and which are NOT part of
the reference tree).

Parity pinning: see `oracle/__init__.py`.  The reference has no RNN-T golden
vectors; `tests/test_oracle_cpu.py` pins `rnnt_lattice_restated` against
`rnnt_loss_reference_call` (torchaudio, called exactly as the reference does)
and against `tests/golden/rnnt_*.npz` produced by the reference modules.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch

Weights = Dict[str, torch.Tensor]


# --------------------------------------------------------------------------- joint (A1)
def joint_forward(enc_out: torch.Tensor, pred_out: torch.Tensor, w: Weights,
                  pre_project: bool = True) -> torch.Tensor:
    """model/component/joint.py:48-69 (prejoin_linear=True, postjoin_linear=False,
    joint_mode='add', activation='tanh' — the only configuration both models build,
    model/rnnt_model.py:122-131, model/online_rnnt_model.py:121-126).
    Returns raw logits [B,T,U,V]; no log_softmax (it is fused in rnnt_loss)."""
    if pre_project:
        enc_out = torch.nn.functional.linear(enc_out, w["enc_ffn.weight"], w["enc_ffn.bias"])
        pred_out = torch.nn.functional.linear(pred_out, w["pred_ffn.weight"], w["pred_ffn.bias"])
    out = enc_out.unsqueeze(2) + pred_out.unsqueeze(1)          # joint.py:57-62
    out = torch.tanh(out)                                        # joint.py:67
    return torch.nn.functional.linear(out, w["ffn_out.weight"], w["ffn_out.bias"])  # joint.py:68


def add_blank(text: torch.Tensor, blank: int) -> torch.Tensor:
    """model/component/transducer.py:8-19 — prepend blank; padding is NOT remapped."""
    ys = torch.zeros((text.size(0), text.size(1) + 1), dtype=text.dtype)
    ys[:, 0] = blank
    ys[:, 1:] = text
    return ys


# --------------------------------------------------------------------------- loss (A2)
def rnnt_loss_reference_call(logits, targets, logit_lengths, target_lengths, blank: int,
                             clamp: float = -1.0, reduction: str = "mean"):
    """The reference's own call: model/component/transducer.py:180-187 (and
    model/online_rnnt_model.py:247-255 with `clamp`).  Arithmetic lives in
    torchaudio 2.11.0 (site-packages/torchaudio/functional/functional.py:1747-1800)."""
    import torchaudio
    return torchaudio.functional.rnnt_loss(logits, targets.to(torch.int32),
                                           logit_lengths.to(torch.int32),
                                           target_lengths.to(torch.int32),
                                           blank=blank, clamp=clamp, reduction=reduction)


def _logaddexp(a, b):
    return torch.logaddexp(a, b)


def rnnt_lattice_restated(logits: torch.Tensor, targets: torch.Tensor,
                          logit_lengths: torch.Tensor, target_lengths: torch.Tensor,
                          blank: int, clamp: float = -1.0, dtype=torch.float64):
    """Restatement of the transducer loss the reference delegates to
    torchaudio.functional.rnnt_loss (fused_log_softmax=True), SURVEY.md §8 A2:

      lse(t,u)       = logsumexp_v logits(t,u,v)
      lp_blank(t,u)  = logits(t,u,blank) - lse ; lp_label(t,u) = logits(t,u,y_{u+1}) - lse
      alpha(0,0)=0 ; alpha(t,u) = LSE(alpha(t-1,u)+lp_blank(t-1,u), alpha(t,u-1)+lp_label(t,u-1))
      beta(T-1,U)=lp_blank(T-1,U); beta(t,u) = LSE(beta(t+1,u)+lp_blank(t,u), beta(t,u+1)+lp_label(t,u))
      cost = -beta(0,0)
      grad(t,u,v) = exp(alpha+beta(t,u) + logits_v - lse + cost)
                    - [v==blank] exp(alpha(t,u)+lp_blank(t,u)+beta(t+1,u)+cost)   (beta(T,U):=0)
                    - [v==y_{u+1}] exp(alpha(t,u)+lp_label(t,u)+beta(t,u+1)+cost)
      zero at padded cells; optional clamp.

    Returns dict(costs[B], grads[B,T,U+1,V], alpha, beta, lp_blank, lp_label, lse)."""
    B, T, U1, V = logits.shape
    x = logits.detach().to(dtype)
    lse = torch.logsumexp(x, dim=-1)                                  # [B,T,U1]
    lp_blank = x[..., blank] - lse
    tgt = targets.to(torch.int64)
    if tgt.size(1) < U1:                                              # pad to U1 for gather
        tgt = torch.cat([tgt, torch.zeros(B, U1 - tgt.size(1), dtype=torch.int64)], dim=1)
    lp_label = torch.gather(x, 3, tgt[:, None, :, None].expand(B, T, U1, 1)).squeeze(-1) - lse
    ninf = float("-inf")
    alpha = torch.full((B, T, U1), ninf, dtype=dtype)
    beta = torch.full((B, T, U1), ninf, dtype=dtype)
    costs = torch.zeros(B, dtype=dtype)
    grads = torch.zeros((B, T, U1, V), dtype=dtype)
    for b in range(B):
        Tb, Ub = int(logit_lengths[b]), int(target_lengths[b])
        if Tb == 0:                                                    # no frames: cost 0, zero gradient
            continue
        a = alpha[b]
        a[0, 0] = 0.0
        for t in range(1, Tb):
            a[t, 0] = a[t - 1, 0] + lp_blank[b, t - 1, 0]
        for u in range(1, Ub + 1):
            a[0, u] = a[0, u - 1] + lp_label[b, 0, u - 1]
        for d in range(2, Tb + Ub):                                    # anti-diagonals t+u=d
            t = torch.arange(max(1, d - Ub), min(Tb - 1, d - 1) + 1)
            u = d - t
            a[t, u] = _logaddexp(a[t - 1, u] + lp_blank[b, t - 1, u], a[t, u - 1] + lp_label[b, t, u - 1])
        be = beta[b]
        be[Tb - 1, Ub] = lp_blank[b, Tb - 1, Ub]
        for t in range(Tb - 2, -1, -1):
            be[t, Ub] = be[t + 1, Ub] + lp_blank[b, t, Ub]
        for u in range(Ub - 1, -1, -1):
            be[Tb - 1, u] = be[Tb - 1, u + 1] + lp_label[b, Tb - 1, u]
        for d in range(Tb + Ub - 3, -1, -1):
            t = torch.arange(max(0, d - (Ub - 1)), min(Tb - 2, d) + 1)
            u = d - t
            be[t, u] = _logaddexp(be[t + 1, u] + lp_blank[b, t, u], be[t, u + 1] + lp_label[b, t, u])
        cost = -be[0, 0]
        costs[b] = cost
        ab = a[:Tb, :Ub + 1] + be[:Tb, :Ub + 1]
        g = torch.exp(ab[..., None] + x[b, :Tb, :Ub + 1, :] - lse[b, :Tb, :Ub + 1, None] + cost)
        beta_next_t = torch.full((Tb, Ub + 1), ninf, dtype=dtype)
        beta_next_t[:-1] = be[1:Tb, :Ub + 1]
        beta_next_t[Tb - 1, Ub] = 0.0
        g[..., blank] -= torch.exp(a[:Tb, :Ub + 1] + lp_blank[b, :Tb, :Ub + 1] + beta_next_t + cost)
        if Ub > 0:
            gl = torch.exp(a[:Tb, :Ub] + lp_label[b, :Tb, :Ub] + be[:Tb, 1:Ub + 1] + cost)   # [Tb,Ub]
            idx = tgt[b, :Ub][None, :, None].expand(Tb, Ub, 1)
            g[:, :Ub, :].scatter_add_(2, idx, -gl[..., None])
        if clamp > 0:
            g = g.clamp(-clamp, clamp)
        grads[b, :Tb, :Ub + 1] = g
    return dict(costs=costs, grads=grads, alpha=alpha, beta=beta,
                lp_blank=lp_blank, lp_label=lp_label, lse=lse)


def fused_joint_rnnt_restated(enc_out, pred_out, w: Weights, targets, logit_lengths, target_lengths,
                              blank: int, clamp: float = -1.0, dtype=torch.float64, grad_costs=None):
    """model/component/transducer.py:161-189 from predictor output to scalar loss
    (reduction='mean'), with gradients wrt enc_out / pred_out / the six joint tensors,
    obtained by chaining the closed-form logits gradient through autograd of `joint_forward`.
    `grad_costs` [B] is the cotangent of the per-utterance costs (None: 1/B each, the mean).  As in
    torchaudio, the logits gradient is clamped first and then scaled by it."""
    ws = {k: v.detach().to(dtype).requires_grad_(True) for k, v in w.items()}
    e = enc_out.detach().to(dtype).requires_grad_(True)
    p = pred_out.detach().to(dtype).requires_grad_(True)
    logits = joint_forward(e, p, ws)
    r = rnnt_lattice_restated(logits, targets, logit_lengths, target_lengths, blank, clamp, dtype)
    B = logits.size(0)
    if grad_costs is None:
        logits.backward(r["grads"] / B)
    else:
        logits.backward(r["grads"] * torch.as_tensor(grad_costs).to(dtype).reshape(B, 1, 1, 1))
    out = dict(loss=r["costs"].mean(), costs=r["costs"], d_enc_out=e.grad, d_pred_out=p.grad)
    for k, v in ws.items():
        out["d_" + k] = v.grad
    return out


def fused_joint_rnnt_reference_call(enc_out, pred_out, w: Weights, targets, logit_lengths,
                                    target_lengths, blank: int, clamp: float = -1.0):
    """Same seam as above but through the third-party ops exactly as the reference wires
    them (joint.py:48-69 -> transducer.py:174-187), fp32, autograd backward."""
    ws = {k: v.detach().clone().float().requires_grad_(True) for k, v in w.items()}
    e = enc_out.detach().clone().float().requires_grad_(True)
    p = pred_out.detach().clone().float().requires_grad_(True)
    logits = joint_forward(e, p, ws)
    loss = rnnt_loss_reference_call(logits, targets, logit_lengths, target_lengths, blank, clamp, "mean")
    loss.backward()
    out = dict(loss=loss.detach(), d_enc_out=e.grad, d_pred_out=p.grad)
    for k, v in ws.items():
        out["d_" + k] = v.grad
    return out


# --------------------------------------------------------------------------- predictor step
def n_layers_of(pw: Weights) -> int:
    n = 0
    while f"rnn.weight_ih_l{n}" in pw:
        n += 1
    return n


def predictor_init_state(pw: Weights, batch: int = 1) -> List[torch.Tensor]:
    """model/component/predictor.py:65-77 / wenet/transducer/predictor.py:165-183."""
    L = n_layers_of(pw)
    H = pw["rnn.weight_hh_l0"].size(1)
    dt = pw["rnn.weight_hh_l0"].dtype
    return [torch.zeros(L, batch, H, dtype=dt), torch.zeros(L, batch, H, dtype=dt)]


def predictor_forward_step(pw: Weights, token: torch.Tensor, state: List[torch.Tensor]):
    """model/component/predictor.py:79-98 with padding==0 (every caller passes zeros,
    SURVEY.md §8 notes): embed -> LSTM cell(s) -> projection.  token: [N] int64;
    state: [h,c] each [L,N,H].  Returns (out [N,P], [h',c'])."""
    x = pw["embed.weight"][token]                                  # [N,E]
    h0, c0 = state
    hs, cs = [], []
    for l in range(n_layers_of(pw)):
        gates = (x @ pw[f"rnn.weight_ih_l{l}"].T + pw[f"rnn.bias_ih_l{l}"]
                 + h0[l] @ pw[f"rnn.weight_hh_l{l}"].T + pw[f"rnn.bias_hh_l{l}"])
        i, f, g, o = gates.chunk(4, dim=-1)
        c = torch.sigmoid(f) * c0[l] + torch.sigmoid(i) * torch.tanh(g)
        h = torch.sigmoid(o) * torch.tanh(c)
        hs.append(h)
        cs.append(c)
        x = h
    out = x @ pw["projection.weight"].T + pw["projection.bias"]
    return out, [torch.stack(hs), torch.stack(cs)]


def predictor_forward(pw: Weights, ys_in: torch.Tensor) -> torch.Tensor:
    """model/component/predictor.py:43-63 (zero initial state, dropout off)."""
    B, L = ys_in.shape
    st = predictor_init_state(pw, B)
    outs = []
    for i in range(L):
        o, st = predictor_forward_step(pw, ys_in[:, i], st)
        outs.append(o)
    return torch.stack(outs, dim=1)


def predictor_forward_backward(pw: Weights, ys_in: torch.Tensor, d_out: torch.Tensor):
    """Forward + backward of model/component/predictor.py:43-63 through the restated cell above: returns
    (out [B,U1,P], {parameter name: gradient of sum(out * d_out)}).  The arithmetic runs in the dtype of `pw`
    (float64 weights give the ground truth the section 8f row 2 kernels are compared with)."""
    leaf = {k: v.detach().clone().requires_grad_(True) for k, v in pw.items()}
    out = predictor_forward(leaf, ys_in)
    (out * d_out.to(out.dtype)).sum().backward()
    return out.detach(), {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in leaf.items()}


def _joint_step(jw: Weights, enc_t: torch.Tensor, pred_u: torch.Tensor) -> torch.Tensor:
    """joint on [1,1,D] x [N,1,P] -> [N,V] raw logits (joint.py:48-69 with T=U=1)."""
    return joint_forward(enc_t.reshape(1, 1, -1).expand(pred_u.size(0), 1, -1),
                         pred_u.reshape(pred_u.size(0), 1, -1), jw)[:, 0, 0, :]


# --------------------------------------------------------------------------- greedy (A5, A6, A6')
def greedy_search_offline(pw: Weights, jw: Weights, blank: int, encoder_out: torch.Tensor,
                          encoder_out_lens: torch.Tensor, n_steps: int = 64) -> List[List[int]]:
    """model/component/transducer.py:22-70 (basic_greedy_search): fresh zero state and
    token=blank per utterance; per frame up to n_steps predictor+joint steps; argmax over
    RAW logits; blank -> next frame; else emit, advance token/state."""
    hyps = []
    for b in range(encoder_out.size(0)):
        hyp, state = [], predictor_init_state(pw, 1)
        hyp, state, _ = greedy_chunk_streaming(pw, jw, blank, encoder_out[b, :int(encoder_out_lens[b])],
                                               state, blank, n_steps)
        hyps.append(hyp)
    return hyps


def greedy_chunk_streaming(pw: Weights, jw: Weights, blank: int, enc_chunk: torch.Tensor,
                           state: Optional[List[torch.Tensor]], prev_token: int, n_steps: int = 10):
    """model/online_rnnt_model.py:166-222 below the encoder call: state (h,c) and the last
    emitted token persist across chunks.  enc_chunk: [Tc,H].  Returns (tokens, state, last_token).
    wenet/transducer/search/greedy_search.py:6-54 is the same walk (predictor re-run skipped
    after a blank, log_softmax before argmax: neither changes the result)."""
    if state is None:
        state = predictor_init_state(pw, 1)
    tok = prev_token
    out: List[int] = []
    for t in range(enc_chunk.size(0)):
        for _ in range(n_steps):
            pred, new_state = predictor_forward_step(pw, torch.tensor([tok]), state)
            logits = _joint_step(jw, enc_chunk[t], pred)[0]
            k = int(torch.argmax(logits))
            if k == blank:
                break
            out.append(k)
            tok = k
            state = new_state
    return out, state, tok


# --------------------------------------------------------------------------- online beam (A7)
class Hyp:
    """model/online_rnnt_model.py:41-55 (BeamHypothesis)."""
    __slots__ = ("tokens", "log_prob", "state")

    def __init__(self, tokens, log_prob, state):
        self.tokens, self.log_prob, self.state = tokens, log_prob, state


def beam_chunk_online(pw: Weights, jw: Weights, blank: int, enc_chunk: torch.Tensor,
                      beam_in: Optional[List[Hyp]], beam_size: int = 4, n_steps: int = 10) -> List[Hyp]:
    """model/online_rnnt_model.py:389-522 below the encoder call.  Scores are Python floats
    (fp64 sums of fp32 log-probs); the sort is Python's stable sort, descending; dedupe keeps
    the first (highest-scoring) candidate per token tuple; no log-add merge."""
    if beam_in is None:
        beam_in = [Hyp([], 0.0, predictor_init_state(pw, 1))]
    beam = beam_in
    for t in range(enc_chunk.size(0)):
        cands: List[Hyp] = []
        for hyp in beam:
            toks = list(hyp.tokens)
            lp_acc = hyp.log_prob
            st = hyp.state
            last = toks[-1] if toks else blank
            for _ in range(n_steps):
                pred, nst = predictor_forward_step(pw, torch.tensor([last]), st)
                logp = torch.log_softmax(_joint_step(jw, enc_chunk[t], pred)[0], dim=-1)
                bl = logp[blank].item()
                cands.append(Hyp(list(toks), lp_acc + bl, st))
                mask = torch.ones_like(logp, dtype=torch.bool)
                mask[blank] = False
                nb = logp[mask]
                nb_idx = torch.arange(logp.size(0))[mask]
                k = min(beam_size, nb.numel())
                tv, ti = torch.topk(nb, k)
                for i in range(k):
                    cands.append(Hyp(toks + [int(nb_idx[ti[i]])], lp_acc + tv[i].item(), nst))
                if bl >= logp.max().item() - 1e-6:
                    break
                bi = int(torch.argmax(nb))
                toks.append(int(nb_idx[bi]))
                lp_acc += nb[bi].item()
                st = nst
                last = toks[-1]
        cands.sort(key=lambda h: h.log_prob, reverse=True)
        seen, uniq = set(), []
        for c in cands:
            key = tuple(c.tokens)
            if key not in seen:
                seen.add(key)
                uniq.append(c)
                if len(uniq) >= beam_size:
                    break
        beam = uniq[:beam_size]
    return beam


# --------------------------------------------------------------------------- wenet prefix beam (A8)
def log_add_list(xs: Sequence[float]) -> float:
    """wenet/utils/common.py:302-310 semantics over a sequence of floats (fp64 `math`)."""
    if all(a == -float("inf") for a in xs):
        return -float("inf")
    m = max(xs)
    return m + math.log(sum(math.exp(a - m) for a in xs))


def prefix_beam_search_wenet(pw: Weights, jw: Weights, blank: int, encoder_out: torch.Tensor,
                             ctc_logp: torch.Tensor, beam_size: int = 5, ctc_weight: float = 0.3,
                             transducer_weight: float = 0.7):
    """wenet/transducer/search/prefix_beam_search.py:42-148 below the encoder call
    (encoder_out: [T,H]; ctc_logp: [T,V] = ctc.log_softmax(encoder_out)).  One symbol per frame;
    CTC shallow fusion logp = log(tw*exp(logp) + cw*exp(ctc_logp[t])) (:99-101); per-hyp topk;
    identical hyps merged with log-add (:130-142); stable sort desc; keep beam.
    NOTE: the vendored reference calls `log_add([a, b])` with a LIST while its own
    `log_add(*args)` (wenet/utils/common.py:302) takes varargs, so the reference raises
    TypeError as soon as two candidates share a hyp; upstream wenet's list form is what is
    restated here (and what tests/golden/make_golden.py patches in to generate fixtures).
    Returns list of (hyp tokens incl. leading blank, score)."""
    beam = [([blank], 0.0, predictor_init_state(pw, 1))]
    for i in range(encoder_out.size(0)):
        toks = torch.tensor([b[0][-1] for b in beam])
        h = torch.cat([b[2][0] for b in beam], dim=1)
        c = torch.cat([b[2][1] for b in beam], dim=1)
        scores = torch.tensor([b[1] for b in beam])                       # fp32, as the reference
        pred, (nh, nc) = predictor_forward_step(pw, toks, [h, c])
        logp = torch.log_softmax(_joint_step(jw, encoder_out[i], pred), dim=-1)
        logp = torch.log(transducer_weight * torch.exp(logp) + ctc_weight * torch.exp(ctc_logp[i].unsqueeze(0)))
        tv, ti = logp.topk(beam_size)
        sc = scores.unsqueeze(1) + tv
        beam_a = []
        for j, (hyp, _, cache) in enumerate(beam):
            for t in range(beam_size):
                k = int(ti[j, t])
                if k == blank:
                    beam_a.append([list(hyp), sc[j, t].item(), cache])
                else:
                    beam_a.append([hyp + [k], sc[j, t].item(), [nh[:, j:j + 1], nc[:, j:j + 1]]])
        fusion = [beam_a[0]]
        for s1 in beam_a[1:]:
            for f in fusion:
                if s1[0] == f[0]:
                    f[1] = log_add_list([f[1], s1[1]])
                    break
            else:
                fusion.append(s1)
        fusion.sort(key=lambda s: s[1], reverse=True)
        beam = [tuple(f) for f in fusion[:beam_size]]
    return [(b[0], b[1]) for b in beam]
