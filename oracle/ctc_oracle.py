"""Oracle (TEST INFRASTRUCTURE ONLY) for the CTC half of the hot path.

Citations are relative to /root/reference.  Pinned by the reference's own known
answers on `example2.pt` (`3.ipynb:87,159`, `3_v2.ipynb:150`; fixture copy in
`tests/golden/example2.npz`) and by `torch.nn.CTCLoss` called exactly as the
reference calls it.
"""
from __future__ import annotations

import math
from collections import defaultdict
from typing import List

import numpy as np
import torch


# --------------------------------------------------------------------------- loss (A4)
def ctc_head_reference_call(hs_pad, hlens, ys_pad, ys_lens, w, b, blank: int, mode: str = "offline"):
    """model/rnnt_model.py:40-60 (mode='offline': reduction='sum' then /B) and
    model/online_rnnt_model.py:25-32 (mode='online': reduction='mean'), dropout p=0.
    Returns (loss, ys_hat [B,T,V] log-probs)."""
    ys_hat = torch.nn.functional.linear(hs_pad, w, b).transpose(0, 1).log_softmax(2)
    red = "sum" if mode == "offline" else "mean"
    loss = torch.nn.functional.ctc_loss(ys_hat, ys_pad, hlens, ys_lens, blank=blank,
                                        reduction=red, zero_infinity=True)
    if mode == "offline":
        loss = loss / ys_hat.size(1)
    return loss, ys_hat.transpose(0, 1)


def ctc_loss_restated(log_probs: np.ndarray, targets: np.ndarray, in_lens, tgt_lens, blank: int):
    """Textbook CTC alpha/beta in fp64 over the extended label sequence l' (blank-interleaved,
    S=2U+1), the algorithm torch.nn.CTCLoss implements (Graves 2006, eq. 6-16).
    log_probs: [B,T,V] log-softmax outputs.  Returns (nll[B], grad wrt *logits* [B,T,V]) where
    grad = softmax - (1/p(l|x)) sum_{s: l'_s = v} alpha_t(s) beta_t(s)/y_t(v); inf losses are
    zeroed (zero_infinity=True) together with their gradients; frames t>=T_b get zero grad."""
    B, T, V = log_probs.shape
    nll = np.zeros(B)
    grad = np.zeros((B, T, V))
    ninf = -np.inf

    def lae(a, b):
        if a == ninf:
            return b
        if b == ninf:
            return a
        m = max(a, b)
        return m + math.log(math.exp(a - m) + math.exp(b - m))

    for b in range(B):
        Tb, Ub = int(in_lens[b]), int(tgt_lens[b])
        lab = [blank]
        for u in range(Ub):
            lab += [int(targets[b, u]), blank]
        S = len(lab)
        lp = log_probs[b].astype(np.float64)
        al = np.full((Tb, S), ninf)
        be = np.full((Tb, S), ninf)
        if Tb == 0:
            nll[b] = 0.0 if Ub == 0 else np.inf
        else:
            al[0, 0] = lp[0, lab[0]]
            if S > 1:
                al[0, 1] = lp[0, lab[1]]
            for t in range(1, Tb):
                for s in range(S):
                    a = al[t - 1, s]
                    if s >= 1:
                        a = lae(a, al[t - 1, s - 1])
                    if s >= 2 and lab[s] != lab[s - 2]:
                        a = lae(a, al[t - 1, s - 2])
                    al[t, s] = a + lp[t, lab[s]] if a != ninf else ninf
            be[Tb - 1, S - 1] = lp[Tb - 1, lab[S - 1]]
            if S > 1:
                be[Tb - 1, S - 2] = lp[Tb - 1, lab[S - 2]]
            for t in range(Tb - 2, -1, -1):
                for s in range(S):
                    a = be[t + 1, s]
                    if s + 1 < S:
                        a = lae(a, be[t + 1, s + 1])
                    if s + 2 < S and lab[s] != lab[s + 2]:
                        a = lae(a, be[t + 1, s + 2])
                    be[t, s] = a + lp[t, lab[s]] if a != ninf else ninf
            ll = al[Tb - 1, S - 1]
            if S > 1:
                ll = lae(ll, al[Tb - 1, S - 2])
            nll[b] = -ll
        if not np.isfinite(nll[b]):
            nll[b] = 0.0
            continue
        for t in range(Tb):
            acc = np.full(V, ninf)
            for s in range(S):
                acc[lab[s]] = lae(acc[lab[s]], al[t, s] + be[t, s])
            grad[b, t] = np.exp(lp[t]) - np.exp(acc - lp[t] + nll[b])
    return nll, grad


# --------------------------------------------------------------------------- greedy (A10)
def ctc_greedy_collapse(frame_ids: List[int], blank: int) -> List[int]:
    """model/rnnt_model.py:199-207 / model/online_rnnt_model.py:661-669: prev is updated on
    every frame (blank included), i.e. standard CTC collapse (== wenet/utils/ctc_utils.py:23-33)."""
    out, prev = [], -1
    for tok in frame_ids:
        if tok != blank and tok != prev:
            out.append(tok)
        prev = tok
    return out


def ctc_greedy_search(log_probs: torch.Tensor, lens, blank: int) -> List[List[int]]:
    """model/rnnt_model.py:188-210: per-frame argmax (topk(1)) then collapse."""
    ids = log_probs.argmax(dim=2)
    return [ctc_greedy_collapse(ids[b, :int(lens[b])].tolist(), blank) for b in range(ids.size(0))]


# --------------------------------------------------------------------------- prefix beam (A9)
def _log_add(*args) -> float:
    """wenet/utils/common.py:302-310."""
    if all(a == -float("inf") for a in args):
        return -float("inf")
    a_max = max(args)
    return a_max + math.log(sum(math.exp(a - a_max) for a in args))


class _PS:
    """wenet/transformer/search.py:62-104 (PrefixScore) without the context graph
    (every caller in scope passes context_graph=None)."""
    __slots__ = ("s", "ns", "v_s", "v_ns", "cur_token_prob", "times_s", "times_ns")

    def __init__(self, s=-math.inf, ns=-math.inf, v_s=-math.inf, v_ns=-math.inf):
        self.s, self.ns, self.v_s, self.v_ns = s, ns, v_s, v_ns
        self.cur_token_prob = -math.inf
        self.times_s, self.times_ns = [], []

    def score(self):
        return _log_add(self.s, self.ns)

    def viterbi_score(self):
        return self.v_s if self.v_s > self.v_ns else self.v_ns

    def times(self):
        return self.times_s if self.v_s > self.v_ns else self.times_ns


def ctc_prefix_beam_search(ctc_probs: torch.Tensor, ctc_lens, beam_size: int, blank_id: int = 0):
    """wenet/transformer/search.py:125-247 with context_graph=None.  Returns, per utterance,
    dict(tokens, score, times, nbest, nbest_scores, nbest_times)."""
    results = []
    for i in range(ctc_probs.shape[0]):
        ctc_prob = ctc_probs[i]
        cur = [(tuple(), _PS(s=0.0, ns=-math.inf, v_s=0.0, v_ns=0.0))]
        for t in range(int(ctc_lens[i])):
            logp = ctc_prob[t]
            nxt = defaultdict(_PS)
            _, top_idx = logp.topk(beam_size)
            for u in top_idx.tolist():
                prob = logp[u].item()
                for prefix, ps in cur:
                    last = prefix[-1] if len(prefix) > 0 else None
                    if u == blank_id:
                        n = nxt[prefix]
                        n.s = _log_add(n.s, ps.score() + prob)
                        n.v_s = ps.viterbi_score() + prob
                        n.times_s = ps.times().copy()
                    elif u == last:
                        n1 = nxt[prefix]
                        n1.ns = _log_add(n1.ns, ps.ns + prob)
                        if n1.v_ns < ps.v_ns + prob:
                            n1.v_ns = ps.v_ns + prob
                            if n1.cur_token_prob < prob:
                                n1.cur_token_prob = prob
                                n1.times_ns = ps.times_ns.copy()
                                n1.times_ns[-1] = t
                        n2 = nxt[prefix + (u,)]
                        n2.ns = _log_add(n2.ns, ps.s + prob)
                        if n2.v_ns < ps.v_s + prob:
                            n2.v_ns = ps.v_s + prob
                            n2.cur_token_prob = prob
                            n2.times_ns = ps.times_s.copy()
                            n2.times_ns.append(t)
                    else:
                        n = nxt[prefix + (u,)]
                        n.ns = _log_add(n.ns, ps.score() + prob)
                        if n.v_ns < ps.viterbi_score() + prob:
                            n.v_ns = ps.viterbi_score() + prob
                            n.cur_token_prob = prob
                            n.times_ns = ps.times().copy()
                            n.times_ns.append(t)
            cur = sorted(nxt.items(), key=lambda x: x[1].score(), reverse=True)[:beam_size]
        results.append(dict(tokens=list(cur[0][0]), score=cur[0][1].score(), times=cur[0][1].times(),
                            nbest=[list(y[0]) for y in cur], nbest_scores=[y[1].score() for y in cur],
                            nbest_times=[y[1].times() for y in cur]))
    return results


# --------------------------------------------------------------------------- CER (section 8f row 4)
def calculate_cer(pre_tokens, gt_tokens):
    """rnnt_eval.py:11-56 restated: Levenshtein table, then a backtrace from (m, n) that prefers, in this order, a
    match, a substitution (diagonal + 1), a deletion (row above + 1) and otherwise an insertion; what is left of either
    sequence when a border is reached counts as deletions / insertions.  Returns (cer, S, D, I, N)."""
    m, n = len(pre_tokens), len(gt_tokens)
    dp = np.zeros((m + 1, n + 1), dtype=np.int64)
    dp[:, 0] = np.arange(m + 1)
    dp[0, :] = np.arange(n + 1)
    for i in range(1, m + 1):
        for j in range(1, n + 1):
            cost = 0 if pre_tokens[i - 1] == gt_tokens[j - 1] else 1
            dp[i, j] = min(dp[i - 1, j] + 1, dp[i, j - 1] + 1, dp[i - 1, j - 1] + cost)
    i, j, S, D, I = m, n, 0, 0, 0
    while i > 0 and j > 0:
        if pre_tokens[i - 1] == gt_tokens[j - 1]:
            i, j = i - 1, j - 1
        elif dp[i, j] == dp[i - 1, j - 1] + 1:
            S, i, j = S + 1, i - 1, j - 1
        elif dp[i, j] == dp[i - 1, j] + 1:
            D, i = D + 1, i - 1
        else:
            I, j = I + 1, j - 1
    D += i
    I += j
    return ((S + D + I) / n if n != 0 else 0.0), S, D, I, n
