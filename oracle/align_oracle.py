"""fp64 numpy restatement of forced alignment (the Viterbi path of a known transcript) for the RNN-T lattice and the CTC
trellis, with the tie rules of csrc/align.cu, and with the margin of every decision on the chosen path: the gap between
the winning candidate and the best other one.  Where every margin on the path exceeds the arithmetic error of an
implementation, its path must equal this one.  Self-contained: numpy only."""
import itertools
import math

import numpy as np

NEG_INF = -math.inf


def rnnt_viterbi(lpb, lpl, Tb, Ub):
    """lpb / lpl [>= Tb, >= Ub + 1] log-probs of one utterance.  delta(0,0) = 0,
    delta(t,u) = max(delta(t-1,u) + lpb(t-1,u), delta(t,u-1) + lpl(t,u-1)); on an exact tie the blank predecessor.
    Returns dict(score, frames [Ub] (frame of each label), token_lp [Ub], margin = smallest decision margin on the
    path (inf when no decision had two candidates)).  No frames or a -inf best path: score -inf, frames all -1."""
    lpb, lpl = np.asarray(lpb, dtype=np.float64), np.asarray(lpl, dtype=np.float64)
    if Tb <= 0:
        return dict(score=NEG_INF, frames=np.full(Ub, -1), token_lp=np.zeros(Ub), margin=math.inf)
    d = np.full((Tb, Ub + 1), NEG_INF)
    lab = np.zeros((Tb, Ub + 1), dtype=bool)
    gap = np.full((Tb, Ub + 1), math.inf)
    d[0, 0] = 0.0
    for t in range(Tb):
        for u in range(Ub + 1):
            if t == 0 and u == 0:
                continue
            xa = d[t - 1, u] + lpb[t - 1, u] if t > 0 else NEG_INF
            xb = d[t, u - 1] + lpl[t, u - 1] if u > 0 else NEG_INF
            lab[t, u] = xb > xa
            d[t, u] = max(xa, xb)
            if t > 0 and u > 0 and min(xa, xb) > NEG_INF:
                gap[t, u] = abs(xa - xb)
    score = d[Tb - 1, Ub] + lpb[Tb - 1, Ub]
    if not score > NEG_INF:
        return dict(score=NEG_INF, frames=np.full(Ub, -1), token_lp=np.zeros(Ub), margin=math.inf)
    frames, tok, margin = np.full(Ub, -1), np.zeros(Ub), math.inf
    t, u = Tb - 1, Ub
    while u > 0:
        margin = min(margin, gap[t, u])
        if t == 0 or lab[t, u]:
            u -= 1
            frames[u], tok[u] = t, lpl[t, u]
        else:
            t -= 1
    return dict(score=float(score), frames=frames, token_lp=tok, margin=margin)   # column 0 below: blanks only


def rnnt_path_score(lpb, lpl, frames, Tb, Ub):
    """Log-probability of the lattice path that emits label u at frames[u] (non-decreasing, in [0, Tb)): every label,
    and at each frame t the blank leaving (t, #labels emitted at frames <= t)."""
    frames = [int(f) for f in frames[:Ub]]
    s = sum(float(lpl[f, u]) for u, f in enumerate(frames))
    for t in range(Tb):
        s += float(lpb[t, sum(1 for f in frames if f <= t)])
    return s


def rnnt_brute_force(lpb, lpl, Tb, Ub):
    """(best score, best frames) over every monotone assignment of the Ub labels to frames: small lattices only."""
    best, arg = NEG_INF, None
    for fr in itertools.combinations_with_replacement(range(Tb), Ub):
        s = rnnt_path_score(lpb, lpl, fr, Tb, Ub)
        if s > best:
            best, arg = s, fr
    return best, arg


def ctc_extended(targets, Ub, blank):
    ext = [blank]
    for u in range(Ub):
        ext += [int(targets[u]), blank]
    return ext


def ctc_viterbi(lp, targets, Tb, Ub, blank):
    """lp [>= Tb, V] log-probs, targets [>= Ub] (labels in [0, V)).  State s-2 precedes s only when l'_s != blank and
    l'_s != l'_{s-2}; an exact tie takes the smaller jump, and between the end states S-1.  Returns dict(score,
    labels [Tb], frame_lp [Tb], spans [Ub, 2] (first frame, last frame + 1 of each token), margin = smallest decision
    margin on the path, end choice included).  No path: score -inf, labels / spans -1, frame_lp 0."""
    lp = np.asarray(lp, dtype=np.float64)
    ext = ctc_extended(targets, Ub, blank)
    S = len(ext)
    dead = dict(score=NEG_INF, labels=np.full(max(Tb, 0), -1), frame_lp=np.zeros(max(Tb, 0)),
                spans=np.full((Ub, 2), -1), margin=math.inf)
    if Tb <= 0:
        return dead
    d = np.full((Tb, S), NEG_INF)
    jump = np.zeros((Tb, S), dtype=np.int64)
    gap = np.full((Tb, S), math.inf)
    d[0, 0] = lp[0, ext[0]]
    if S > 1:
        d[0, 1] = lp[0, ext[1]]
    for t in range(1, Tb):
        for s in range(S):
            cands = [d[t - 1, s]]
            if s >= 1:
                cands.append(d[t - 1, s - 1])
            if s >= 2 and ext[s] != blank and ext[s] != ext[s - 2]:
                cands.append(d[t - 1, s - 2])
            j = int(np.argmax(cands))               # first maximum: the smaller jump on a tie
            jump[t, s] = j
            d[t, s] = cands[j] + lp[t, ext[s]]
            rest = [c for i, c in enumerate(cands) if i != j]
            if rest and max(rest) > NEG_INF:
                gap[t, s] = cands[j] - max(rest)
    a1, a2 = d[Tb - 1, S - 1], (d[Tb - 1, S - 2] if S > 1 else NEG_INF)
    end2 = a2 > a1
    score = a2 if end2 else a1
    if not score > NEG_INF:
        return dead
    margin = abs(a1 - a2) if S > 1 and min(a1, a2) > NEG_INF else math.inf
    s = S - 2 if end2 else S - 1
    labels, flp, spans = np.full(Tb, -1), np.zeros(Tb), np.full((Ub, 2), -1)
    for t in range(Tb - 1, -1, -1):
        labels[t], flp[t] = ext[s], lp[t, ext[s]]
        if s & 1:
            if spans[s >> 1, 1] < 0:
                spans[s >> 1, 1] = t + 1
            spans[s >> 1, 0] = t
        if t > 0:
            margin = min(margin, gap[t, s])
            s -= jump[t, s]
    return dict(score=float(score), labels=labels, frame_lp=flp, spans=spans, margin=margin)


def ctc_min_frames(targets, Ub):
    """Frames of the shortest CTC alignment: one per label and one blank between equal neighbours."""
    return Ub + sum(1 for u in range(1, Ub) if targets[u] == targets[u - 1])
