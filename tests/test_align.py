"""Forced alignment (csrc/align.cu): `rnnt_viterbi`, `rnnt_forced_align` through the fused joint, `ctc_forced_align`
and the module methods, held per utterance to the fp64 oracle of oracle/align_oracle.py and to torchaudio.

Two kinds of inputs run through every kernel form:
  * 'grid': log-probs on a 1/8 grid.  Every sum of them is exact in fp32 and fp64, so exact ties are frequent and the
    kernels must reproduce the oracle's path, tie rule included, and its score bit for bit;
  * 'cont': continuous log-probs.  Paths must match wherever every decision margin on the oracle's path exceeds the
    larger of 1e-4 and a bound on the fp32 rounding of the recursion (2 (T_b + U_b) 2^-24 |score|: each of the two
    candidates of a decision is a sum of at most T_b + U_b terms); scores within 1e-5 relative.  Elsewhere the path the
    kernel returns, re-scored in fp64, must score within 1e-5 of the oracle's best.

The CPU tests check the oracle (against torchaudio.functional.forced_align / merge_tokens and against brute-force path
enumeration), the checkers (planted faults are caught) and, through a mirror of the dispatch, that the GPU case tables
reach every kernel form."""
import math
import types

import numpy as np
import pytest
import torch

from oracle import align_oracle as AO
from oracle import transducer_oracle as TO

SCORE_TOL = 1e-5
MARGIN_FLOOR = 1e-4
BF16_COST, BF16_COST_STEP = 2e-3, 1e-3     # the fused loss's bf16 cost bar (functional.fused_joint_rnnt_loss)


# ------------------------------------------------------------------------------ mirror of the dispatch (csrc/align.cu)
# It restates rnnt_viterbi_shared and ctc_viterbi_shared and must change when they do.
def rnnt_form(T, U1):
    if U1 > 256:
        return "ws"
    nj = 1 if U1 <= 32 else 2 if U1 <= 64 else 4 if U1 <= 128 else 8
    pitch = (U1 + 1) & ~1
    return f"NJ={nj}" if 2 * T * pitch * 4 + (T + U1) * nj * 4 <= 227 * 1024 else "ws"


def ctc_form(T, umax):
    sp = (2 * umax + 1 + 31) // 32 * 32
    if sp > 1024:
        return "umax"
    nj = sp // 32
    return f"NJ={nj}" if nj <= 8 and (T * (2 * umax + 1) + sp + T * nj * 2) * 4 <= 220 * 1024 else "ws"


# ------------------------------------------------------------------------------------------------------- case tables
def _rcase(name, form, T, U1, tl, ul, seed):
    return dict(name=name, form=form, T=T, U1=U1, tl=list(tl), ul=list(ul), seed=seed)


RNNT_CASES = [
    _rcase("nj1", "NJ=1", 30, 20, (30, 17, 1, 30, 0), (19, 5, 19, 0, 3), 1),
    _rcase("nj2", "NJ=2", 40, 50, (40, 33, 12, 2), (49, 33, 48, 1), 2),
    _rcase("nj4", "NJ=4", 60, 100, (60, 41, 7), (99, 64, 63), 3),
    _rcase("nj8", "NJ=8", 50, 200, (50, 23, 50), (199, 128, 130), 4),
    _rcase("ws_smem", "ws", 1000, 32, (1000, 517, 3), (31, 17, 31), 5),       # beyond shared memory at NJ = 1
    _rcase("ws_u1", "ws", 20, 300, (20, 9, 20), (299, 260, 31), 6),           # U1 > 256
]


def _ccase(name, form, T, umax, tl, ul, seed, V=30, blank=0, kinds=None):
    return dict(name=name, form=form, T=T, umax=umax, tl=list(tl), ul=list(ul), seed=seed, V=V, blank=blank,
                kinds=kinds or "r" * len(tl))


CTC_CASES = [
    _ccase("nj1", "NJ=1", 40, 15, (40, "min", "min-1", 1, 0), (15, 15, 15, 0, 4), 11, kinds="rpprr"),
    _ccase("nj2", "NJ=2", 60, 20, (60, 45, "min"), (20, 31, 20), 12, V=33, blank=16, kinds="rpp"),
    _ccase("nj3_cfg5", "NJ=3", 200, 40, (200, 130, "min-1", "min"), (40, 25, 40, 40), 13, V=412, blank=5,
           kinds="rpps"),
    _ccase("nj4", "NJ=4", 150, 63, (150, 100), (63, 40), 14),
    _ccase("nj5", "NJ=5", 150, 79, (150, "min"), (79, 79), 15, kinds="rp"),
    _ccase("nj6", "NJ=6", 180, 95, (180, 120), (95, 50), 16, blank=29),
    _ccase("nj7", "NJ=7", 200, 111, (200, "min-1"), (111, 111), 17, kinds="rp"),
    _ccase("nj8", "NJ=8", 200, 127, (200, 140), (127, 127), 18),
    _ccase("ws_u", "ws", 300, 128, (300, "min", 120), (128, 128, 3), 19, kinds="rpr"),
    _ccase("ws_u511", "ws", 700, 511, (700, "min-1", 600), (511, 511, 17), 20, kinds="ppr"),
    _ccase("ws_t", "ws", 3000, 10, (3000, 1700, 2), (10, 4, 10), 21),         # beyond shared memory at NJ = 1
]

# out-of-range values: lengths negative, 0 and beyond the extents; labels >= V and < 0 (read as blank)
BAD_TL, BAD_UL = (-3, 0, 7, 100), (2, -5, 100, 3)


# ------------------------------------------------------------------------------------------------------------ inputs
def lattice_inputs(c, kind):
    """lp_blank / lp_label [B,T,U1] fp32 of case c: 'grid' values on a 1/8 grid, 'cont' continuous."""
    g = torch.Generator().manual_seed(3000 + c["seed"] + (kind == "grid") * 100)
    B = len(c["tl"])
    lpb = -torch.empty(B, c["T"], c["U1"]).exponential_(1.0, generator=g) * 2.0
    lpl = -torch.empty(B, c["T"], c["U1"]).exponential_(1.0, generator=g) * 2.0
    if kind == "grid":
        lpb, lpl = (lpb * 8).round() / 8, (lpl * 8).round() / 8
    return lpb.float(), lpl.float()


def ctc_inputs(c, kind):
    """log_probs [B,T,V] fp32 (log_softmax of random logits, on a 1/8 grid for 'grid'), targets [B,Umax] int64 (never
    blank; kinds: r random, p every fifth label repeats its predecessor, s one label throughout), lengths resolved."""
    g = torch.Generator().manual_seed(5000 + c["seed"] + (kind == "grid") * 100)
    B, T, V, umax, blank = len(c["tl"]), c["T"], c["V"], c["umax"], c["blank"]
    lp = torch.log_softmax(2.0 * torch.randn(B, T, V, generator=g, dtype=torch.float64), -1)
    if kind == "grid":
        lp = (lp * 8).round() / 8
    tgt = torch.randint(0, V - 1, (B, umax), generator=g)
    tgt += (tgt >= blank).long()
    tl = []
    for b, k in enumerate(c["kinds"]):
        U = min(max(c["ul"][b], 0), umax)
        if k == "p":
            for u in range(1, U, 5):
                tgt[b, u] = tgt[b, u - 1]
        elif k == "s":
            tgt[b, :] = tgt[b, 0]
        t = c["tl"][b]
        if isinstance(t, str):
            t = AO.ctc_min_frames(tgt[b].tolist(), U) - (t == "min-1")
        tl.append(t)
    return lp.float(), tgt, tl, list(c["ul"])


def clamp_len(v, hi):
    return [min(max(int(x), 0), hi) for x in v]


def margin_bar(score, n):
    return max(MARGIN_FLOOR, 2.0 * n * 2.0 ** -24 * abs(score)) if math.isfinite(score) else MARGIN_FLOOR


# ---------------------------------------------------------------------------------------------------------- checkers
def check_rnnt(got, lpb, lpl, tl, ul, score_tol=SCORE_TOL, exact=False, path_bar=None):
    """Per-utterance check of got = (frames [B,U], token_lp [B,U], scores [B]) against the oracle on fp64 copies of
    lpb / lpl; tl / ul are the clamped lengths.  exact: paths and scores equal bit for bit (grid inputs).  path_bar(b,
    oracle) overrides the margin above which frames must equal the oracle's.  Returns (failures, worst score error)."""
    frames, tok, scores = (np.asarray(x) for x in got)
    lpb, lpl = np.asarray(lpb, dtype=np.float64), np.asarray(lpl, dtype=np.float64)
    fails, worst = [], 0.0
    for b in range(len(tl)):
        Tb, Ub = tl[b], ul[b]
        o = AO.rnnt_viterbi(lpb[b], lpl[b], Tb, Ub)
        fr, s = frames[b], float(scores[b])
        if bool((fr[Ub:] != -1).any()) or bool((tok[b, Ub:] != 0).any()):
            fails.append(f"b={b}: entries beyond U_b = {Ub}")
        if o["score"] == -math.inf:
            if s != -math.inf or bool((fr != -1).any()):
                fails.append(f"b={b}: no path (T_b = {Tb}) but score {s}, frames {fr[:4].tolist()}...")
            continue
        f = fr[:Ub]
        if bool((f < 0).any()) or bool((f >= Tb).any()) or bool((np.diff(f) < 0).any()):
            fails.append(f"b={b}: frames not a monotone path in [0, {Tb}): {f.tolist()}")
            continue
        bar = path_bar(b, o) if path_bar else margin_bar(o["score"], Tb + Ub)
        if (exact or o["margin"] > bar) and not np.array_equal(f, o["frames"]):
            k = int(np.argmax(f != o["frames"]))
            fails.append(f"b={b}: label {k} at frame {f[k]}, oracle {o['frames'][k]} (margin {o['margin']:.2e})")
        if not np.allclose(tok[b, :Ub], lpl[b, f, np.arange(Ub)], rtol=0, atol=1e-6):
            fails.append(f"b={b}: token log-probs are not lp_label at the frames")
        e = abs(s - o["score"]) / max(1.0, abs(o["score"]))
        er = abs(AO.rnnt_path_score(lpb[b], lpl[b], f, Tb, Ub) - o["score"]) / max(1.0, abs(o["score"]))
        worst = max(worst, e, er)
        if (exact and s != o["score"]) or e > score_tol or er > score_tol:
            fails.append(f"b={b}: score {s} / re-scored path {er:.2e} against {o['score']} (rel {e:.2e})")
    return fails, worst


def check_ctc(got, lp, tgt, tl, ul, blank, exact=False):
    """Per-utterance check of got = (labels [B,T], frame_lp [B,T], scores [B], spans [B,Umax,2]) against the oracle;
    tgt / tl / ul clamped.  Returns (failures, worst score error)."""
    labels, flp, scores, spans = (np.asarray(x) for x in got)
    lp = np.asarray(lp, dtype=np.float64)
    fails, worst = [], 0.0
    for b in range(len(tl)):
        Tb, Ub = tl[b], ul[b]
        tg = [int(x) for x in tgt[b, :Ub]]
        o = AO.ctc_viterbi(lp[b], tg, Tb, Ub, blank)
        s = float(scores[b])
        if bool((labels[b, Tb:] != -1).any()) or bool((flp[b, Tb:] != 0).any()) or bool((spans[b, Ub:] != -1).any()):
            fails.append(f"b={b}: entries beyond T_b = {Tb} / U_b = {Ub}")
        if o["score"] == -math.inf:
            if s != -math.inf or bool((labels[b] != -1).any()) or bool((spans[b] != -1).any()) or bool((flp[b] != 0).any()):
                fails.append(f"b={b}: no path but score {s} / labels / spans set")
            continue
        lab, sp = labels[b, :Tb], spans[b, :Ub]
        # the path: labels are the target's tokens on their spans, blank elsewhere, spans ordered and disjoint
        want = np.full(Tb, blank)
        ok = bool((sp[:, 0] < sp[:, 1]).all()) and bool((sp[1:, 0] >= sp[:-1, 1]).all()) if Ub else True
        ok = ok and (Ub == 0 or (sp[0, 0] >= 0 and sp[-1, 1] <= Tb))
        if ok:
            for u in range(Ub):
                want[sp[u, 0]:sp[u, 1]] = tg[u]
            ok = bool((lab == want).all()) and all(sp[u, 1] < sp[u + 1, 0] for u in range(Ub - 1) if tg[u] == tg[u + 1])
        if not ok:
            fails.append(f"b={b}: labels / spans are not a CTC path of the target")
            continue
        bar = margin_bar(o["score"], Tb)
        if (exact or o["margin"] > bar) and not (np.array_equal(lab, o["labels"]) and np.array_equal(sp, o["spans"])):
            t = int(np.argmax(lab != o["labels"]))
            fails.append(f"b={b}: frame {t} label {lab[t]}, oracle {o['labels'][t]} (margin {o['margin']:.2e})")
        if not np.allclose(flp[b, :Tb], lp[b, np.arange(Tb), lab], rtol=0, atol=1e-6):
            fails.append(f"b={b}: frame log-probs are not those of the labels")
        e = abs(s - o["score"]) / max(1.0, abs(o["score"]))
        er = abs(float(lp[b, np.arange(Tb), lab].sum()) - o["score"]) / max(1.0, abs(o["score"]))
        worst = max(worst, e, er)
        if (exact and s != o["score"]) or e > SCORE_TOL or er > SCORE_TOL:
            fails.append(f"b={b}: score {s} / re-scored path {er:.2e} against {o['score']} (rel {e:.2e})")
    return fails, worst


# --------------------------------------------------------------------------------------------------------------- CPU
def test_oracle_ctc_matches_torchaudio():
    """On tie-free random inputs, one utterance at a time: labels equal torchaudio's forced_align, scores within
    1e-9, spans equal merge_tokens; repeated labels included."""
    taf = pytest.importorskip("torchaudio.functional")
    c = _ccase("ta", "NJ=2", 50, 12, (50, 40, "min", 29), (12, 9, 12, 1), 31, V=20, blank=3, kinds="rppr")
    lp, tgt, tl, ul = ctc_inputs(c, "cont")
    lp = lp.double()
    for b in range(len(tl)):
        Tb, Ub = tl[b], ul[b]
        o = AO.ctc_viterbi(lp[b].numpy(), tgt[b].tolist(), Tb, Ub, c["blank"])
        al, sc = taf.forced_align(lp[b:b + 1, :Tb], tgt[b:b + 1, :Ub].int(), blank=c["blank"])
        assert np.array_equal(al[0].numpy(), o["labels"]), b
        assert abs(float(sc[0].sum()) - o["score"]) <= 1e-9 * abs(o["score"]), b
        spans = [(s.token, s.start, s.end) for s in taf.merge_tokens(al[0], sc[0].exp(), blank=c["blank"])]
        assert spans == [(tgt[b, u].item(), int(o["spans"][u, 0]), int(o["spans"][u, 1])) for u in range(Ub)], b


def test_oracle_rnnt_matches_brute_force():
    """Small lattices (T <= 5, U <= 3), continuous and on the grid (ties: the oracle's path is the one emitting each
    label at its earliest frame among the best paths, which the lexicographic order of the enumeration finds first)."""
    g = torch.Generator().manual_seed(7)
    n = 0
    for Tb in range(1, 6):
        for Ub in range(0, 4):
            for grid in (False, True):
                lpb = -torch.empty(Tb, Ub + 1).exponential_(1.0, generator=g).double() * 2
                lpl = -torch.empty(Tb, Ub + 1).exponential_(1.0, generator=g).double() * 2
                if grid:
                    lpb, lpl = (lpb * 2).round() / 2, (lpl * 2).round() / 2
                o = AO.rnnt_viterbi(lpb.numpy(), lpl.numpy(), Tb, Ub)
                best, arg = AO.rnnt_brute_force(lpb.numpy(), lpl.numpy(), Tb, Ub)
                assert abs(o["score"] - best) <= 1e-12 * max(1, abs(best))
                assert abs(AO.rnnt_path_score(lpb.numpy(), lpl.numpy(), o["frames"], Tb, Ub) - best) <= 1e-12 * max(1, abs(best))
                if grid:
                    assert tuple(o["frames"]) == tuple(arg), (Tb, Ub)
                n += 1
    assert n == 40


def test_oracle_rnnt_score_below_log_likelihood():
    """Every Viterbi score is <= the log-likelihood (-cost) of the restated loss on the same log-probs."""
    g = torch.Generator().manual_seed(8)
    B, T, U1, V, blank = 4, 9, 5, 7, 0
    logits = torch.randn(B, T, U1, V, generator=g, dtype=torch.float64)
    tgt = torch.randint(1, V, (B, U1 - 1), generator=g, dtype=torch.int32)
    tl, ul = torch.tensor([9, 6, 1, 9]), torch.tensor([4, 2, 4, 0])
    r = TO.rnnt_lattice_restated(logits, tgt, tl, ul, blank)
    for b in range(B):
        o = AO.rnnt_viterbi(r["lp_blank"][b].numpy(), r["lp_label"][b].numpy(), int(tl[b]), int(ul[b]))
        assert o["score"] <= -float(r["costs"][b]) + 1e-12


def test_checkers_reject_planted_faults():
    """The checkers accept the oracle's own answers and reject a label shifted by a frame, two spans swapped and a
    score off by 1e-4 relative."""
    c = RNNT_CASES[0]
    lpb, lpl = lattice_inputs(c, "grid")
    tl, ul = clamp_len(c["tl"], c["T"]), clamp_len(c["ul"], c["U1"] - 1)
    B, U = len(tl), c["U1"] - 1
    fr, tk, sc = np.full((B, U), -1), np.zeros((B, U), np.float32), np.zeros(B, np.float32)
    for b in range(B):
        o = AO.rnnt_viterbi(lpb[b].double().numpy(), lpl[b].double().numpy(), tl[b], ul[b])
        fr[b, :ul[b]], tk[b, :ul[b]], sc[b] = o["frames"], o["token_lp"], o["score"]
    assert check_rnnt((fr, tk, sc), lpb, lpl, tl, ul, exact=True)[0] == []
    f2 = fr.copy()
    k = next(u for u in range(ul[0]) if f2[0, u] < (f2[0, u + 1] if u + 1 < ul[0] else tl[0] - 1))
    f2[0, k] += 1
    assert any(f.startswith("b=0:") for f in check_rnnt((f2, tk, sc), lpb, lpl, tl, ul, exact=True)[0])
    s2 = sc.copy()
    s2[1] *= 1 + 1e-4
    assert any(f.startswith("b=1: score") for f in check_rnnt((fr, tk, s2), lpb, lpl, tl, ul)[0])

    cc = CTC_CASES[0]
    lp, tgt, ctl, cul = ctc_inputs(cc, "grid")
    ctl, cul = clamp_len(ctl, cc["T"]), clamp_len(cul, cc["umax"])
    B, T = len(ctl), cc["T"]
    lab, flp, csc, sp = np.full((B, T), -1), np.zeros((B, T), np.float32), np.zeros(B, np.float32), np.full((B, cc["umax"], 2), -1)
    for b in range(B):
        o = AO.ctc_viterbi(lp[b].double().numpy(), tgt[b].tolist(), ctl[b], cul[b], cc["blank"])
        csc[b] = o["score"]
        if o["score"] > -math.inf:
            lab[b, :ctl[b]], flp[b, :ctl[b]], sp[b, :cul[b]] = o["labels"], o["frame_lp"], o["spans"]
    assert check_ctc((lab, flp, csc, sp), lp, tgt, ctl, cul, cc["blank"], exact=True)[0] == []
    sp2 = sp.copy()
    sp2[0, [2, 3]] = sp2[0, [3, 2]]
    assert any(f.startswith("b=0:") for f in check_ctc((lab, flp, csc, sp2), lp, tgt, ctl, cul, cc["blank"])[0])
    c2 = csc.copy()
    c2[0] *= 1 + 1e-4
    assert any(f.startswith("b=0: score") for f in check_ctc((lab, flp, c2, sp), lp, tgt, ctl, cul, cc["blank"])[0])


def test_case_tables_reach_every_form():
    """Through the mirror of the dispatch: every case reaches the form it names; together they reach NJ = 1/2/4/8 and
    both workspace triggers for RNN-T, NJ = 1..8 and both workspace triggers (Sp > 256, shared memory) for CTC, and
    Umax = 511; the batches hold zero, negative-free ragged lengths, infeasible rows and repeats."""
    assert rnnt_form(1000, 32) == "ws" and rnnt_form(800, 32) == "NJ=1" and rnnt_form(20, 257) == "ws"
    assert {c["form"] for c in RNNT_CASES} == {"NJ=1", "NJ=2", "NJ=4", "NJ=8", "ws"}
    for c in RNNT_CASES:
        assert rnnt_form(c["T"], c["U1"]) == c["form"], c["name"]
    assert any(c["U1"] > 256 for c in RNNT_CASES) and any(c["U1"] <= 256 and c["form"] == "ws" for c in RNNT_CASES)
    assert ctc_form(100, 512) == "umax" and ctc_form(3000, 10) == "ws"
    assert {c["form"] for c in CTC_CASES} == {f"NJ={n}" for n in range(1, 9)} | {"ws"}
    seen = set()
    for c in CTC_CASES:
        assert ctc_form(c["T"], c["umax"]) == c["form"], c["name"]
        lp, tgt, tl, ul = ctc_inputs(c, "cont")
        for b in range(len(tl)):
            m = AO.ctc_min_frames(tgt[b].tolist(), min(ul[b], c["umax"]))
            seen |= {k for k, ok in (("infeasible", 0 < tl[b] < m), ("T_b=0", tl[b] == 0), ("min", tl[b] == m > 0),
                                     ("repeat", m > min(ul[b], c["umax"]))) if ok}
    assert seen == {"infeasible", "T_b=0", "min", "repeat"}
    assert max(c["umax"] for c in CTC_CASES) == 511
    assert any(c["form"] == "ws" and c["umax"] <= 127 for c in CTC_CASES)


# --------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def C():
    import ctcvr_b200
    assert torch.cuda.is_available()
    ctcvr_b200._lib.lib()
    return ctcvr_b200


def _i32(v):
    return torch.as_tensor(v, dtype=torch.int32).cuda()


def _cpu(xs):
    return tuple(x.cpu() for x in xs)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["grid", "cont"])
@pytest.mark.parametrize("c", RNNT_CASES, ids=[c["name"] for c in RNNT_CASES])
def test_rnnt_viterbi_vs_fp64(C, c, kind):
    lpb, lpl = lattice_inputs(c, kind)
    got = _cpu(C.rnnt_viterbi(lpb.cuda(), lpl.cuda(), _i32(c["tl"]), _i32(c["ul"])))
    fails, worst = check_rnnt(got, lpb, lpl, clamp_len(c["tl"], c["T"]), clamp_len(c["ul"], c["U1"] - 1),
                              exact=kind == "grid")
    print(f"rnnt_viterbi {c['name']} [{c['form']}] {kind}: worst score rel {worst:.2e}")
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["grid", "cont"])
@pytest.mark.parametrize("c", CTC_CASES, ids=[c["name"] for c in CTC_CASES])
def test_ctc_viterbi_vs_fp64(C, c, kind):
    lp, tgt, tl, ul = ctc_inputs(c, kind)
    got = _cpu(C.ctc_forced_align(lp.cuda(), tgt.cuda(), _i32(tl), _i32(ul), c["blank"]))
    fails, worst = check_ctc(got, lp, tgt, clamp_len(tl, c["T"]), clamp_len(ul, c["umax"]), c["blank"],
                             exact=kind == "grid")
    print(f"ctc_viterbi {c['name']} [{c['form']}] {kind}: worst score rel {worst:.2e}")
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("c", [c for c in CTC_CASES if c["name"] in ("nj1", "nj3_cfg5", "ws_u", "ws_u511")],
                         ids=lambda c: c["name"])
def test_ctc_forced_align_vs_torchaudio(C, c):
    """Per utterance of a padded batch against torchaudio.functional.forced_align on CPU and CUDA (fp32, one utterance
    per call): labels equal where the oracle's margins clear the bar (else the two paths score alike), frame
    log-probs within 1e-5, spans equal merge_tokens; infeasible rows are -inf / -1 next to feasible ones."""
    taf = pytest.importorskip("torchaudio.functional")
    lp, tgt, tl, ul = ctc_inputs(c, "cont")
    labels, flp, scores, spans = _cpu(C.ctc_forced_align(lp.cuda(), tgt.cuda(), _i32(tl), _i32(ul), c["blank"]))
    n_dead = 0
    for b in range(len(tl)):
        Tb, Ub = tl[b], ul[b]
        o = AO.ctc_viterbi(lp[b].double().numpy(), tgt[b].tolist(), Tb, Ub, c["blank"])
        if o["score"] == -math.inf:
            n_dead += 1
            assert float(scores[b]) == -math.inf and bool((labels[b] == -1).all()) and bool((spans[b] == -1).all())
            continue
        if Ub == 0:                                  # torchaudio takes no empty target; the oracle tests cover it
            continue
        for dev in ("cpu", "cuda"):
            al, sc = taf.forced_align(lp[b:b + 1, :Tb].to(dev), tgt[b:b + 1, :Ub].int().to(dev), blank=c["blank"])
            al, sc = al[0].cpu(), sc[0].cpu()
            if o["margin"] > margin_bar(o["score"], Tb):
                assert torch.equal(labels[b, :Tb], al.int()), (b, dev)
                assert torch.allclose(flp[b, :Tb], sc.float(), rtol=0, atol=1e-5), (b, dev)
                ts = [(s.start, s.end) for s in taf.merge_tokens(al, sc.exp(), blank=c["blank"])]
                assert ts == [tuple(x) for x in spans[b, :Ub].tolist()], (b, dev)
            else:
                assert abs(float(flp[b, :Tb].double().sum()) - float(sc.double().sum())) <= 1e-5 * abs(o["score"])
    assert n_dead == sum(1 for t in c["tl"] if t in ("min-1", 0))


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["NJ=1", "ws"])
def test_bad_values_act_as_clamped(C, form):
    """Lengths beyond the extents, zero and negative, and labels >= V or < 0 give exactly what the clamped inputs give
    (labels read as blank), in both kernel forms of both ops; no fault."""
    T, U1, umax, V, blank = (12, 6, 5, 9, 2) if form == "NJ=1" else (12, 300, 200, 9, 2)
    assert rnnt_form(T, U1) == form and ctc_form(T, umax) == form
    c = _rcase("bad", form, T, U1, (0,) * 4, (0,) * 4, 40)
    lpb, lpl = lattice_inputs(c, "cont")
    tl_ok, ul_ok = clamp_len(BAD_TL, T), clamp_len(BAD_UL, U1 - 1)
    bad = _cpu(C.rnnt_viterbi(lpb.cuda(), lpl.cuda(), _i32(BAD_TL), _i32(BAD_UL)))
    ok = _cpu(C.rnnt_viterbi(lpb.cuda(), lpl.cuda(), _i32(tl_ok), _i32(ul_ok)))
    assert all(torch.equal(x, y) for x, y in zip(bad, ok))
    assert not check_rnnt(bad, lpb, lpl, tl_ok, ul_ok)[0]

    g = torch.Generator().manual_seed(41)
    lp = torch.log_softmax(torch.randn(4, T, V, generator=g), -1)
    tgt = torch.randint(0, V, (4, umax), generator=g)
    tgt[2, 0], tgt[3, 1], tgt[3, 2] = V, -4, 10 ** 6
    tgt_ok = torch.where((tgt >= 0) & (tgt < V), tgt, torch.full_like(tgt, blank))
    ctl, cul = clamp_len(BAD_TL, T), clamp_len(BAD_UL, umax)
    bad = _cpu(C.ctc_forced_align(lp.cuda(), tgt.cuda(), _i32(BAD_TL), _i32(BAD_UL), blank))
    ok = _cpu(C.ctc_forced_align(lp.cuda(), tgt_ok.cuda(), _i32(ctl), _i32(cul), blank))
    assert all(torch.equal(x, y) for x, y in zip(bad, ok))
    assert float(bad[2][0]) == -math.inf and float(bad[2][1]) == -math.inf     # T_b = 0 (negative), T_b = 0


# ---------------------------------------------------------------------------------------- through the fused joint
def joint_case(seed=60, B=4, T=30, U1=9, D=128, V=40, blank=3):
    g = torch.Generator().manual_seed(seed)
    enc = 0.5 * torch.randn(B, T, D, generator=g)
    pred = 0.5 * torch.randn(B, U1, D, generator=g)
    w = torch.randn(V, D, generator=g) / math.sqrt(D)
    b = 0.1 * torch.randn(V, generator=g)
    tgt = torch.randint(0, V, (B, U1 - 1), generator=g, dtype=torch.int32)
    tl, ul = [T, 21, 9, 1], [U1 - 1, 5, 8, 0]
    return enc, pred, w, b, tgt, tl, ul, blank


COMBOS = [(p, a, False) for p in ("fp32", "bf16x3", "bf16") for a in ("tanh", "relu", "gelu")] + \
         [("bf16", a, True) for a in ("tanh", "relu")]


@pytest.mark.gpu
@pytest.mark.parametrize("precision,act,bf16_inputs", COMBOS,
                         ids=[f"{p}-{a}" + ("-bf16in" if i else "") for p, a, i in COMBOS])
def test_rnnt_forced_align_through_fused_joint(C, precision, act, bf16_inputs):
    """The path, re-scored in fp64 on the oracle's log-probs (fp64 joint of the same inputs), within tolerance of the
    oracle's best: 1e-4 relative for fp32 / bf16x3, the loss's bf16 cost bar for bf16; with fp32 / bf16x3 the frames
    equal the oracle's where every margin exceeds that tolerance; frames monotone; score <= -cost of the fused loss
    (up to the fp32 rounding of the two, 1e-6 relative)."""
    from test_joint_activations import joint_forward_act
    enc, pred, w, b, tgt, tl, ul, blank = joint_case()
    if bf16_inputs:
        enc, pred = enc.bfloat16(), pred.bfloat16()
    e, p = enc.cuda(), pred.cuda()
    frames, tok, scores = _cpu(C.rnnt_forced_align(e, p, w.cuda(), b.cuda(), tgt.cuda(), _i32(tl), _i32(ul), blank,
                                                   precision=precision, activation=act))
    costs = C.fused_joint_rnnt_loss(e, p, w.cuda(), b.cuda(), tgt.cuda(), _i32(tl), _i32(ul), blank, reduction="none",
                                    precision=precision, activation=act).cpu()
    D = enc.shape[-1]
    ws = {"enc_ffn.weight": torch.eye(D), "enc_ffn.bias": torch.zeros(D), "ffn_out.weight": w, "ffn_out.bias": b,
          "pred_ffn.weight": torch.eye(D), "pred_ffn.bias": torch.zeros(D)}
    logits = joint_forward_act(enc.double(), pred.double(), {k: v.double() for k, v in ws.items()}, True, act)
    r = TO.rnnt_lattice_restated(logits, tgt, torch.tensor(tl), torch.tensor(ul), blank)
    lpb, lpl = r["lp_blank"].numpy(), r["lp_label"].numpy()
    fails = []
    for i in range(len(tl)):
        Tb, Ub = tl[i], ul[i]
        o = AO.rnnt_viterbi(lpb[i], lpl[i], Tb, Ub)
        tol = 1e-4 * abs(o["score"]) if precision != "bf16" else max(BF16_COST * abs(o["score"]), BF16_COST_STEP * (Tb + Ub))
        f = frames[i, :Ub].numpy()
        if bool((np.diff(f) < 0).any()) or bool((f < 0).any()) or bool((f >= Tb).any()):
            fails.append(f"b={i}: frames {f.tolist()} not monotone in [0, {Tb})")
            continue
        if abs(AO.rnnt_path_score(lpb[i], lpl[i], f, Tb, Ub) - o["score"]) > tol or abs(float(scores[i]) - o["score"]) > tol:
            fails.append(f"b={i}: score {float(scores[i])} / re-scored path against {o['score']} (tol {tol:.1e})")
        if precision != "bf16" and o["margin"] > tol and not np.array_equal(f, o["frames"]):
            fails.append(f"b={i}: frames {f.tolist()} against {o['frames'].tolist()} (margin {o['margin']:.2e})")
        if not float(scores[i]) <= -float(costs[i]) + 1e-6 * abs(float(costs[i])):
            fails.append(f"b={i}: score {float(scores[i])} above -cost {-float(costs[i])}")
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
def test_rnnt_forced_align_loud_errors(C):
    enc, pred, w, b, tgt, tl, ul, blank = joint_case(D=100)
    args = (enc.cuda(), pred.cuda(), w.cuda(), b.cuda(), tgt.cuda(), _i32(tl), _i32(ul), blank)
    with pytest.raises(RuntimeError, match="rnnt_forced_align: precision='bf16' needs D % 128 == 0"):
        C.rnnt_forced_align(*args, precision="bf16")
    with pytest.raises(RuntimeError, match="targets must be"):
        C.rnnt_forced_align(*args[:4], tgt[:, :-1].cuda(), *args[5:])
    C.rnnt_forced_align(*args)                       # fp32 takes the shape


# ------------------------------------------------------------------------------------------------------ module level
@pytest.mark.gpu
@pytest.mark.parametrize("act", ["tanh", "relu", "gelu"])
@pytest.mark.parametrize("post", [False, True])
def test_transducer_joint_forced_align(C, act, post):
    """TransducerJoint.forced_align equals the functional op on the pre-projected (and post-join folded) inputs."""
    from ctcvr_b200.joint import fused_joint_inputs
    torch.manual_seed(61)
    D, V, blank = 128, 33, 0
    joint = C.TransducerJoint(V, 96, 80, D, postjoin_linear=post, activation=act).cuda()
    _, _, _, _, tgt, tl, ul, _ = joint_case()
    enc, pred = torch.randn(4, 30, 96).cuda(), torch.randn(4, 9, 80).cuda()
    tgt = (tgt % (V - 1) + 1).cuda()
    for precision in ("fp32", "bf16"):
        got = joint.forced_align(enc, pred, tgt, _i32(tl), _i32(ul), blank, precision=precision)
        if precision == "fp32":
            with torch.no_grad():
                e, p = fused_joint_inputs(joint, enc, pred)
            want = C.rnnt_forced_align(e, p, joint.ffn_out.weight, joint.ffn_out.bias, tgt, _i32(tl), _i32(ul), blank,
                                       activation=act)
            assert all(torch.equal(x, y) for x, y in zip(got, want))
        assert bool((got[0][0] >= 0).all()) and float(got[2][0]) < 0


@pytest.mark.gpu
def test_compute_rnnt_alignment_reference_shaped(C):
    """compute_rnnt_alignment on a reference-shaped model (the attributes the reference's Transducer has, no
    `precision`): the prologue, predictor and joint of compute_rnnt_loss, then the alignment of the joint's inputs."""
    from ctcvr_b200.transducer import compute_rnnt_alignment, rnnt_prologue
    torch.manual_seed(62)
    V, D, blank = 29, 128, 0
    pr = C.RNNPredictor(V, D, D, 0.0, D, 1, dropout=0.0).cuda().eval()
    joint = C.TransducerJoint(V, D, D, D).cuda()
    model = types.SimpleNamespace(predictor=pr, joint=joint, blank=blank, ignore_id=-1)
    enc = torch.randn(3, 40, D).cuda()
    enc_lens = torch.tensor([40, 31, 12]).cuda()
    text = torch.randint(1, V, (3, 7)).cuda()
    text[1, 5:] = 0                                  # padding beyond text_lens: any valid token id
    text_lens = torch.tensor([7, 5, 7]).cuda()
    frames, tok, scores = compute_rnnt_alignment(model, enc, enc_lens, text, text_lens)
    ys_in, tg, tl, ul = rnnt_prologue(text, text_lens, enc_lens, blank, -1)
    with torch.no_grad():
        want = joint.forced_align(enc, pr(ys_in), tg, tl, ul, blank)
    assert all(torch.equal(x, y) for x, y in zip((frames, tok, scores), want))
    assert frames.shape == (3, 7) and bool((frames[1, 5:] == -1).all()) and bool((frames[1, :5] >= 0).all())
    with torch.no_grad():
        loss = C.transducer.compute_rnnt_loss(model, enc, enc_lens, text, text_lens)
    assert float(scores.mean()) <= -float(loss)


@pytest.mark.gpu
@pytest.mark.parametrize("cls", ["CTC", "OnlineCTC"])
def test_ctc_module_forced_align(C, cls):
    torch.manual_seed(63)
    V, H, blank = 40, 64, 0
    head = getattr(C, cls)(V, H, dropout_rate=0.5, **({"blank_id": blank})).cuda()
    hs = torch.randn(3, 50, H).cuda()
    hl, ys, yl = _i32([50, 41, 3]), torch.randint(1, V, (3, 9)).cuda(), _i32([9, 6, 9])
    got = head.forced_align(hs, hl, ys, yl)
    want = C.ctc_forced_align(head.log_softmax(hs), ys, hl, yl, blank)
    assert all(torch.equal(x, y) for x, y in zip(got, want))
    assert float(got[2][2]) == -math.inf and float(got[2][0]) > -math.inf


@pytest.mark.gpu
def test_cuda_graph_replay(C):
    """A graph captured around rnnt_forced_align and ctc_forced_align replays to the eager result (new inputs copied
    into the captured buffers)."""
    enc, pred, w, b, tgt, tl, ul, blank = joint_case()
    e, p, wc, bc, tg, tlc, ulc = enc.cuda(), pred.cuda(), w.cuda(), b.cuda(), tgt.cuda(), _i32(tl), _i32(ul)
    c = CTC_CASES[2]
    lp, ctg, ctl, cul = ctc_inputs(c, "cont")
    lpc, ctgc, ctlc, culc = lp.cuda(), ctg.cuda(), _i32(ctl), _i32(cul)
    run = lambda: (C.rnnt_forced_align(e, p, wc, bc, tg, tlc, ulc, blank, precision="bf16x3"),
                   C.ctc_forced_align(lpc, ctgc, ctlc, culc, c["blank"]))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        run()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = run()
    e.copy_(e.flip(1))
    lpc.copy_(lpc.flip(1))
    graph.replay()
    torch.cuda.synchronize()
    want = run()
    for x, y in zip(out[0] + out[1], want[0] + want[1]):
        assert torch.equal(x, y)
