"""The CTC loss (`functional.ctc_loss_from_logits`, reduction='none') held to ATen's CPU ctc_loss in fp64 per utterance, in
every kernel form `ctc_loss` (csrc/ctc.cu) dispatches to and at the edges of each:

  * the shuffle form `ctc_alpha_beta_kernel<NJ>`, NJ = 1..8 (Sp = 32 NJ states), each at the smallest and the largest
    S = 2 U + 1 it takes; the barrier form (NJ = 0) at U = 128 and 255; the single-kernel fallback by Sp (U = 256, 511)
    and by shared memory (T one past the largest the split form accepts, at U = 40, 128 and 255);
  * vocabularies of 1, 2, 33 and 4097 entries, blank first, last and in the middle;
  * inside the batches: empty and full targets, a few labels in a wide form, one frame, all frames, one frame short
    of the shortest alignment (infeasible: zero_infinity) and exactly the shortest one, repeated labels, one label
    throughout, targets equal to blank, and -inf logits in a label's and in another column;
  * a cotangent that differs per utterance in sign and size (0, negative, 0.1 .. 3);
  * out-of-range lengths and labels, which the op clamps, in the split form and the fallback.

Every utterance's cost, its gradient and, on its own, its blank column are compared with the reference, so one bad
utterance cannot hide in a batch norm.  The CPU tests check the checker (planted faults are caught) and, through a
mirror of the dispatch, that the case table reaches the form each case names."""
import numpy as np
import pytest
import torch

COST_TOL = 1e-4            # each cost within 1e-4 x max(1, |cost|) of the fp64 reference
GRAD_TOL = 1e-4            # gradients: rel-L2 within max(1e-4, 3 x the error of ATen's own fp32 arithmetic)
REF_NEG = -1.0e4           # a -inf logit, as the references see it (see reference())
V0, BLANK0 = 412, 5        # BASELINE.json cfg5
GCS = (1.7, -0.6, 0.1, 3.0, 0.0)


# ---------------------------------------------------------------------- mirror of ctc_loss's dispatch (csrc/ctc.cu)
# It restates Sp, smemA, the 2 Sp <= 1024 condition, the Sp / 32 switch and the shared-memory limits of ctc_grad_kernel
# (smemB) and ctc_loss_kernel, for a call that asks for the gradient.  It must change when the C++ dispatch does.
def sp_of(umax):
    return (2 * umax + 1 + 31) // 32 * 32


def ctc_form(T, V, umax):
    """'NJ=1'..'NJ=8' (shuffle form), 'NJ=0' (barrier form), 'fallback', or the loud errors 'umax' and 'vocab'."""
    Sp = sp_of(umax)
    if Sp > 1024:
        return "umax"
    smem_a = (T * (2 * umax + 1) + 4 * (Sp + 4)) * 4 + (V + 2 * Sp) * 4
    if smem_a <= 220 * 1024 and 2 * Sp <= 1024:
        if (7 * Sp + 4 * V) * 4 > 200 * 1024:
            return "vocab"
        nj = Sp // 32
        return f"NJ={nj if nj <= 8 else 0}"
    if (3 * Sp + 32) * 4 + (V + Sp) * 4 > 200 * 1024:
        return "vocab"
    return "fallback"


def max_split_T(V, umax):
    T = 1
    while ctc_form(T + 1, V, umax) != "fallback":
        T += 1
    return T


# -------------------------------------------------------------------------------------------------------- case table
def _case(name, form, T, umax, tl, ul, kinds, gc, V=V0, blank=BLANK0, neg_inf=(), seed=0, cost_tol=COST_TOL):
    """tl entries are frame counts or 'min' / 'min-1': the shortest alignment of the utterance's target and one frame
    less.  kinds, one letter per utterance: r random labels (never blank), p every eighth label repeats its
    predecessor, s one label throughout, b blank at the first, middle and last target positions.  neg_inf: (b, t,
    'label' | 'other'), a -inf logit at frame t in the column of the utterance's first label other than blank, or
    of a label it does not use."""
    assert len(tl) == len(ul) == len(kinds) == len(gc)
    return dict(name=name, form=form, B=len(tl), T=T, umax=umax, tl=tuple(tl), ul=tuple(ul), kinds=kinds, gc=tuple(gc),
                V=V, blank=blank, neg_inf=tuple(neg_inf), seed=seed, cost_tol=cost_tol)


def _rot(k, n=5):
    return tuple(GCS[(i + k) % 5] for i in range(n))


def _nj_case(nj, edge):
    """The shuffle form at its low (U = 16 (NJ - 1), S = Sp - 31) or high (U = 16 NJ - 1, S = Sp - 1) edge."""
    umax = 16 * (nj - 1) if edge == "lo" else 16 * nj - 1
    T = max(umax + 40, 48)
    small = 2 if nj % 2 else umax // 2          # a few labels in a wide form, or one label over half the width
    return _case(f"nj{nj}_{edge}_u{umax}", f"NJ={nj}", T, umax,
                 tl=(T, 1, "min", "min-1", T - 3), ul=(umax, 0 if edge == "lo" else 1, umax, umax, small),
                 kinds="brpp" + ("r" if nj % 2 else "s"), gc=_rot(nj + (edge == "hi")),
                 neg_inf=((0, 1, "label"), (0, 2, "other")), seed=nj * 2 + (edge == "hi"))


CASES = [
    _case("nj1_lo_u0", "NJ=1", 40, 0, tl=(40, 1, 17), ul=(0, 0, 0), kinds="rrr", gc=(1.7, -0.6, 0.0),
          neg_inf=((0, 3, "other"),), seed=1),
    _case("nj1_hi_u15", "NJ=1", 55, 15, tl=(55, 1, "min", "min-1", 52), ul=(15, 1, 15, 15, 7), kinds="brpps",
          gc=_rot(1), neg_inf=((0, 1, "label"), (0, 2, "other")), seed=2),
] + [_nj_case(nj, edge) for nj in range(2, 9) for edge in ("lo", "hi")] + [
    # BASELINE.json cfg5 at B = 3, held to the 1e-5 cost bar it has always met
    _case("cfg5", "NJ=3", 500, 40, tl=(500, 311, 97), ul=(40, 17, 40), kinds="prb", gc=(1.7, -0.6, 0.25), seed=3,
          cost_tol=1e-5),
    # split / fallback T boundary at U = 40 (Sp = 96)
    _case("split_u40_t682", "NJ=3", 682, 40, tl=(682, "min-1", 682, 300), ul=(40, 40, 0, 20), kinds="pbrs",
          gc=(-0.6, 3.0, 0.25, 1.7), neg_inf=((0, 600, "label"), (3, 7, "other")), seed=4),
    _case("fallback_u40_t683", "fallback", 683, 40, tl=(683, "min-1", 683, 300), ul=(40, 40, 0, 20), kinds="pbrs",
          gc=(-0.6, 3.0, 0.25, 1.7), neg_inf=((0, 600, "label"), (3, 7, "other")), seed=4),
    # barrier form at its two widths, each at the largest T it takes and one frame more (fallback)
    _case("nj0_u128_t210", "NJ=0", 210, 128, tl=(210, "min", 150, 60, 1), ul=(128, 128, 0, 3, 1), kinds="rprbr",
          gc=_rot(2), neg_inf=((0, 5, "label"), (0, 9, "other")), seed=5),
    _case("fallback_u128_t211", "fallback", 211, 128, tl=(211, "min", 150, 60, 1), ul=(128, 128, 0, 3, 1),
          kinds="rprbr", gc=_rot(2), neg_inf=((0, 5, "label"), (0, 9, "other")), seed=5),
    _case("nj0_u255_t103", "NJ=0", 103, 255, tl=(103, "min", 103, 1, 50), ul=(255, 60, 100, 1, 0), kinds="rpbrr",
          gc=_rot(3), seed=6),
    _case("fallback_u255_t104", "fallback", 104, 255, tl=(104, "min", 104, 1, 50), ul=(255, 60, 100, 1, 0),
          kinds="rpbrr", gc=_rot(3), seed=6),
    # fallback by Sp: 544 and the largest, 1024
    _case("fallback_u256", "fallback", 300, 256, tl=(300, "min", 300, 299), ul=(256, 256, 2, 0), kinds="rpbr",
          gc=(1.7, -0.6, 3.0, 0.0), neg_inf=((0, 1, "label"),), seed=7),
    _case("fallback_u511", "fallback", 600, 511, tl=(600, "min-1", 599), ul=(511, 511, 5), kinds="prb",
          gc=(-0.6, 1.7, 0.25), seed=8),
    # vocabularies: blank only; two entries (one label: every target is one label throughout) with blank first and
    # last; blank in the middle; a large vocabulary with blank last
    _case("vocab1", "NJ=1", 30, 3, tl=(30, 1, 0, 17), ul=(0, 0, 0, 0), kinds="rrrr", gc=(1.7, -0.6, 3.0, 0.0),
          V=1, blank=0, seed=9),
    _case("vocab2_blank0", "NJ=1", 30, 8, tl=(30, "min", "min-1", 12), ul=(8, 8, 8, 3), kinds="rrrb",
          gc=(1.7, -0.6, 3.0, 0.0), V=2, blank=0, seed=10),
    _case("vocab2_blank1", "NJ=1", 30, 8, tl=(30, "min", 1, 12), ul=(8, 5, 1, 3), kinds="brrr",
          gc=(-0.6, 1.7, 0.25, 3.0), V=2, blank=1, seed=11),
    _case("vocab33_blank16", "NJ=2", 40, 20, tl=(40, "min", 33, 40), ul=(20, 20, 9, 0), kinds="bpsr",
          gc=(3.0, 0.25, -0.6, 1.7), V=33, blank=16, neg_inf=((0, 4, "label"), (2, 30, "other")), seed=12),
    _case("vocab4097_blank4096", "NJ=2", 40, 20, tl=(40, "min", 25, 1), ul=(20, 20, 7, 0), kinds="bprr",
          gc=(0.25, 3.0, -0.6, 0.0), V=4097, blank=4096, neg_inf=((2, 3, "other"),), seed=13),
]

# out-of-range values, in the split form (NJ = 1) and the fallback (Sp = 544): lengths -1, -5, 0, T + 50 and -3,
# Umax + 9; labels -7, V, 10^6 (two of them side by side, and one next to a target equal to blank)
BAD_V, BAD_BLANK = 40, 3
BAD_LABELS = {(3, 0): BAD_V, (5, 1): -7, (5, 2): 10 ** 6, (6, 0): BAD_V, (6, 1): BAD_BLANK, (7, 4): 10 ** 6}


def _bad_case(form, T, umax, seed):
    return _case(f"badvalues_{form}", form, T, umax, tl=(-1, -5, 0, T + 50, T, T, 7, T - 1),
                 ul=(4, 0, 3, umax + 9, -3, 5, 3, 5), kinds="rrrrrrrr", gc=(1.7, -0.6, 0.25, 3.0, 0.0, 0.8, -2.2, 1.1),
                 V=BAD_V, blank=BAD_BLANK, seed=seed)


BAD_CASES = [_bad_case("NJ=1", 14, 6, 20), _bad_case("fallback", 300, 256, 21)]


# ----------------------------------------------------------------------------------------------------------- inputs
def min_frames(labels):
    """Frames of the shortest alignment: one per label and one blank between equal neighbours."""
    return len(labels) + sum(int(labels[i] == labels[i - 1]) for i in range(1, len(labels)))


def make_inputs(c):
    """(logits [B,T,V] fp32 with any -inf planted, targets [B,Umax] int64, input lengths, target lengths) of case c,
    lengths resolved but not clamped."""
    g = torch.Generator().manual_seed(7000 + c["seed"])
    B, T, V, umax, blank = c["B"], c["T"], c["V"], c["umax"], c["blank"]
    logits = 2.0 * torch.randn(B, T, V, generator=g)
    if V > 1:
        tgt = torch.randint(0, V - 1, (B, umax), generator=g)
        tgt += (tgt >= blank).long()                            # never blank
    else:
        tgt = torch.zeros((B, umax), dtype=torch.long)
    tl = []
    for b, kind in enumerate(c["kinds"]):
        U = min(max(c["ul"][b], 0), umax)
        if kind == "p":
            for u in range(1, U, 8):
                tgt[b, u] = tgt[b, u - 1]
        elif kind == "s":
            tgt[b, :] = tgt[b, 0]
        elif kind == "b" and U > 0:
            for u in {0, U // 2, U - 1}:
                tgt[b, u] = blank
        t = c["tl"][b]
        if isinstance(t, str):
            t = min_frames(tgt[b, :U].tolist()) - (t == "min-1")
            assert 0 < t <= T, (c["name"], b, t)
        tl.append(t)
    for (b, t, where) in c["neg_inf"]:
        U = min(max(c["ul"][b], 0), umax)
        labels = tgt[b, :U].tolist()
        col = next(v for v in labels if v != blank) if where == "label" else \
            min(v for v in range(V) if v != blank and v not in labels)
        logits[b, t, col] = -float("inf")
    return logits, tgt, tl, list(c["ul"])


def clamped(c, tgt, tl, ul):
    """The op's contract: lengths clamped to [0, T] / [0, Umax], labels outside [0, V) read as blank."""
    tl = [min(max(t, 0), c["T"]) for t in tl]
    ul = [min(max(u, 0), c["umax"]) for u in ul]
    tgt = torch.where((tgt >= 0) & (tgt < c["V"]), tgt, torch.full_like(tgt, c["blank"]))
    return tgt, tl, ul


def rel_l2(a, b):
    return float((a - b).norm() / max(float(b.norm()), 1e-300))


def reference(logits, tgt, tl, ul, blank):
    """ATen's CPU ctc_loss (reduction='none', zero_infinity=True) on log_softmax(logits), in fp64 and in fp32.  Returns
    the fp64 costs and d cost_b / d logits_b, and per utterance the rel-L2 error of the fp32 gradient and of its blank
    column against fp64: the reference's own rounding.

    ATen's backward forms exp(lcab + nll - lp) with lp = -inf for a -inf logit, which is NaN.  The references see -1e4
    in its place: its probability, e^-1e4, is exactly 0 in fp64 and fp32, so their costs and gradients are those of the
    -inf limit (d cost / d logit = 0 in that column).

    On the last frame ATen sets, rather than adds, the entry of the last target, which drops the final blank state when
    that target is blank (tests/test_oracle_cpu.py shows it against central differences).  Both final states are then
    labelled blank, so the last frame's gradient is softmax - onehot(blank); the references take that row instead."""
    x = torch.where(torch.isneginf(logits), torch.full_like(logits, REF_NEG), logits)
    out = {}
    for dt in (torch.float64, torch.float32):
        xr = x.to(dt).requires_grad_(True)
        costs = torch.nn.functional.ctc_loss(xr.transpose(0, 1).log_softmax(2), tgt, torch.tensor(tl), torch.tensor(ul),
                                             blank=blank, reduction="none", zero_infinity=True)
        costs.sum().backward()                 # cost_b depends on logits[b] alone: this is each utterance's gradient
        grad = xr.grad.clone()
        for b, (Tb, Ub) in enumerate(zip(tl, ul)):
            if Ub > 0 and int(tgt[b, Ub - 1]) == blank and Tb >= max(1, min_frames(tgt[b, :Ub].tolist())):
                grad[b, Tb - 1] = torch.softmax(xr.detach()[b, Tb - 1], 0)
                grad[b, Tb - 1, blank] -= 1
        out[dt] = costs.detach().double(), grad.double()
    (c64, g64), (_, g32) = out[torch.float64], out[torch.float32]
    err32 = [rel_l2(g32[b], g64[b]) for b in range(len(tl))]
    err32_blank = [rel_l2(g32[b, :, blank], g64[b, :, blank]) for b in range(len(tl))]
    return dict(costs=c64, grad=g64, err32=err32, err32_blank=err32_blank)


def check(got, ref, tgt, tl, ul, gc, blank, cost_tol=COST_TOL):
    """Per-utterance comparison of got = {costs [B], grad [B,T,V] = d sum_b gc_b cost_b / d logits} with the
    reference on clamped inputs.  Returns (failures, worst errors).  An utterance without frames or without a valid
    alignment has cost exactly 0 and an all-zero gradient, as has one with gc_b = 0; frames t >= T_b have zero
    gradient.  "use" is the largest gradient error / bar ratio."""
    fails, worst = [], dict(cost=0.0, grad=0.0, blank=0.0, use=0.0)
    for k in ("costs", "grad"):
        if not bool(torch.isfinite(got[k]).all()):
            fails.append(f"{k}: not finite")
    for b in range(len(gc)):
        Tb, Ub = tl[b], ul[b]
        c, r = float(got["costs"][b]), float(ref["costs"][b])
        dead = Tb == 0 or Tb < min_frames(tgt[b, :Ub].tolist())
        if dead:
            if c != 0.0 or r != 0.0:
                fails.append(f"b={b}: cost {c} (reference {r}) without a valid alignment, T_b = {Tb}")
        else:
            e = abs(c - r) / max(1.0, abs(r))
            worst["cost"] = max(worst["cost"], e)
            if not e <= cost_tol:
                fails.append(f"b={b}: cost {c} against {r} (rel {e:.2e} > {cost_tol:.0e})")
        g = got["grad"][b]
        if bool((g[Tb:] != 0).any()):
            fails.append(f"b={b}: nonzero gradient beyond T_b = {Tb}")
        if gc[b] == 0 or dead:
            if bool((g != 0).any()):
                fails.append(f"b={b}: nonzero gradient for cotangent {gc[b]} / T_b = {Tb} / infeasible = {dead}")
            continue
        want = gc[b] * ref["grad"][b]
        for tag, e, bar in (("grad", rel_l2(g, want), max(GRAD_TOL, 3 * ref["err32"][b])),
                            ("blank", rel_l2(g[:, blank], want[:, blank]), max(GRAD_TOL, 3 * ref["err32_blank"][b]))):
            worst[tag] = max(worst[tag], e)
            worst["use"] = max(worst["use"], e / bar)
            if not e <= bar:
                fails.append(f"b={b}: {tag} rel-L2 {e:.2e} > {bar:.1e}")
    return fails, worst


# ------------------------------------------------------------------------------------------------------------- CPU
def test_checker_rejects_planted_faults():
    """The checker accepts the reference itself and rejects four faults a batch-wide comparison can dilute: the blank
    entry of one frame off by 1e-3 relative, two utterances' gradients swapped, one nonzero entry in a padded frame
    and a gradient for an utterance whose cotangent is 0."""
    c = _case("planted", "NJ=1", 8, 3, tl=(8, 6, 8, 7), ul=(3, 2, 3, 1), kinds="bprr", gc=(1.7, -0.6, 0.0, 3.0), V=7,
              blank=2, seed=40)
    logits, tgt, tl, ul = make_inputs(c)
    ref = reference(logits, tgt, tl, ul, c["blank"])
    truth = dict(costs=ref["costs"].clone(), grad=ref["grad"] * torch.tensor(c["gc"], dtype=torch.float64)[:, None, None])
    assert check(truth, ref, tgt, tl, ul, c["gc"], c["blank"])[0] == []

    def planted(edit):
        got = {k: v.clone() for k, v in truth.items()}
        edit(got)
        return check(got, ref, tgt, tl, ul, c["gc"], c["blank"])[0]

    def blank_entry(got):
        t = int(got["grad"][0, :, c["blank"]].abs().argmax())
        got["grad"][0, t, c["blank"]] *= 1 + 1e-3

    def swapped(got):
        got["grad"][[0, 3]] = got["grad"][[3, 0]]

    def padded(got):
        got["grad"][1, 7, 4] = 1e-6

    def zero_cotangent(got):
        got["grad"][2] = ref["grad"][2]

    for edit, what in ((blank_entry, "b=0: blank"), (swapped, "b=3: grad"), (padded, "b=1: nonzero gradient beyond"),
                       (zero_cotangent, "b=2: nonzero gradient for cotangent")):
        fails = planted(edit)
        assert any(f.startswith(what) for f in fails), (what, fails)
    assert any(f.startswith("b=0: grad") for f in planted(swapped))


def test_reference_matches_the_restated_loss():
    """reference() against the fp64 restatement of oracle/ctc_oracle.py on targets equal to blank in the first, middle
    and last position, with -inf logits, an infeasible utterance and an empty target."""
    from oracle import ctc_oracle as CO
    c = _case("ref", "NJ=1", 12, 5, tl=(12, 10, "min-1", 12), ul=(5, 4, 5, 0), kinds="bbpr", gc=(1.0, 1.0, 1.0, 1.0), V=9,
              blank=4, neg_inf=((0, 3, "label"), (1, 6, "other")), seed=41)
    logits, tgt, tl, ul = make_inputs(c)
    ref = reference(logits, tgt, tl, ul, c["blank"])
    x = torch.where(torch.isneginf(logits), torch.full_like(logits, REF_NEG), logits).double()
    nll, grad = CO.ctc_loss_restated(x.log_softmax(2).numpy(), tgt.numpy(), tl, ul, c["blank"])
    assert int(tgt[0, 4]) == int(tgt[1, 3]) == c["blank"] and nll[2] == 0.0
    np.testing.assert_allclose(ref["costs"].numpy(), nll, rtol=1e-12)
    np.testing.assert_allclose(ref["grad"].numpy(), grad, rtol=1e-9, atol=1e-12)


def test_case_table_reaches_every_form_and_edge():
    """Through the mirror of the dispatch: every case reaches the form it names; together they reach every form, both
    S edges of every NJ, both sides of the split form's T limit, the largest Sp and both loud errors; and the batches
    hold the utterance edges the module docstring lists."""
    assert (max_split_T(V0, 40), max_split_T(V0, 128), max_split_T(V0, 255)) == (682, 210, 103)
    assert ctc_form(30, 12744, 15) == "NJ=1" and ctc_form(30, 12745, 15) == "vocab"
    assert ctc_form(30, V0, 511) == "fallback" and sp_of(511) == 1024 and ctc_form(30, V0, 512) == "umax"
    edges = {nj: set() for nj in range(9)}
    seen = set()
    for c in CASES + BAD_CASES:
        assert ctc_form(c["T"], c["V"], c["umax"]) == c["form"], c["name"]
        logits, tgt, tl, ul = make_inputs(c)
        tgt, tl, ul = clamped(c, tgt, tl, ul)
        Sp = sp_of(c["umax"])
        if c["form"].startswith("NJ="):
            edges[int(c["form"][3:])].add((Sp - (2 * max(ul) + 1), c["T"]))
        for b in range(c["B"]):
            U, labels = ul[b], tgt[b, :ul[b]].tolist()
            m = min_frames(labels)
            seen |= {k for k, ok in (("U=0 wide", U == 0 and Sp >= 64), ("U=Umax", U == c["umax"] > 0),
                                      ("small U wide", 0 < U <= 3 and Sp >= 128), ("T_b=1", tl[b] == 1),
                                      ("T_b=T", tl[b] == c["T"]), ("min-1", tl[b] == m - 1 > 0), ("min", tl[b] == m > 0),
                                      ("repeat", any(labels[i] == labels[i - 1] for i in range(1, U))),
                                      ("one label", U >= 8 and len(set(labels)) == 1),
                                      ("blank target", c["blank"] in labels)) if ok}
        seen |= {"-inf " + w for (_, _, w) in c["neg_inf"]}
        assert len(set(c["gc"])) == c["B"] and min(c["gc"]) < 0, c["name"]
    assert {"U=0 wide", "U=Umax", "small U wide", "T_b=1", "T_b=T", "min-1", "min", "repeat", "one label",
            "blank target", "-inf label", "-inf other"} <= seen, seen
    for nj in range(1, 9):                       # S = Sp - 31 and S = Sp - 1
        assert {31, 1} <= {d for d, _ in edges[nj]}, (nj, edges[nj])
    assert {(c["umax"], c["T"]) for c in CASES if c["form"] == "NJ=0"} == {(128, 210), (255, 103)}
    fb = {(c["umax"], c["T"]) for c in CASES if c["form"] == "fallback"}
    assert {(40, 683), (128, 211), (255, 104)} <= fb and {256, 511} <= {u for u, _ in fb}
    assert {(40, 682)} <= {(c["umax"], c["T"]) for c in CASES if c["form"] == "NJ=3"}
    vb = {(c["V"], c["blank"]) for c in CASES}
    assert {1, 2, 33, 4097} <= {v for v, _ in vb}
    assert any(b == 0 < v - 1 for v, b in vb) and any(b == v - 1 > 0 for v, b in vb) and any(0 < b < v - 1 for v, b in vb)
    gcs = {g for c in CASES for g in c["gc"]}
    assert 0.0 in gcs and min(gcs) < 0 and min(abs(g) for g in gcs if g) <= 0.1 and max(gcs) >= 3.0
    for c in BAD_CASES:
        assert {-1, -5, 0, c["T"] + 50} <= set(c["tl"]) and {-3, c["umax"] + 9} <= set(c["ul"])
        assert {-7, BAD_V, 10 ** 6} <= set(BAD_LABELS.values())


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def C():
    import ctcvr_b200
    assert torch.cuda.is_available()
    ctcvr_b200._lib.lib()
    return ctcvr_b200


def run_op(C, logits, tgt, tl, ul, blank, gc):
    x = logits.cuda().requires_grad_(True)
    i32 = lambda v: torch.as_tensor(v, dtype=torch.int32).cuda()
    costs, _ = C.ctc_loss_from_logits(x, tgt.cuda(), i32(tl), i32(ul), blank, reduction="none")
    costs.backward(torch.tensor(gc, dtype=torch.float32, device="cuda"))
    return dict(costs=costs.detach().double().cpu(), grad=x.grad.double().cpu())


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[c["name"] for c in CASES])
def test_ctc_loss_per_utterance_vs_fp64(C, c):
    logits, tgt, tl, ul = make_inputs(c)
    ref = reference(logits, tgt, tl, ul, c["blank"])
    got = run_op(C, logits, tgt, tl, ul, c["blank"], c["gc"])
    fails, worst = check(got, ref, tgt, tl, ul, c["gc"], c["blank"], c["cost_tol"])
    print(f"CTC {c['name']} [{c['form']}]: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("c", BAD_CASES, ids=[c["name"] for c in BAD_CASES])
def test_bad_lengths_and_labels_act_as_clamped(C, c):
    """Lengths outside [0, extent] and labels outside [0, V) give what their clamped values give (lengths clamped to
    the extents, such labels read as blank): costs bit for bit, gradients within 1e-6 per utterance; and both agree
    with the fp64 reference on the clamped inputs."""
    logits, tgt, tl, ul = make_inputs(c)
    for (b, u), lab in BAD_LABELS.items():
        tgt[b, u] = lab
    tgt_ok, tl_ok, ul_ok = clamped(c, tgt, tl, ul)
    bad = run_op(C, logits, tgt, tl, ul, c["blank"], c["gc"])
    ok = run_op(C, logits, tgt_ok, tl_ok, ul_ok, c["blank"], c["gc"])
    fails = []
    if not torch.equal(bad["costs"], ok["costs"]):
        fails.append(f"costs {bad['costs'].tolist()} against clamped {ok['costs'].tolist()}")
    for b in range(c["B"]):
        if not rel_l2(bad["grad"][b], ok["grad"][b]) <= 1e-6:
            fails.append(f"b={b}: gradient rel-L2 {rel_l2(bad['grad'][b], ok['grad'][b]):.2e} from the clamped run")
    ref = reference(logits, tgt_ok, tl_ok, ul_ok, c["blank"])
    f, worst = check(bad, ref, tgt_ok, tl_ok, ul_ok, c["gc"], c["blank"])
    print(f"CTC {c['name']} [{c['form']}]: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
    assert not fails + f, "\n".join(fails + f)


@pytest.mark.gpu
@pytest.mark.parametrize("form,T,umax", [("NJ=2", 40, 20), ("fallback", 40, 300)])
def test_grad_scale_through_the_c_abi(C, form, T, umax):
    """ctcvr_ctc_loss's grad_scale: the kernels compute g * scale_b in fp32, so the scaled gradient is bit for bit
    the unscaled one times the scale; the costs do not change."""
    from ctcvr_b200._lib import call, ptr, query, stream
    B, V, blank = 4, 50, 7
    assert ctc_form(T, V, umax) == form
    c = _case("scale", form, T, umax, tl=(T, 33, "min", 17), ul=(20, 20, 12, 0), kinds="bprr", gc=(1.7, -0.6, 0.0, 3.0),
              V=V, blank=blank, seed=50)
    logits, tgt, tl, ul = make_inputs(c)
    lp = torch.log_softmax(logits.cuda(), -1).contiguous()
    tg, il, ulv = tgt.cuda().contiguous(), torch.tensor(tl, dtype=torch.int32).cuda(), torch.tensor(ul, dtype=torch.int32).cuda()
    scale = torch.tensor(c["gc"], dtype=torch.float32, device="cuda")
    ws = torch.empty(max(256, query("ctcvr_ctc_loss_ws_bytes", B, T, umax)), dtype=torch.uint8, device="cuda")

    def go(sc):
        nll, grad = torch.empty(B, device="cuda"), torch.empty(B, T, V, device="cuda")
        call("ctcvr_ctc_loss", ptr(lp), ptr(tg), ptr(il), ptr(ulv), ptr(sc), ptr(nll), ptr(grad), B, T, V, umax, blank, 1,
             ptr(ws), ws.numel(), stream())
        return nll, grad

    n1, g1 = go(None)
    n2, g2 = go(scale)
    torch.cuda.synchronize()
    assert float(g1.abs().sum()) > 0
    assert torch.equal(n1, n2)
    assert torch.equal(g2, g1 * scale[:, None, None])


@pytest.mark.gpu
def test_loud_errors(C):
    """Shapes the kernels do not take raise an error that names the problem: targets wider than 511, a vocabulary one
    past ctc_grad_kernel's shared memory at Sp = 32 (V = 12745 by the mirror), and concatenated 1-D targets."""
    def call(B, T, V, targets, tl, ul):
        x = torch.randn(B, T, V, device="cuda", requires_grad=True)
        return C.ctc_loss_from_logits(x, targets.cuda(), torch.tensor(tl).cuda(), torch.tensor(ul).cuda(), 0,
                                      reduction="none")

    assert ctc_form(600, 20, 512) == "umax"
    with pytest.raises(RuntimeError, match="too long"):
        call(2, 600, 20, torch.ones(2, 512, dtype=torch.long), [600, 600], [512, 3])
    assert ctc_form(8, 12745, 4) == "vocab" and ctc_form(8, 12744, 4) == "NJ=1"
    with pytest.raises(RuntimeError, match="vocabulary 12745 too large"):
        call(2, 8, 12745, torch.ones(2, 4, dtype=torch.long), [8, 8], [4, 2])
    call(2, 8, 12744, torch.ones(2, 4, dtype=torch.long), [8, 8], [4, 2])
    with pytest.raises(ValueError, match=r"\[B, Umax\]"):
        call(2, 8, 20, torch.ones(6, dtype=torch.long), [8, 8], [4, 2])
