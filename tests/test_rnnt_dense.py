"""The dense-logits RNN-T loss (`functional.rnnt_loss`, the C ABI's `ctcvr_rnnt_loss_dense`) and the dense joint
(`functional.joint_logits`, `ctcvr_joint_logits`) held to an fp64 restatement per utterance, at the shapes and values
where their kernels branch:

  * lattice forms: `rnnt_lattice` (csrc/lattice.cu) picks NJ = 1 / 2 / 4 / 8 label columns per lane from U + 1, then
    the padded kernel, the unpadded kernel or, beyond shared memory and for U + 1 > 256, the generic sweep, from the
    padded batch shape (T, U + 1).  Every form runs with ragged lengths (T_b = 1, U_b = 0, T_b = 0, T_b < T with
    U_b = U, the full lattice) and with a clamp that bites;
  * vocabularies around the warp loops over V (1, 2, 31, 32, 33, 412, 1000, 4097), blank at 0, in the middle and last
    (also as blank = -1), targets equal to blank (the blank and label terms land on one column);
  * a cotangent that differs per utterance in sign and size (0, negative, 0.1 .. 3);
  * out-of-range lengths and labels, through Python and through the C ABI: they act as their clamped values;
  * the seam a caller that materialises logits runs (TransducerJoint.forward -> rnnt_loss) against the fused fp32 loss;
  * `joint_logits` and its backward at the tile edges of the SIMT kernel, and its shared-memory limit on D.

Every utterance's cost and its d_logits[b] slice are compared on their own, so one bad utterance cannot hide in a
batch average.  The CPU tests check the oracle against torchaudio, the checker itself (planted faults are caught) and
the coverage of the case table through a mirror of the lattice dispatch."""
import contextlib
import math
import os

import numpy as np
import pytest
import torch

from oracle import transducer_oracle as TO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32_TOL = 1e-4          # fp32: each cost within 1e-4 relative, each utterance's gradient within 1e-4 rel-L2 (+ fp32 noise)
BITE = 0.05             # a clamp that bites: |d cost / d logit| exceeds it on the blank / label entries
JOINT_TOL = 1e-5        # joint_logits rows and _JointLogits.backward against fp64
GC = (1.7, 0.25, -0.6, 3.0, 0.1, 0.0)


# ---------------------------------------------------------------------------------------------------------- case table
def ragged(T, U):
    """(T_b, U_b) of six utterances: the full lattice, T_b = 1, U_b = 0, T_b = 0, T_b < T with U_b = U, and one in the
    middle (which takes the zero cotangent of GC)."""
    return [(T, U), (1, U // 2), (T - T // 3, 0), (0, U // 3), (max(T - 1, 1), U), (max(T // 2, 1), U // 2)]


def _case(name, T, U1, V, blank, seed, rot=0):
    lens = ragged(T, U1 - 1)
    lens, gc = lens[rot:] + lens[:rot], list(GC[rot:] + GC[:rot])        # the full lattice is not always utterance 0
    # targets equal to blank: label 0 of the first and label 2 of the second utterance with frames and U_b >= 3
    live = [b for b, (t, u) in enumerate(lens) if t > 0 and u >= 3][:2]
    return dict(name=name, B=len(lens), T=T, U1=U1, V=V, blank=blank, tl=[t for t, _ in lens], ul=[u for _, u in lens],
                gc=gc, blank_targets=tuple(zip(live, (0, 2))), seed=seed)


# (T, U + 1) of each lattice form, from lattice_form() below; V = 13 keeps the fp64 oracle cheap on the long lattices
FORM_SHAPES = [
    ((50, 32), (1, 1), (12, 1), (1, 9)),              # NJ 1, padded
    ((9, 33), (260, 41)),                              # NJ 2, padded ((260, 41) is 2.6 KiB under its limit)
    ((20, 65),),                                       # NJ 4, padded
    ((400, 32),),                                      # NJ 1, unpadded
    ((150, 64),),                                      # NJ 2, unpadded
    ((7, 128), (100, 128)),                            # NJ 4, unpadded
    ((5, 129), (30, 256)),                             # NJ 8, unpadded
    ((1800, 9), (420, 64), (600, 100)),                # beyond shared memory: the generic sweep
    ((2, 257), (1, 300)),                              # U + 1 > 256: the generic sweep
]
LATTICE_CASES = [_case(f"T{T}_U1{U1}", T, U1, 13, 5, seed=i, rot=i % 6)
                 for i, (T, U1) in enumerate(s for group in FORM_SHAPES for s in group)]

VOCABS = (1, 2, 31, 32, 33, 412, 1000, 4097)
VOCAB_CASES = [_case(f"V{V}_blank{blank}", 13, 7, V, blank, seed=100 + 3 * i + j, rot=j)
               for i, V in enumerate(VOCABS) for j, blank in enumerate(dict.fromkeys((0, V // 2, -1)))]

# out-of-range values through Python: negative target lengths and logit lengths of 0 / -5 on utterances that are not
# the longest; labels < 0 on an utterance that is not the first and >= V on one that is not the last (so the reads of a
# kernel that did not map them stay inside the logits and fail on values)
BAD = dict(B=7, T=12, U1=8, V=40, blank=3, tl=[12, 7, 0, -5, 9, 12, 10], ul=[7, -1, 5, 3, -100, 4, 6],
           gc=[1.7, -0.6, 0.25, 3.0, -2.2, 0.8, 0.1], seed=30)
BAD_LABELS = {(5, 1): -1, (5, 3): -7, (0, 2): 40, (0, 5): 45, (6, 4): 3}          # (b, u) -> label; V = 40, blank = 3


def resolved_blank(c):
    return c["blank"] % c["V"]


def clamped_lengths(c):
    """The op's contract for lengths: clamped to [0, T] and [0, U]."""
    return [min(max(t, 0), c["T"]) for t in c["tl"]], [min(max(u, 0), c["U1"] - 1) for u in c["ul"]]


# ------------------------------------------------------------------- mirror of the C++ lattice dispatch (csrc/lattice.cu)
# lattice_form restates rnnt_lattice and launch_lattice for the coverage check below; LATTICE_DISPATCH holds the source
# lines it restates, so the check fails when the C++ changes and the mirror does not.
LATTICE_DISPATCH = (
    "const int pad3 = U1, pitch3 = (U1 + 2) & ~1;",
    "const size_t smem3 = (size_t)4 * (T + 2 * pad3) * pitch3 * sizeof(float);",
    "if (smem3 <= 227 * 1024) {",
    "const int pitch = (U1 % 2 == 0) ? U1 : U1 + 1;",
    "const size_t smem4 = (size_t)4 * T * pitch * sizeof(float);",
    "if (smem4 <= 220 * 1024) {",
    "if (U1 <= 32) return launch_lattice<1>(",
    "if (U1 <= 64) return launch_lattice<2>(",
    "if (U1 <= 128) return launch_lattice<4>(",
    "if (U1 <= 256) return launch_lattice<8>(",
)


def lattice_form(T, U1):
    """('padded' | 'unpadded', NJ) or ('generic', 'smem' | 'U1>256'): the kernel rnnt_lattice runs for a batch shape."""
    if U1 > 256:
        return ("generic", "U1>256")
    NJ = 1 if U1 <= 32 else 2 if U1 <= 64 else 4 if U1 <= 128 else 8
    if 16 * (T + 2 * U1) * ((U1 + 2) & ~1) <= 227 * 1024:
        return ("padded", NJ)
    if 16 * T * (U1 if U1 % 2 == 0 else U1 + 1) <= 220 * 1024:
        return ("unpadded", NJ)
    return ("generic", "smem")


# padded NJ = 8 cannot happen: U + 1 >= 129 needs 16 * (1 + 258) * 130 bytes > 227 KiB
ALL_FORMS = {("padded", 1), ("padded", 2), ("padded", 4), ("unpadded", 1), ("unpadded", 2), ("unpadded", 4),
             ("unpadded", 8), ("generic", "smem"), ("generic", "U1>256")}


# ----------------------------------------------------------------------------------------------------------- inputs
def make_inputs(c):
    g = torch.Generator().manual_seed(2000 + c["seed"])
    B, T, U1, V = c["B"], c["T"], c["U1"], c["V"]
    logits = torch.randn(B, T, U1, V, generator=g)
    tgt = torch.randint(0, V, (B, U1 - 1), generator=g, dtype=torch.int32)
    for (i, u) in c.get("blank_targets", ()):
        tgt[i, u] = resolved_blank(c)
    return logits, tgt


def oracle(logits, tgt, tl, ul, blank, clamp, gc, dtype=torch.float64):
    """fp64 restatement on valid inputs: costs [B] and d_logits [B,T,U1,V], the clamped gradient times gc[b]."""
    r = TO.rnnt_lattice_restated(logits, tgt, torch.tensor(tl), torch.tensor(ul), blank, clamp, dtype)
    gcd = torch.tensor(gc, dtype=torch.float64).reshape(-1, 1, 1, 1)
    return dict(costs=r["costs"].double(), grads=r["grads"].double() * gcd)


def rel_l2(a, b):
    return float((a - b).norm() / max(float(b.norm()), 1e-300))


def lattice_base2_fp32(logits, targets, logit_lengths, target_lengths, blank, clamp=-1.0, dtype=torch.float32):
    """rnnt_lattice_restated in fp32 with the alpha / beta recursions of the shared-memory lattice kernels (padded and
    unpadded, csrc/lattice.cu): log-probs scaled by log2(e), log2(2^a + 2^c) per step, beta started from
    beta(T_b, U_b) = 0, alpha / beta / cost scaled back by ln 2; then the closed-form gradient.  Exact exp2 / log2 stand
    in for the kernels' ex2 / lg2 approximations.  This is the same quantity computed in fp32 by the kernels' formulas,
    for the bars below."""
    assert dtype == torch.float32
    r = _LATTICE(logits, targets, logit_lengths, target_lengths, blank, clamp, torch.float32)
    B, T, U1, V = logits.shape
    l2e, ln2, ninf = torch.tensor(math.log2(math.e)), torch.tensor(math.log(2.0)), float("-inf")
    x = logits.detach().float()
    costs, grads = torch.zeros(B), torch.zeros(B, T, U1, V)
    tgt = targets.long()

    def lse2(a, c):
        m, n = torch.maximum(a, c), torch.minimum(a, c)
        return m + torch.log2(1 + torch.exp2(torch.where(n == ninf, torch.full_like(n, ninf), n - m)))

    for b in range(B):
        Tb, Ub = int(logit_lengths[b]), int(target_lengths[b])
        if Tb == 0:
            continue
        lpb, lpl = r["lp_blank"][b] * l2e, r["lp_label"][b] * l2e
        a, be = torch.full((Tb, Ub + 1), ninf), torch.full((Tb + 1, Ub + 2), ninf)
        a[0, 0], be[Tb, Ub] = 0.0, 0.0
        for d in range(1, Tb + Ub):
            t = torch.arange(max(0, d - Ub), min(Tb - 1, d) + 1)
            u, tm, um = d - t, (t - 1).clamp(min=0), (d - t - 1).clamp(min=0)
            a[t, u] = lse2(torch.where(t > 0, a[tm, u] + lpb[tm, u], torch.tensor(ninf)),
                           torch.where(u > 0, a[t, um] + lpl[t, um], torch.tensor(ninf)))
        for d in range(Tb - 1 + Ub, -1, -1):
            t = torch.arange(max(0, d - Ub), min(Tb - 1, d) + 1)
            u = d - t
            be[t, u] = lse2(be[t + 1, u] + lpb[t, u], torch.where(u < Ub, be[t, u + 1] + lpl[t, u], torch.tensor(ninf)))
        al, bt, cost = a * ln2, be[:Tb + 1, :Ub + 1] * ln2, -be[0, 0] * ln2
        xb, lse = x[b, :Tb, :Ub + 1], r["lse"][b, :Tb, :Ub + 1]
        k = al + cost - lse
        g = torch.exp(xb + (k + bt[:Tb])[..., None])
        g[..., blank] -= torch.exp(xb[..., blank] + k + bt[1:])
        if Ub > 0:
            idx = tgt[b, :Ub][None, :, None].expand(Tb, Ub, 1)
            gl = torch.exp(torch.gather(xb[:, :Ub], 2, idx)[..., 0] + k[:, :Ub] + bt[:Tb, 1:])
            g[:, :Ub].scatter_add_(2, idx, -gl[..., None])
        if clamp > 0:
            g = g.clamp(-clamp, clamp)
        costs[b], grads[b, :Tb, :Ub + 1] = cost, g
    return dict(costs=costs, grads=grads, lse=r["lse"])


_LATTICE = TO.rnnt_lattice_restated


@contextlib.contextmanager
def base2_lattice():
    """The oracle's lattice (also inside TO.fused_joint_rnnt_restated) replaced by lattice_base2_fp32."""
    TO.rnnt_lattice_restated = lattice_base2_fp32
    try:
        yield
    finally:
        TO.rnnt_lattice_restated = _LATTICE


def fp32_refs(logits, tgt, tl, ul, blank, clamp, gc):
    """fp32 computations of the op on valid inputs: the restatement, and the base-2 lattice where the shared-memory
    kernels run (not the generic sweep, which computes in natural logarithms like the restatement)."""
    refs = [oracle(logits, tgt, tl, ul, blank, clamp, gc, torch.float32)]
    if lattice_form(logits.shape[1], logits.shape[2])[0] != "generic":
        with base2_lattice():
            refs.append(oracle(logits, tgt, tl, ul, blank, clamp, gc, torch.float32))
    return refs


def bars(ref64, ref32s, tl, gc):
    """Per-utterance gradient bars: 1e-4 plus the rounding of an fp32 computation of the same gradient, estimated by
    the largest distance of the fp32 computations ref32s from fp64 (times 2: one sample of fp32 noise).  That rounding
    is not small on long lattices: the gradient is exp(alpha + beta + cost - lse + x) with alpha + beta + cost the
    difference of numbers as large as the cost (5 000 nats at T = 1800), so an fp32 restatement is 2e-3 off there on
    its own.  The shared-memory lattice kernels recurse in base 2 (log-probs times log2(e), results times ln 2), which
    rounds differently: at T = 30, U + 1 = 256 that formula in fp32 is 3e-4 from fp64 where the restatement is 6e-5."""
    grad = np.full(len(tl), F32_TOL)
    for b, Tb in enumerate(tl):
        if Tb > 0 and gc[b] != 0:
            grad[b] += 2.0 * max(rel_l2(r["grads"][b], ref64["grads"][b]) for r in ref32s)
    return grad


def check(got, ref, tl, ul, gc, grad_tol):
    """Per-utterance comparison.  Returns (failures, worst errors).  tl / ul are the clamped lengths.  A cost is within
    1e-4 relative (1e-4 nats below 1 nat: with V = 1 a cost is -log(number of alignments), 0 for U_b = 0), an
    utterance's gradient within grad_tol[b] rel-L2.  Beyond its lengths, for a zero cotangent and
    without frames, an utterance's gradient is exactly 0; a cost without frames is exactly 0.  `worst` also holds the
    largest error / bar ratio ("use")."""
    fails, worst = [], {"cost": 0.0, "grad": 0.0, "use": 0.0}
    for k in ("costs", "grads"):
        if not bool(torch.isfinite(got[k]).all()):
            fails.append(f"{k}: not finite")
    for b in range(len(gc)):
        Tb, Ub = tl[b], ul[b]
        c, r = float(got["costs"][b]), float(ref["costs"][b])
        if Tb == 0:
            if c != 0.0:
                fails.append(f"b={b}: cost {c} without frames")
        else:
            e = abs(c - r) / max(abs(r), 1.0)
            worst["cost"] = max(worst["cost"], e)
            worst["use"] = max(worst["use"], e / F32_TOL)
            if not e <= F32_TOL:
                fails.append(f"b={b}: cost {c} against {r} (rel {e:.2e} > {F32_TOL:.1e})")
        g = got["grads"][b]
        if bool((g[Tb:] != 0).any()) or bool((g[:, Ub + 1:] != 0).any()):
            fails.append(f"b={b}: nonzero gradient beyond T_b = {Tb} / U_b = {Ub}")
        if gc[b] == 0 or Tb == 0:
            if bool((g != 0).any()):
                fails.append(f"b={b}: nonzero gradient for cotangent {gc[b]} / T_b = {Tb}")
            continue
        if g.shape[-1] == 1:
            # one symbol: the three terms of an entry are all its occupancy and cancel, so the fp64 gradient is rounding
            # noise and a relative bar says nothing; the gradient must be as small as fp32 rounding
            if not float(g.abs().max()) <= F32_TOL * abs(gc[b]):
                fails.append(f"b={b}: V = 1 gradient {float(g.abs().max()):.2e} is not 0")
            continue
        e = rel_l2(g, ref["grads"][b])
        worst["grad"] = max(worst["grad"], e)
        worst["use"] = max(worst["use"], e / grad_tol[b])
        if not e <= grad_tol[b]:
            fails.append(f"b={b}: grad rel-L2 {e:.2e} > {grad_tol[b]:.1e}")
    return fails, worst


# ------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("blank", [0, 4, 8])
def test_oracle_matches_torchaudio(blank):
    """The fp64 oracle restates torchaudio's CPU rnnt_loss (fp32): costs and per-utterance gradients under a cotangent,
    with ragged lengths, with and without a clamp that bites, within the fp32 floor (measured ~1e-7 on costs, ~2e-6 on
    gradients).  Targets avoid blank: there torchaudio's gradient drops the label term (next test)."""
    ta = pytest.importorskip("torchaudio")
    g = torch.Generator().manual_seed(40 + blank)
    B, T, U1, V = 5, 10, 6, 9
    tl, ul, gc = [10, 7, 1, 10, 4], [3, 5, 2, 0, 5], [1.7, -0.6, 0.0, 3.0, 0.1]
    for clamp in (-1.0, BITE):
        x = torch.randn(B, T, U1, V, generator=g)
        tgt = torch.randint(0, V - 1, (B, U1 - 1), generator=g, dtype=torch.int32)
        tgt[tgt >= blank] += 1
        xx = x.clone().requires_grad_(True)
        costs = ta.functional.rnnt_loss(xx, tgt, torch.tensor(tl, dtype=torch.int32),
                                        torch.tensor(ul, dtype=torch.int32), blank=blank, clamp=clamp,
                                        reduction="none")
        costs.backward(torch.tensor(gc))
        ref = oracle(x, tgt, tl, ul, blank, clamp, gc)
        if clamp > 0:
            assert not torch.equal(ref["grads"], oracle(x, tgt, tl, ul, blank, -1.0, gc)["grads"]), "clamp does not bite"
        got = dict(costs=costs.detach().double(), grads=xx.grad.double())
        fails, worst = check(got, ref, tl, ul, gc, np.full(B, 1e-5))
        assert not fails and worst["cost"] <= 1e-6, (clamp, fails, worst)


def test_oracle_gradient_at_blank_targets_is_the_derivative():
    """Where a target equals blank, both the blank and the label term land on one column.  The oracle (and the
    library) subtract both, which is the derivative of the cost (central differences in fp64); torchaudio's CPU op
    subtracts only the blank term there, so its gradient is not the derivative of its own cost."""
    ta = pytest.importorskip("torchaudio")
    g = torch.Generator().manual_seed(41)
    T, U1, V, blank = 3, 3, 4, 1
    x = torch.randn(1, T, U1, V, generator=g, dtype=torch.float64)
    tgt = torch.tensor([[blank, 2]], dtype=torch.int32)
    tl, ul = [T], [U1 - 1]
    grad = oracle(x, tgt, tl, ul, blank, -1.0, [1.0])["grads"]
    fd, h = torch.zeros_like(x), 1e-6
    for i in range(x.numel()):
        xp, xm = x.clone(), x.clone()
        xp.view(-1)[i] += h
        xm.view(-1)[i] -= h
        fd.view(-1)[i] = (oracle(xp, tgt, tl, ul, blank, -1.0, [1.0])["costs"][0] -
                          oracle(xm, tgt, tl, ul, blank, -1.0, [1.0])["costs"][0]) / (2 * h)
    assert rel_l2(grad, fd) < 1e-7
    xx = x.float().requires_grad_(True)
    ta.functional.rnnt_loss(xx, tgt, torch.tensor(tl, dtype=torch.int32), torch.tensor(ul, dtype=torch.int32),
                            blank=blank, reduction="sum").backward()
    assert rel_l2(xx.grad.double(), fd) > 1e-2


def test_checker_rejects_planted_faults():
    """The per-utterance checker at the fp32 bars accepts the truth and rejects: the label term dropped at one cell, the
    clamp not applied, one utterance's cotangent ignored (a negative one and a zero one), a tiny nonzero gradient beyond
    U_b and beyond T_b, the terminal cell's blank term missing, and one cost off by 2e-4."""
    g = torch.Generator().manual_seed(7)
    B, T, U1, V, blank = 4, 9, 6, 11, 2
    x = torch.randn(B, T, U1, V, generator=g)
    tgt = torch.randint(0, V, (B, U1 - 1), generator=g, dtype=torch.int32)
    tl, ul, gc = [9, 6, 9, 3], [5, 2, 4, 0], [1.7, -0.6, 0.0, 3.0]
    ref = oracle(x, tgt, tl, ul, blank, -1.0, gc)
    tol = bars(ref, [oracle(x, tgt, tl, ul, blank, -1.0, gc, torch.float32)], tl, gc)
    assert check(ref, ref, tl, ul, gc, tol)[0] == []
    r = TO.rnnt_lattice_restated(x, tgt, torch.tensor(tl), torch.tensor(ul), blank)

    def planted(edit, ref=ref):
        got = {k: v.clone() for k, v in ref.items()}
        edit(got)
        return check(got, ref, tl, ul, gc, tol)[0]

    def label_dropped(got):
        b, t, u = 0, 4, 2
        term = math.exp(float(r["alpha"][b, t, u] + r["lp_label"][b, t, u] + r["beta"][b, t, u + 1] + r["costs"][b]))
        got["grads"][b, t, u, int(tgt[b, u])] += gc[b] * term

    def terminal_blank_off(got):
        b = 1
        t, u = tl[b] - 1, ul[b]
        got["grads"][b, t, u, blank] += gc[b] * math.exp(float(r["alpha"][b, t, u] + r["lp_blank"][b, t, u] + r["costs"][b]))

    def cotangent_ignored(got):
        got["grads"][1] /= gc[1]

    def zero_cotangent_ignored(got):
        got["grads"][2] = oracle(x, tgt, tl, ul, blank, -1.0, [1.0] * B)["grads"][2]

    def beyond_u(got):
        got["grads"][3, 1, ul[3] + 1, 0] = 1e-30

    def beyond_t(got):
        got["grads"][1, tl[1], 0, 5] = -1e-30

    def cost(got):
        got["costs"][0] *= 1 + 2e-4

    for edit, what in ((label_dropped, "b=0: grad"), (terminal_blank_off, "b=1: grad"), (cotangent_ignored, "b=1: grad"),
                       (zero_cotangent_ignored, "b=2: nonzero gradient for cotangent"),
                       (beyond_u, "b=3: nonzero gradient beyond"), (beyond_t, "b=1: nonzero gradient beyond"),
                       (cost, "b=0: cost")):
        fails = planted(edit)
        assert any(f.startswith(what) for f in fails), (edit.__name__, fails)
    # the clamp not applied: an unclamped gradient against the clamped reference
    clamped = oracle(x, tgt, tl, ul, blank, BITE, gc)
    fails = check(ref, clamped, tl, ul, gc, tol)[0]
    assert any("grad rel-L2" in f for f in fails), fails


def test_case_table_reaches_every_lattice_form():
    """Through the mirror of the C++ dispatch: the case table reaches every lattice form, each form's shapes are where
    the table says, and every case has the five ragged kinds, a zero, a negative and a large cotangent."""
    src = open(os.path.join(ROOT, "ctc-vr_b200", "csrc", "lattice.cu")).read()
    for line in LATTICE_DISPATCH:
        assert line in src, f"lattice.cu changed ({line!r}): update lattice_form()"
    assert {lattice_form(c["T"], c["U1"]) for c in LATTICE_CASES} == ALL_FORMS
    # every reachable form is listed: sweep the shapes
    assert {lattice_form(T, U1) for T in range(1, 2000, 7) for U1 in range(1, 300, 3)} == ALL_FORMS
    want = [("padded", 1), ("padded", 2), ("padded", 4), ("unpadded", 1), ("unpadded", 2), ("unpadded", 4),
            ("unpadded", 8), ("generic", "smem"), ("generic", "U1>256")]
    for form, group in zip(want, FORM_SHAPES):
        assert all(lattice_form(T, U1) == form for T, U1 in group), (form, group)
    for c in LATTICE_CASES + VOCAB_CASES:
        tl, ul = clamped_lengths(c)
        T, U = c["T"], c["U1"] - 1
        pairs = set(zip(tl, ul))
        assert (T, U) in pairs and 0 in tl and any(t == 1 for t in tl) and any(u == 0 and t > 0 for t, u in pairs)
        assert any(t < T and u == U for t, u in pairs) or T == 1, c["name"]
        assert max(tl) == T and max(ul) == U, c["name"]       # rnnt_loss checks the longest lengths against the shape
        assert 0.0 in c["gc"] and min(c["gc"]) < 0 and max(c["gc"]) >= 1.7 and 0.1 in c["gc"], c["name"]
        assert c["T"] * c["U1"] <= 4096 or c["V"] <= 16, c["name"]
    assert {c["V"] for c in VOCAB_CASES} == set(VOCABS) and all(len(c["blank_targets"]) == 2 for c in VOCAB_CASES)
    assert any(c["blank"] == -1 for c in VOCAB_CASES) and any(0 < c["blank"] < c["V"] - 1 for c in VOCAB_CASES)


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def C():
    import ctcvr_b200
    assert torch.cuda.is_available()
    ctcvr_b200._lib.lib()
    return ctcvr_b200


def i32(x):
    return torch.as_tensor(x, dtype=torch.int32).cuda()


def run_dense(C, logits, tgt, tl, ul, blank, clamp, gc):
    """functional.rnnt_loss(..., reduction='none') and costs.backward(gc): costs [B] and d_logits, as fp64 on the CPU."""
    x = logits.cuda().requires_grad_(True)
    costs = C.rnnt_loss(x, tgt.cuda(), i32(tl), i32(ul), blank=blank, clamp=clamp, reduction="none")
    costs.backward(torch.tensor(gc, dtype=torch.float32, device="cuda"))
    return dict(costs=costs.detach().double().cpu(), grads=x.grad.double().cpu())


def run_case(C, c, tag):
    logits, tgt = make_inputs(c)
    tl, ul = clamped_lengths(c)
    blank, gc, fails = resolved_blank(c), c["gc"], []
    refs = {}
    for clamp in (-1.0, BITE):
        ref64 = refs[clamp] = oracle(logits, tgt, tl, ul, blank, clamp, gc)
        ref32 = fp32_refs(logits, tgt, tl, ul, blank, clamp, gc)
        got = run_dense(C, logits, tgt, c["tl"], c["ul"], c["blank"], clamp, gc)
        f, worst = check(got, ref64, tl, ul, gc, bars(ref64, ref32, tl, gc))
        name = f"{c['name']} {tag} clamp={clamp}"
        print(f"DENSE {name}: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
        fails += [f"{name}: {m}" for m in f]
    if c["V"] > 1:
        assert not torch.equal(refs[-1.0]["grads"], refs[BITE]["grads"]), f"{c['name']}: the clamp does not bite"
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("c", LATTICE_CASES, ids=[c["name"] for c in LATTICE_CASES])
def test_lattice_forms_vs_fp64(C, c):
    run_case(C, c, "form=" + ":".join(map(str, lattice_form(c["T"], c["U1"]))))


@pytest.mark.gpu
@pytest.mark.parametrize("c", VOCAB_CASES, ids=[c["name"] for c in VOCAB_CASES])
def test_vocabulary_vs_fp64(C, c):
    run_case(C, c, f"V={c['V']}")


@pytest.mark.gpu
def test_bad_lengths_and_labels_act_as_clamped(C):
    """Negative target lengths, logit lengths of 0 and -5, and labels -1, -7, V and V + 5 through rnnt_loss give what
    their clamped values give (lengths clamped to [0, T] and [0, U], such labels read as blank): costs bit for bit and
    gradients equal; and both agree with the fp64 oracle on the clamped inputs."""
    c = BAD
    logits, tgt = make_inputs(c)
    tgt_bad = tgt.clone()
    for (i, u), lab in BAD_LABELS.items():
        tgt_bad[i, u] = lab
    tgt_ok = torch.where((tgt_bad >= 0) & (tgt_bad < c["V"]), tgt_bad, torch.full_like(tgt_bad, c["blank"]))
    tl, ul = clamped_lengths(c)
    fails = []
    for clamp in (-1.0, BITE):
        ref64 = oracle(logits, tgt_ok, tl, ul, c["blank"], clamp, c["gc"])
        ref32 = fp32_refs(logits, tgt_ok, tl, ul, c["blank"], clamp, c["gc"])
        bad = run_dense(C, logits, tgt_bad, c["tl"], c["ul"], c["blank"], clamp, c["gc"])
        ok = run_dense(C, logits, tgt_ok, tl, ul, c["blank"], clamp, c["gc"])
        print(f"DENSE badvalues clamp={clamp}: costs {bad['costs'].tolist()} clamped {ok['costs'].tolist()}")
        if not torch.equal(bad["costs"], ok["costs"]):
            fails.append(f"clamp={clamp}: costs {bad['costs'].tolist()} against clamped {ok['costs'].tolist()}")
        if not torch.equal(bad["grads"], ok["grads"]):
            fails.append(f"clamp={clamp}: gradients differ from the clamped run "
                         f"(rel-L2 {rel_l2(bad['grads'], ok['grads']):.2e})")
        for name, got in (("bad", bad), ("clamped", ok)):
            f, worst = check(got, ref64, tl, ul, c["gc"], bars(ref64, ref32, tl, c["gc"]))
            print(f"DENSE badvalues {name} clamp={clamp}: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
            fails += [f"{name} clamp={clamp}: {m}" for m in f]
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
def test_c_abi_lengths_beyond_extents_act_as_clamped(C):
    """ctcvr_rnnt_loss_dense called directly with t_len = T + 3 and u_len = U + 2 (which Python cannot pass) on the
    first utterance: costs bit for bit and gradients equal to the call with T and U, every gradient entry written, and
    both within the bars of the fp64 oracle."""
    from ctcvr_b200._lib import call, ptr, query, stream
    c = dict(B=3, T=10, U1=6, V=17, blank=4, seed=60)
    B, T, U1, V, blank = c["B"], c["T"], c["U1"], c["V"], c["blank"]
    logits, tgt = make_inputs(c)
    tl_ok, ul_ok = [T, 7, T], [U1 - 1, 3, U1 - 1]
    tl_bad, ul_bad = [T + 3, 7, T], [U1 + 2, 3, U1 - 1]
    x, tg = logits.cuda(), tgt.cuda()

    def abi(tl, ul):
        tl_d, ul_d = i32(tl), i32(ul)
        costs = torch.full((B,), float("nan"), device="cuda")
        grads = torch.full_like(x, float("nan"))
        ws = torch.empty(query("ctcvr_rnnt_loss_dense_ws_bytes", B, T, U1), dtype=torch.uint8, device="cuda")
        call("ctcvr_rnnt_loss_dense", ptr(x), ptr(tg), ptr(tl_d), ptr(ul_d), ptr(costs), ptr(grads), B, T, U1, V, blank,
             -1.0, ptr(ws), ws.numel(), stream())
        torch.cuda.synchronize()
        return dict(costs=costs.double().cpu(), grads=grads.double().cpu())

    bad, ok = abi(tl_bad, ul_bad), abi(tl_ok, ul_ok)
    gc = [1.0] * B
    ref64 = oracle(logits, tgt, tl_ok, ul_ok, blank, -1.0, gc)
    ref32 = fp32_refs(logits, tgt, tl_ok, ul_ok, blank, -1.0, gc)
    print(f"DENSE C ABI: costs {bad['costs'].tolist()} clamped {ok['costs'].tolist()}")
    assert torch.equal(bad["costs"], ok["costs"]), (bad["costs"], ok["costs"])
    assert torch.equal(bad["grads"], ok["grads"]), rel_l2(bad["grads"], ok["grads"])
    fails, worst = check(bad, ref64, tl_ok, ul_ok, gc, bars(ref64, ref32, tl_ok, gc))
    print("DENSE C ABI vs fp64: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
    assert not fails, "\n".join(fails)


# ------------------------------------------------------------------------------ the dense seam against the fused loss
@contextlib.contextmanager
def fp32_matmuls():
    """cuBLAS fp32 matmuls in full fp32 (torch's default; TF32 off), restored on exit."""
    m = torch.backends.cuda.matmul
    old = m.fp32_precision
    m.fp32_precision = "ieee"
    try:
        yield
    finally:
        m.fp32_precision = old


JOINT_PARAMS = ("enc_ffn.weight", "enc_ffn.bias", "pred_ffn.weight", "pred_ffn.bias", "ffn_out.weight", "ffn_out.bias")


def seam_oracle(enc, pred, w, tgt, tl, ul, blank, gc, dtype=torch.float64):
    r = TO.fused_joint_rnnt_restated(enc, pred, w, tgt, torch.tensor(tl), torch.tensor(ul), blank, -1.0, dtype,
                                     grad_costs=torch.tensor(gc, dtype=torch.float64))
    out = dict(costs=r["costs"].double(), d_enc=r["d_enc_out"].double(), d_pred=r["d_pred_out"].double())
    out.update({k: r["d_" + k].double() for k in JOINT_PARAMS})
    return out


def run_seam(C, joint, path, enc, pred, tgt, tl, ul, blank, gc):
    """Costs, d_enc / d_pred and every joint parameter gradient of one path (reduction='none', costs.backward(gc)):
    'dense' is TransducerJoint.forward -> rnnt_loss, 'fused' is rnnt_loss_fused(precision='fp32')."""
    e, p = enc.cuda().requires_grad_(True), pred.cuda().requires_grad_(True)
    joint.zero_grad(set_to_none=True)
    with fp32_matmuls():
        if path == "dense":
            costs = C.rnnt_loss(joint(e, p), i32(tgt), i32(tl), i32(ul), blank=blank, reduction="none")
        else:
            costs = joint.rnnt_loss_fused(e, p, i32(tgt), i32(tl), i32(ul), blank, reduction="none", precision="fp32")
        costs.backward(torch.tensor(gc, dtype=torch.float32, device="cuda"))
    out = dict(costs=costs.detach().double().cpu(), d_enc=e.grad.double().cpu(), d_pred=p.grad.double().cpu())
    out.update({k: v.grad.double().cpu() for k, v in joint.named_parameters()})
    return out


def seam_check(got, ref, tl, ul, gc, grad_bar, shared_bar):
    """Per utterance: cost within 1e-4 relative, d_enc / d_pred within grad_bar[b] (exact zeros beyond the lengths and
    for a zero cotangent); every parameter gradient within shared_bar[k]."""
    fails, worst = [], {}
    for b in range(len(gc)):
        e = abs(float(got["costs"][b] - ref["costs"][b])) / abs(float(ref["costs"][b]))
        worst["cost"] = max(worst.get("cost", 0.0), e)
        if not e <= F32_TOL:
            fails.append(f"b={b}: cost rel {e:.2e}")
        if bool((got["d_enc"][b, tl[b]:] != 0).any()) or bool((got["d_pred"][b, ul[b] + 1:] != 0).any()):
            fails.append(f"b={b}: nonzero gradient beyond the lengths")
        for k in ("d_enc", "d_pred"):
            if gc[b] == 0:
                if bool((got[k][b] != 0).any()):
                    fails.append(f"b={b}: nonzero {k} for a zero cotangent")
                continue
            e = rel_l2(got[k][b], ref[k][b])
            worst[k] = max(worst.get(k, 0.0), e)
            if not e <= grad_bar[b]:
                fails.append(f"b={b}: {k} rel-L2 {e:.2e} > {grad_bar[b]:.1e}")
    for k in JOINT_PARAMS:
        e = worst[k] = rel_l2(got[k], ref[k])
        if not e <= shared_bar[k]:
            fails.append(f"{k} rel-L2 {e:.2e} > {shared_bar[k]:.1e}")
    return fails, worst


def seam_bars(ref64, ref32s, gc):
    """Bars of one path against fp64: 1e-4 plus twice the largest distance of the fp32 computations ref32s, per
    utterance for d_enc / d_pred (the larger of the two) and per parameter."""
    grad = [F32_TOL + (2.0 * max(rel_l2(r[k][b], ref64[k][b]) for k in ("d_enc", "d_pred") for r in ref32s)
                       if gc[b] != 0 else 0.0) for b in range(len(gc))]
    return grad, {k: F32_TOL + 2.0 * max(rel_l2(r[k], ref64[k]) for r in ref32s) for k in JOINT_PARAMS}


def seam_case(C, joint, enc, pred, tgt, tl, ul, blank, gc, n_ref, tag):
    """Both paths against fp64 on the first n_ref utterances, then against each other on the whole batch, bounded by
    the sum of the two paths' fp64 bars (the largest per-utterance bar of the checked utterances for d_enc / d_pred)."""
    w = {k: v.detach().cpu() for k, v in joint.state_dict().items()}
    s = slice(0, n_ref)
    args = (enc[s], pred[s], w, tgt[s], tl[:n_ref], ul[:n_ref], blank, gc[:n_ref])
    ref64, ref32s = seam_oracle(*args), [seam_oracle(*args, dtype=torch.float32)]
    if lattice_form(enc.shape[1], pred.shape[1])[0] != "generic":
        with base2_lattice():
            ref32s.append(seam_oracle(*args, dtype=torch.float32))
    grad_bar, shared_bar = seam_bars(ref64, ref32s, gc[:n_ref])
    fails = []
    for path in ("dense", "fused"):
        got = run_seam(C, joint, path, enc[s], pred[s], tgt[s], tl[:n_ref], ul[:n_ref], blank, gc[:n_ref])
        f, worst = seam_check(got, ref64, tl[:n_ref], ul[:n_ref], gc[:n_ref], grad_bar, shared_bar)
        print(f"SEAM {tag} {path} vs fp64: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
        fails += [f"{tag} {path}: {m}" for m in f]
    assert not fails, "\n".join(fails)
    dense = run_seam(C, joint, "dense", enc, pred, tgt, tl, ul, blank, gc)
    fused = run_seam(C, joint, "fused", enc, pred, tgt, tl, ul, blank, gc)
    pair = [2 * max(grad_bar)] * len(gc)
    f, worst = seam_check(dense, fused, tl, ul, gc, pair, {k: 2 * v for k, v in shared_bar.items()})
    f = [m for m in f if "cost rel" not in m]
    cost = float(((dense["costs"] - fused["costs"]).abs() / fused["costs"].abs()).max())
    if not cost <= 2 * F32_TOL:
        f.append(f"cost rel {cost:.2e} between the paths")
    print(f"SEAM {tag} dense vs fused (bar {pair[0]:.1e}): " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
    assert not f, "\n".join(f)


@pytest.mark.gpu
def test_dense_seam_matches_fused_cfg1(C):
    """cfg1_example1.npz (B = 2, T = 129, U = 24, D = 256, V = 412): TransducerJoint.forward -> rnnt_loss against
    rnnt_loss_fused(precision='fp32'), both against fp64 and against each other."""
    from conftest import load_golden
    fx = load_golden("cfg1_example1.npz")
    joint = C.TransducerJoint(412, 256, 256, 256).cuda()
    joint.load_state_dict({k[len("joint."):]: torch.from_numpy(v) for k, v in fx.items() if k.startswith("joint.")})
    enc, pred = torch.from_numpy(fx["encoder_out"]), torch.from_numpy(fx["predictor_out"])
    tgt = torch.from_numpy(fx["texts"]).int()
    tl, ul = fx["encoder_out_lens"].tolist(), fx["text_lens"].tolist()
    seam_case(C, joint, enc, pred, tgt, tl, ul, int(fx["blank"]), [1.7, -0.6], 2, "cfg1")


@pytest.mark.gpu
def test_dense_seam_matches_fused_cfg2(C):
    """A cfg2-shaped batch (B = 32, T = 250, U = 40, D = 512, V = 412; 515 MiB of logits): four utterances against
    fp64, the whole batch dense against fused."""
    B, T, U1, D, V, blank = 32, 250, 41, 512, 412, 0
    g = torch.Generator().manual_seed(12)
    torch.manual_seed(12)
    joint = C.TransducerJoint(V, D, D, D)
    joint = joint.cuda()
    enc = torch.randn(B, T, D, generator=g)
    pred = torch.randn(B, U1, D, generator=g)
    tgt = torch.randint(1, V, (B, U1 - 1), generator=g, dtype=torch.int32)
    tl = [T, 187, 250, 131] + torch.randint(T // 2, T + 1, (B - 4,), generator=g).tolist()
    ul = [U1 - 1, 33, 21, 40] + torch.randint(U1 // 2, U1, (B - 4,), generator=g).tolist()
    gc = [1.7, -0.6, 0.25, 3.0] + (torch.rand(B - 4, generator=g) * 2 - 0.5).tolist()
    gc[9] = 0.0
    seam_case(C, joint, enc, pred, tgt, tl, ul, blank, gc, 4, "cfg2")


# ------------------------------------------------------------------------------------------ joint_logits against fp64
# (B, T, U + 1, D, V): T (U + 1) off the 64-row tile, V off the 128-column pass and the 8-column thread group, D off the
# 32-deep k-chunk, D = 784 at the shared-memory limit of the SIMT tile (272 D + 18 688 bytes <= 227 KiB), decode-shaped
JOINT_CASES = [(2, 7, 9, 40, 13), (3, 5, 13, 100, 130), (2, 9, 8, 128, 129), (2, 11, 6, 784, 412), (1, 1, 1, 256, 412),
               (2, 13, 5, 64, 1000)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", JOINT_CASES, ids=["B{}_T{}_U1{}_D{}_V{}".format(*s) for s in JOINT_CASES])
def test_joint_logits_vs_fp64(C, shape):
    """Every (b, t, u) row of joint_logits within 1e-5 rel-L2 of fp64, and _JointLogits.backward (d_enc / d_pred per
    utterance, d_w, d_b) within 1e-5 of fp64 autograd."""
    B, T, U1, D, V = shape
    g = torch.Generator().manual_seed(sum(shape))
    enc, pred = 0.5 * torch.randn(B, T, D, generator=g), 0.5 * torch.randn(B, U1, D, generator=g)
    w, b = torch.randn(V, D, generator=g) / math.sqrt(D), 0.1 * torch.randn(V, generator=g)
    cot = torch.randn(B, T, U1, V, generator=g)
    ins = [t.double().requires_grad_(True) for t in (enc, pred, w, b)]
    ref = torch.nn.functional.linear(torch.tanh(ins[0].unsqueeze(2) + ins[1].unsqueeze(1)), ins[2], ins[3])
    (ref * cot.double()).sum().backward()
    dev = [t.cuda().requires_grad_(True) for t in (enc, pred, w, b)]
    with fp32_matmuls():
        out = C.joint_logits(*dev)
        out.backward(cot.cuda())
    out = out.detach().double().cpu()
    row = ((out - ref.detach()).norm(dim=-1) / ref.detach().norm(dim=-1)).max().item()
    errs = {"rows": row}
    for name, got, want in zip(("d_enc", "d_pred", "d_w", "d_b"), dev, ins):
        gg, ww = got.grad.double().cpu(), want.grad
        errs[name] = max(rel_l2(gg[i], ww[i]) for i in range(B)) if name in ("d_enc", "d_pred") else rel_l2(gg, ww)
    print(f"JOINT {shape}: " + " ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    assert all(v <= JOINT_TOL for v in errs.values()), errs


@pytest.mark.gpu
def test_joint_logits_shared_memory_limit(C):
    """D = 786 needs 232 480 bytes of shared memory for the SIMT tile, over the 227 KiB an SM gives a block: an error,
    not a launch failure or a silent result (D = 784 runs in test_joint_logits_vs_fp64)."""
    D = 786
    with pytest.raises(RuntimeError, match="join_dim 786 too large"):
        C.joint_logits(torch.zeros(1, 2, D, device="cuda"), torch.zeros(1, 2, D, device="cuda"),
                       torch.zeros(5, D, device="cuda"), torch.zeros(5, device="cuda"))
