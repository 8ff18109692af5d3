"""The fused joint + RNN-T loss (`functional.fused_joint_rnnt_loss`, reduction='none') held to an fp64 restatement per
utterance, at the shapes and values where its kernels branch:

  * u-splits: the tensor-core backward cuts an utterance's W = U_b + 1 label columns into S = ceil(W / P) slabs of a
    P x TT tile (21 x 6 or 16 x 8); d_enc is the sum of S partial slabs.  The table reaches S = 8 and S >= 5 with both
    geometries, every W mod 4 (the forward's 4 / 2 / 1-column groups) and both backward kernels (CTA pair when
    D % 256 == 0, single CTA otherwise; the D = 256 / 512 cases run the single-CTA kernel a second time);
  * frame edges: the forward's 32 / 64 / 128-frame blocks at +-1, odd frame-block counts (the pair backward pads them);
  * vocabularies: V padded to a multiple of 32, blank in each of the three warp groups that patch its exact gradient,
    targets equal to blank;
  * a cotangent that differs per utterance in sign and size (0, negative, 0.1 .. 3), with and without a clamp;
  * fp32 beyond the tensor-core limits;
  * out-of-range labels and lengths (negative ones included), which the op clamps.

Every utterance's cost and its d_enc / d_pred rows are compared on their own, so one bad utterance cannot hide in a
batch average.  The CPU tests check the checker itself (planted faults are caught), the coverage of the case table
through a mirror of the tile selection, and the shape predicate of the tensor-core path."""
import contextlib
import math

import numpy as np
import pytest
import torch

from oracle import transducer_oracle as TO

F32_TOL = 1e-4                       # precision 'fp32' and 'bf16x3': cost and gradients within 1e-4 of the reference
BF16_COST, BF16_GRAD = 2e-3, 3e-2    # precision 'bf16' (functional.fused_joint_rnnt_loss docstring) ...
BF16_COST_STEP = 1e-3                # ... or 1e-3 nats per lattice step (T_b + U_b) of a cost, where that is larger
COLUMNS = ("fp32", "bf16x3", "bf16", "bf16in")     # bf16in: precision 'bf16' on bf16 activations (bf16 gradients)
GRADS = ("d_enc", "d_pred")
SHARED = ("d_w", "d_b")


# ---------------------------------------------------------------------------------------------------------- case table
def _case(name, B, T, U1, D, V, blank, tl, ul, gc, clamps=(-1.0,), blank_targets=(), seed=0):
    return dict(name=name, B=B, T=T, U1=U1, D=D, V=V, blank=blank, tl=list(tl), ul=list(ul), gc=list(gc),
                clamps=tuple(clamps), blank_targets=tuple(blank_targets), seed=seed)


BITE = 0.05                          # a clamp that bites: |d cost / d logit| reaches 1 on the blank / label entries

TC_CASES = [
    # 16 x 8 geometry (40 tiles against 49), S = 8, 8, 7, 4, 1 and W mod 4 = 0, 2, 3, 2, 1; D = 512: CTA-pair backward
    _case("usplit16x8", 5, 40, 128, 512, 416, 0, tl=(40, 33, 17, 8, 1), ul=(127, 113, 98, 61, 0),
          gc=(1.7, -0.6, 3.0, 0.25, 0.0), clamps=(-1.0, BITE), seed=1),
    # 21 x 6 geometry (60 tiles against 64), S = 6, 5, 4, 3, 1; D = 384: single-CTA backward; V = 385 is padded to 416
    # and blank is its last column
    _case("usplit21x6", 5, 60, 126, 384, 385, 384, tl=(60, 47, 31, 60, 12), ul=(125, 104, 83, 42, 7),
          gc=(-0.6, 1.7, 0.25, 3.0, 0.0), clamps=(-1.0, BITE), seed=2),
    # forward 128 / 64 / 32-frame blocks at +-1 (W = 9, 8, 7, 6, 4, 3, 2 covers the 4-, 2- and 1-column groups); 16 x 8
    # geometry with odd frame-block counts (33, 17, 9, 5) that the pair backward (D = 256) pads to even
    _case("frames", 7, 257, 9, 256, 33, 16, tl=(257, 256, 129, 128, 65, 33, 31), ul=(8, 7, 6, 5, 3, 2, 1),
          gc=(1.7, -0.6, 0.25, 3.0, -0.1, 0.8, 0.0), seed=3),
    # 21 x 6 geometry (22 tiles against 24) with 11, 10, 2, 1, 1 frame blocks: the pair backward (D = 512) pads the odd
    # sweeps with a tile beyond T_b
    _case("oddblocks21x6", 5, 61, 41, 512, 412, 5, tl=(61, 55, 7, 6, 1), ul=(40, 21, 20, 33, 0),
          gc=(1.7, -0.6, 0.0, 3.0, 0.25), seed=4),
]

# padding columns of V, and blank in each of the three warp groups ((blank >> 4) % 3) that patch its exact entry
VOCABS = [(2, 0), (2, 1), (31, 30), (33, 16), (416, 0), (416, 415), (416, 208), (416, 224)]
VOCAB_CASES = [_case(f"vocab{V}_blank{blank}", 3, 13, 7, 128, V, blank, tl=(13, 9, 4), ul=(6, 4, 2), gc=(1.7, -0.6, 0.0),
                     clamps=(-1.0, BITE), blank_targets=((0, 0), (1, 2)), seed=10 + i)
               for i, (V, blank) in enumerate(VOCABS)]

# U + 1 = 200 and D = 100 are outside the tensor-core tiling: fp32 only, and the tensor-core precisions refuse the shape
F32_ONLY = _case("fp32only", 3, 30, 200, 100, 50, 3, tl=(30, 17, 5), ul=(199, 120, 3), gc=(-0.6, 1.7, 0.0), seed=20)

# out-of-range values: lengths above the extents, zero and negative (u_len = -100 <= -2P), labels >= V, < 0 and == blank
BAD = _case("badvalues", 8, 12, 8, 128, 40, 3, tl=(12, 20, 0, -5, 7, 12, 9, 12), ul=(7, 11, -1, 3, -100, -17, 5, 2),
            gc=(1.7, -0.6, 0.25, 3.0, -2.2, 0.8, 0.0, 1.1), seed=30)
BAD_LABELS = {(0, 1): 10 ** 6, (0, 3): -7, (1, 0): 3, (6, 2): 40, (7, 0): -1}        # (b, u) -> label


# ------------------------------------------------------------------- mirror of the C++ tile selection (csrc/joint_tc.cu)
# These restate pick_rect_geom, the u-split count of build_tiles_block and joint_tc_bwd_supported for the coverage check
# below.  They must change when the C++ selection does.
def pad_v(V):
    return (V + 31) // 32 * 32


def tc_shape(U1, D, V):
    return D % 128 == 0 and 128 <= D <= 512 and pad_v(V) <= 416 and U1 <= 128


def rect_geom(T, U1):
    tiles = lambda P, TT: -(-U1 // P) * -(-T // TT)
    return (21, 6) if tiles(21, 6) < tiles(16, 8) else (16, 8)


def clamped_lengths(c):
    """The op's contract for lengths: clamped to [0, T] and [0, U]."""
    tl = [min(max(t, 0), c["T"]) for t in c["tl"]]
    ul = [min(max(u, 0), c["U1"] - 1) for u in c["ul"]]
    return tl, ul


def u_splits(u_len, P):
    return -(-(u_len + 1) // P)


# ----------------------------------------------------------------------------------------------------------- inputs
def make_inputs(c):
    g = torch.Generator().manual_seed(1000 + c["seed"])
    B, T, U1, D, V = c["B"], c["T"], c["U1"], c["D"], c["V"]
    enc = 0.5 * torch.randn(B, T, D, generator=g)
    pred = 0.5 * torch.randn(B, U1, D, generator=g)
    w = torch.randn(V, D, generator=g) / math.sqrt(D)
    b = 0.1 * torch.randn(V, generator=g)
    tgt = torch.randint(0, V, (B, U1 - 1), generator=g, dtype=torch.int32)
    for (i, u) in c["blank_targets"]:
        tgt[i, u] = c["blank"]
    return enc, pred, w, b, tgt


def oracle(enc, pred, w, b, tgt, tl, ul, blank, clamp, gc, dtype=torch.float64):
    """fp64 restatement of the op on valid inputs: identity pre-projections make enc / pred the joint's inputs."""
    D = enc.shape[-1]
    eye, zero = torch.eye(D), torch.zeros(D)
    ws = {"enc_ffn.weight": eye, "enc_ffn.bias": zero, "pred_ffn.weight": eye, "pred_ffn.bias": zero,
          "ffn_out.weight": w, "ffn_out.bias": b}
    r = TO.fused_joint_rnnt_restated(enc, pred, ws, tgt, torch.tensor(tl), torch.tensor(ul), blank, clamp, dtype,
                                     grad_costs=torch.tensor(gc, dtype=torch.float64))
    return dict(costs=r["costs"].double(), d_enc=r["d_enc_out"].double(), d_pred=r["d_pred_out"].double(),
                d_w=r["d_ffn_out.weight"].double(), d_b=r["d_ffn_out.bias"].double())


def rel_l2(a, b):
    return float((a - b).norm() / max(float(b.norm()), 1e-300))


def check(got, ref, tl, ul, gc, cost_tol, cost_step, grad_tol, shared_tol):
    """Per-utterance comparison.  Returns (failures, worst errors).  tl / ul are the clamped lengths; a cost may be off
    by max(cost_tol x |cost|, cost_step x (T_b + U_b)); `grad_tol` is one
    bar or one per (utterance, d_enc / d_pred); `shared_tol` maps d_w / d_b to their bars.  Beyond its lengths, and for
    a zero cotangent or no frames, an utterance's gradients must be exact zeros; a cost without frames is exactly 0.
    `worst` also holds the largest error / bar ratio of the gradients ("use")."""
    fails, worst = [], {k: 0.0 for k in ("cost",) + GRADS + SHARED + ("use",)}
    grad_tol = np.broadcast_to(np.asarray(grad_tol, dtype=np.float64), (len(gc), len(GRADS)))
    for k in ("costs",) + GRADS + SHARED:
        if not bool(torch.isfinite(got[k]).all()):
            fails.append(f"{k}: not finite")
    for b in range(len(gc)):
        Tb, Ub = tl[b], ul[b]
        c, r = float(got["costs"][b]), float(ref["costs"][b])
        if Tb == 0:
            if c != 0.0:
                fails.append(f"b={b}: cost {c} without frames")
        else:
            e, tol = abs(c - r) / abs(r), max(cost_tol, cost_step * (Tb + Ub) / abs(r))
            worst["cost"] = max(worst["cost"], e)
            if not e <= tol:
                fails.append(f"b={b}: cost {c} against {r} (rel {e:.2e} > {tol:.1e})")
        if bool((got["d_enc"][b, Tb:] != 0).any()) or bool((got["d_pred"][b, Ub + 1:] != 0).any()):
            fails.append(f"b={b}: nonzero gradient beyond T_b = {Tb} / U_b = {Ub}")
        if gc[b] == 0 or Tb == 0:
            if bool((got["d_enc"][b] != 0).any()) or bool((got["d_pred"][b] != 0).any()):
                fails.append(f"b={b}: nonzero gradient for cotangent {gc[b]} / T_b = {Tb}")
            continue
        for i, k in enumerate(GRADS):
            e = rel_l2(got[k][b], ref[k][b])
            worst[k] = max(worst[k], e)
            worst["use"] = max(worst["use"], e / grad_tol[b, i])
            if not e <= grad_tol[b, i]:
                fails.append(f"b={b}: {k} rel-L2 {e:.2e} > {grad_tol[b, i]:.1e}")
    for k in SHARED:
        e = rel_l2(got[k], ref[k])
        worst[k] = e
        worst["use"] = max(worst["use"], e / shared_tol[k])
        if not e <= shared_tol[k]:
            fails.append(f"{k} rel-L2 {e:.2e} > {shared_tol[k]:.1e}")
    return fails, worst


def bars(col, ref64, ref32, tl):
    """(cost, cost per lattice step, per-utterance gradient, {d_w, d_b}) bars of a column, for check().

    fp32 / bf16x3 promise 1e-4 of the reference, which computes in fp32 itself.  Against fp64 that is 1e-4 plus the
    reference's own rounding, estimated by the fp32 restatement's error (times 2: one sample of fp32 noise), per
    utterance for d_enc / d_pred.  The rounding is not small: the lattice adds log-probabilities up to twice the cost,
    and at a cost of ~800 nats an fp32 restatement is 2e-4 off on its own.

    bf16 promises 2e-3 on a cost, or 1e-3 nats per lattice step where that is larger (costs under ~0.5 nats a step,
    as with V = 2), and 3e-2 on every gradient."""
    if col in ("fp32", "bf16x3"):
        grad = np.full((len(tl), len(GRADS)), F32_TOL)
        for b, Tb in enumerate(tl):
            if Tb > 0 and float(ref64["d_enc"][b].norm()) > 0:
                grad[b] += [2.0 * rel_l2(ref32[k][b], ref64[k][b]) for k in GRADS]
        return F32_TOL, 0.0, grad, {k: F32_TOL + 2.0 * rel_l2(ref32[k], ref64[k]) for k in SHARED}
    return BF16_COST, BF16_COST_STEP, BF16_GRAD, {k: BF16_GRAD for k in SHARED}


# ------------------------------------------------------------------------------------------------------------- CPU
def test_checker_rejects_planted_faults():
    """The per-utterance checker at the bf16 bars accepts the truth and rejects three faults a batch-wide comparison can
    dilute: one utterance's gradients scaled by its neighbour's cotangent, one lost 6-frame backward tile of d_enc, and
    one cost off by 0.3 %."""
    torch.manual_seed(5)
    B, T, U1, D, V, blank = 4, 17, 6, 32, 20, 2
    enc, pred = 0.5 * torch.randn(B, T, D), 0.5 * torch.randn(B, U1, D)
    w, b = torch.randn(V, D) / math.sqrt(D), 0.1 * torch.randn(V)
    tgt = torch.randint(0, V, (B, U1 - 1), dtype=torch.int32)
    tl, ul, gc = [17, 12, 17, 9], [5, 3, 4, 0], [1.7, -0.6, 0.25, 3.0]
    ref = oracle(enc, pred, w, b, tgt, tl, ul, blank, -1.0, gc)
    tol = bars("bf16", ref, None, tl)
    fails, _ = check(ref, ref, tl, ul, gc, *tol)
    assert fails == []

    def planted(edit):
        got = {k: v.clone() for k, v in ref.items()}
        edit(got)
        return check(got, ref, tl, ul, gc, *tol)[0]

    def neighbour(got):
        for k in GRADS:
            got[k][2] *= gc[3] / gc[2]

    def lost_tile(got):
        got["d_enc"][0, 6:12] = 0

    def cost(got):
        got["costs"][1] *= 1.003

    for edit, what in ((neighbour, "b=2: d_enc"), (lost_tile, "b=0: d_enc"), (cost, "b=1: cost")):
        fails = planted(edit)
        assert any(f.startswith(what) for f in fails), (what, fails)


def test_oracle_grad_costs_and_empty_utterance():
    """grad_costs=None is the mean; a cotangent scales each utterance's gradient after the clamp; an utterance without
    frames has cost 0 and no gradient."""
    torch.manual_seed(6)
    B, T, U1, D, V, blank = 3, 7, 4, 16, 11, 1
    enc, pred = torch.randn(B, T, D), torch.randn(B, U1, D)
    w = {"enc_ffn.weight": torch.randn(D, D) / 4, "enc_ffn.bias": torch.zeros(D), "pred_ffn.weight": torch.randn(D, D) / 4,
         "pred_ffn.bias": torch.zeros(D), "ffn_out.weight": torch.randn(V, D) / 4, "ffn_out.bias": torch.zeros(V)}
    tgt = torch.randint(0, V, (B, U1 - 1), dtype=torch.int32)
    tl, ul = torch.tensor([7, 0, 5]), torch.tensor([3, 2, 1])
    for clamp in (-1.0, 0.02):
        mean = TO.fused_joint_rnnt_restated(enc, pred, w, tgt, tl, ul, blank, clamp)
        same = TO.fused_joint_rnnt_restated(enc, pred, w, tgt, tl, ul, blank, clamp, grad_costs=torch.full((B,), 1 / B, dtype=torch.float64))
        assert torch.allclose(mean["d_enc_out"], same["d_enc_out"], rtol=1e-12, atol=1e-15)
        gc = torch.tensor([2.0, 5.0, -0.5])
        r = TO.fused_joint_rnnt_restated(enc, pred, w, tgt, tl, ul, blank, clamp, grad_costs=gc)
        assert float(r["costs"][1]) == 0.0 and bool((r["d_enc_out"][1] == 0).all())
        for b in (0, 2):
            assert torch.allclose(r["d_enc_out"][b], mean["d_enc_out"][b] * gc[b] * B, rtol=1e-10, atol=1e-14)


def test_case_table_reaches_the_tiling_branches():
    """Through the mirror of the C++ tile selection: the tensor-core cases reach S = 8, S >= 5 in both geometries,
    every W mod 4, both backward kernels, blank in each patch warp group and frame counts on both sides of 32, 64 and
    128; every case has a zero, a negative and a large cotangent; the bad-values case passes u_len <= -2P."""
    geoms_s5, svals, wmod, bwd, owners, tbs = set(), set(), set(), set(), set(), set()
    for c in TC_CASES + VOCAB_CASES:
        assert tc_shape(c["U1"], c["D"], c["V"]), c["name"]
        P, _ = rect_geom(c["T"], c["U1"])
        tl, ul = clamped_lengths(c)
        for t, u in zip(tl, ul):
            s = u_splits(u, P)
            svals.add(s)
            if s >= 5:
                geoms_s5.add(P)
            wmod.add((u + 1) % 4)
            tbs.add(t)
        bwd.add("pair" if c["D"] % 256 == 0 else "single")
        owners.add((c["blank"] >> 4) % 3)
    assert geoms_s5 == {16, 21} and 8 in svals and wmod == {0, 1, 2, 3} and bwd == {"pair", "single"}
    assert owners == {0, 1, 2}
    assert any(c["V"] != pad_v(c["V"]) for c in VOCAB_CASES) and any(c["V"] < 32 for c in VOCAB_CASES)
    for edge in (32, 64, 128):
        assert any(t <= edge for t in tbs) and any(t > edge for t in tbs), edge
    for c in TC_CASES + VOCAB_CASES + [F32_ONLY, BAD]:
        assert len(c["tl"]) == len(c["ul"]) == len(c["gc"]) == c["B"], c["name"]
        assert 0.0 in c["gc"] and min(c["gc"]) < 0 and max(abs(g) for g in c["gc"]) >= 1.7, c["name"]
    assert not tc_shape(F32_ONLY["U1"], F32_ONLY["D"], F32_ONLY["V"])
    P, _ = rect_geom(BAD["T"], BAD["U1"])
    assert min(BAD["ul"]) <= -2 * P and min(BAD["tl"]) < 0 and 0 in BAD["tl"] and max(BAD["tl"]) > BAD["T"]
    assert max(BAD["ul"]) > BAD["U1"] - 1
    assert {BAD["blank"], -1, BAD["V"]} <= set(BAD_LABELS.values())


def test_tensor_core_shape_predicate_boundaries():
    from ctcvr_b200._lib import query
    for (U1, D, V), want in (((128, 512, 416), 1), ((128, 384, 385), 1), ((129, 512, 416), 0), ((128, 512, 417), 0),
                             ((128, 448, 416), 0), ((128, 640, 416), 0)):
        assert query("ctcvr_joint_tc_supported", U1, D, V) == want, (U1, D, V)
        assert tc_shape(U1, D, V) == bool(want), (U1, D, V)


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def C():
    import ctcvr_b200
    assert torch.cuda.is_available()
    ctcvr_b200._lib.lib()
    return ctcvr_b200


@contextlib.contextmanager
def single_cta_backward(C):
    """ctcvr_debug_set_mode(3): the bf16 backward runs its single-CTA kernel; mode 1 (the default) is restored."""
    C._lib.lib().ctcvr_debug_set_mode(3)
    try:
        yield
    finally:
        C._lib.lib().ctcvr_debug_set_mode(1)


def run_column(C, col, enc, pred, w, b, tgt, tl, ul, blank, clamp, gc):
    dt = torch.bfloat16 if col == "bf16in" else torch.float32
    e = enc.to("cuda", dt).requires_grad_(True)
    p = pred.to("cuda", dt).requires_grad_(True)
    wo, bo = w.cuda().requires_grad_(True), b.cuda().requires_grad_(True)
    i32 = lambda x: torch.as_tensor(x, dtype=torch.int32).cuda()
    costs = C.functional.fused_joint_rnnt_loss(e, p, wo, bo, i32(tgt), i32(tl), i32(ul), blank, clamp=clamp,
                                               reduction="none", precision="bf16" if col == "bf16in" else col)
    costs.backward(torch.tensor(gc, dtype=torch.float32, device="cuda"))
    torch.cuda.synchronize()
    flag = C._lib.lib().ctcvr_debug_tc_error()
    assert flag == 0, f"{col}: tcgen05 kernel hit a bounded mbarrier wait: 0x{flag:08x}"
    if col == "bf16in":
        assert e.grad.dtype == torch.bfloat16 and p.grad.dtype == torch.bfloat16
    return dict(costs=costs.detach().double().cpu(), d_enc=e.grad.double().cpu(), d_pred=p.grad.double().cpu(),
                d_w=wo.grad.double().cpu(), d_b=bo.grad.double().cpu())


def run_case(C, c, columns=COLUMNS):
    """Every column and clamp of case c against the fp64 oracle (computed once per clamp and input rounding).  The D = 256
    and 512 cases run the bf16 columns again with the single-CTA backward.  All failures are gathered before asserting."""
    enc, pred, w, b, tgt = make_inputs(c)
    tl, ul = clamped_lengths(c)
    blank, gc, fails = c["blank"], c["gc"], []
    enc16, pred16 = enc.to(torch.bfloat16).float(), pred.to(torch.bfloat16).float()
    for clamp in c["clamps"]:
        ref64 = oracle(enc, pred, w, b, tgt, tl, ul, blank, clamp, gc)
        ref32 = oracle(enc, pred, w, b, tgt, tl, ul, blank, clamp, gc, torch.float32)
        ref16 = oracle(enc16, pred16, w, b, tgt, tl, ul, blank, clamp, gc) if "bf16in" in columns else None
        runs = [(col, False) for col in columns]
        if c["D"] % 256 == 0:
            runs += [(col, True) for col in columns if col in ("bf16", "bf16in")]
        for col, single in runs:
            with single_cta_backward(C) if single else contextlib.nullcontext():
                got = run_column(C, col, enc, pred, w, b, tgt, tl, ul, blank, clamp, gc)
            ref = ref16 if col == "bf16in" else ref64
            f, worst = check(got, ref, tl, ul, gc, *bars(col, ref64, ref32, tl))
            tag = f"{c['name']} clamp={clamp} {col}{' single-CTA bwd' if single else ''}"
            print(f"EDGE {tag}: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
            fails += [f"{tag}: {m}" for m in f]
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("c", TC_CASES, ids=[c["name"] for c in TC_CASES])
def test_tiling_edges_vs_fp64(C, c):
    run_case(C, c)


@pytest.mark.gpu
@pytest.mark.parametrize("c", VOCAB_CASES, ids=[c["name"] for c in VOCAB_CASES])
def test_vocabulary_edges_vs_fp64(C, c):
    run_case(C, c)


@pytest.mark.gpu
def test_fp32_beyond_tensor_core_limits_vs_fp64(C):
    run_case(C, F32_ONLY, columns=("fp32",))
    enc, pred, w, b, tgt = make_inputs(F32_ONLY)
    for col in ("bf16x3", "bf16", "bf16in"):
        with pytest.raises(RuntimeError, match="needs"):
            run_column(C, col, enc, pred, w, b, tgt, F32_ONLY["tl"], F32_ONLY["ul"], F32_ONLY["blank"], -1.0,
                       F32_ONLY["gc"])


@pytest.mark.gpu
def test_bad_lengths_and_labels_act_as_clamped(C):
    """Lengths outside [0, extent] and labels outside [0, V) give what their clamped values give (lengths clamped to the
    extents, such labels read as blank): costs bit for bit, gradients up to the order of the fp32 atomics; and both
    agree with the fp64 oracle on the clamped inputs."""
    c = BAD
    enc, pred, w, b, tgt = make_inputs(c)
    tgt_bad = tgt.clone()
    for (i, u), lab in BAD_LABELS.items():
        tgt_bad[i, u] = lab
    tgt_ok = torch.where((tgt_bad >= 0) & (tgt_bad < c["V"]), tgt_bad, torch.full_like(tgt_bad, c["blank"]))
    tl, ul = clamped_lengths(c)
    blank, gc, fails = c["blank"], c["gc"], []
    enc16, pred16 = enc.to(torch.bfloat16).float(), pred.to(torch.bfloat16).float()
    ref64 = oracle(enc, pred, w, b, tgt_ok, tl, ul, blank, -1.0, gc)
    ref32 = oracle(enc, pred, w, b, tgt_ok, tl, ul, blank, -1.0, gc, torch.float32)
    ref16 = oracle(enc16, pred16, w, b, tgt_ok, tl, ul, blank, -1.0, gc)
    for col in COLUMNS:
        bad = run_column(C, col, enc, pred, w, b, tgt_bad, c["tl"], c["ul"], blank, -1.0, gc)
        ok = run_column(C, col, enc, pred, w, b, tgt_ok, tl, ul, blank, -1.0, gc)
        if not torch.equal(bad["costs"], ok["costs"]):
            fails.append(f"{col}: costs {bad['costs'].tolist()} against clamped {ok['costs'].tolist()}")
        for k in GRADS + SHARED:
            if not rel_l2(bad[k], ok[k]) <= 1e-6:
                fails.append(f"{col}: {k} rel-L2 {rel_l2(bad[k], ok[k]):.2e} from the clamped run")
        f, worst = check(bad, ref16 if col == "bf16in" else ref64, tl, ul, gc, *bars(col, ref64, ref32, tl))
        print(f"EDGE badvalues {col}: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
        fails += [f"{col}: {m}" for m in f]
    assert not fails, "\n".join(fails)
