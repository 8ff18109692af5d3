"""The fused joint + RNN-T loss on the tensor cores for vocabularies beyond 416 entries (`vocab_tiling=True`, the
`ctcvr_joint_rnnt_*_vt` entry points), held to an fp64 restatement per utterance.

The vocabulary is cut into n = ceil(pad32(V) / 416) tiles of Vc = pad32(ceil(V / n)) columns, each run through the
kernels of the untiled path, with the log-sum-exp merged over the tiles.  The cases put the blank at column 0, at the
first and last column of an inner tile and at V - 1, give the last tile 1 - 16 real columns in its final 32-column
group, hold labels in every tile, and run both backward kernels (CTA pair at D % 256 == 0, single CTA at D = 384) and
both backward tile geometries (21 x 6, 16 x 8).  Every precision x activation column runs with the clamp off and biting
and with a cotangent that differs per utterance in sign and size.  The bars are those of tests/test_joint_edges.py."""
import math
import types

import numpy as np
import pytest
import torch

from oracle import align_oracle as AO
from test_joint_activations import ACTS, joint_weights, restated
from test_joint_edges import BF16_COST, BF16_COST_STEP, BITE, F32_TOL, GRADS, SHARED, bars, check, rel_l2

TILE_MAX = 416                       # the widest vocabulary of the untiled tensor-core kernels
V_CAP = 32768                        # ctcvr_joint_tc_vt_supported


# ------------------------------------------------------------------- mirror of the C++ tile rule (csrc/joint_tc.cu)
def pad_v(V):
    return (V + 31) // 32 * 32


def vocab_tiles(V):
    """[(v0, real columns)] of the tiles of a vocabulary of V entries, each Vc = pad32(ceil(V / n)) wide."""
    n = -(-pad_v(V) // TILE_MAX)
    Vc = pad_v(-(-V // n))
    return Vc, [(c * Vc, min(V - c * Vc, Vc)) for c in range(n)]


def vt_shape(U1, D, V):
    return D % 128 == 0 and 128 <= D <= 512 and 1 <= U1 <= 128 and 1 <= V <= V_CAP


# ----------------------------------------------------------------------------------------------------------- cases
def _case(name, B, T, U1, D, V, blank, tl, ul, gc, seed, blank_targets=((0, 0),)):
    return dict(name=name, B=B, T=T, U1=U1, D=D, V=V, blank=blank, tl=list(tl), ul=list(ul), gc=list(gc), seed=seed,
                blank_targets=blank_targets)


CASES = [
    # the smallest tiled vocabulary: two tiles of 224 columns (224 + 193 real); blank at column 0; D = 512: CTA-pair
    # backward; 16 x 8 geometry
    _case("v417_d512_blank0", 4, 33, 10, 512, 417, 0, tl=(33, 20, 9, 1), ul=(9, 6, 3, 0), gc=(1.7, -0.6, 3.0, 0.0),
          seed=1),
    # three tiles of 352 (the last with 296 real: 8 in its final 32-group); blank at the first column of the inner tile;
    # D = 384: single-CTA backward; 21 x 6 geometry
    _case("v1000_d384_blank352", 3, 24, 21, 384, 1000, 352, tl=(24, 17, 7), ul=(20, 13, 4), gc=(-0.6, 1.7, 0.25),
          seed=2),
    # the same tiles with blank at the last column of the inner tile; D = 512: CTA-pair backward; 21 x 6 geometry
    _case("v1000_d512_blank703", 3, 24, 21, 512, 1000, 703, tl=(24, 11, 19), ul=(20, 20, 9), gc=(3.0, 0.0, -0.6),
          seed=3),
    # exactly two full tiles of 416; blank at V - 1; D = 256: CTA-pair backward; 16 x 8 geometry
    _case("v832_d256_blank831", 3, 40, 9, 256, 832, 831, tl=(40, 29, 8), ul=(8, 5, 7), gc=(0.25, 3.0, -0.6), seed=4),
]
# (precision, activation, inputs rounded to bf16): bf16 relu runs on bf16-valued inputs, where rounding the inputs
# cannot flip the side of the kink (functional.fused_joint_rnnt_loss docstring)
COLUMNS = [("bf16x3", "tanh", False), ("bf16x3", "relu", False), ("bf16x3", "gelu", False),
           ("bf16", "tanh", False), ("bf16", "gelu", False), ("bf16", "relu", True)]

# out-of-range values at a tiled V: lengths above the extents, zero and negative; labels >= V, < 0 and == blank
BAD = _case("badvalues", 6, 12, 8, 128, 1000, 700, tl=(12, 20, 0, -5, 7, 12), ul=(7, 11, -1, 3, -100, 5),
            gc=(1.7, -0.6, 0.25, 3.0, -2.2, 0.8), seed=30)
BAD_LABELS = {(0, 1): 10 ** 6, (0, 3): -7, (1, 0): 700, (5, 2): 1000, (5, 0): -1}        # (b, u) -> label


def make_inputs(c, rounded=False):
    g = torch.Generator().manual_seed(2000 + c["seed"])
    B, T, U1, D, V = c["B"], c["T"], c["U1"], c["D"], c["V"]
    enc = 0.5 * torch.randn(B, T, D, generator=g)
    pred = 0.5 * torch.randn(B, U1, D, generator=g)
    w = torch.randn(V, D, generator=g) / math.sqrt(D)
    b = 0.1 * torch.randn(V, generator=g)
    tgt = torch.randint(0, V, (B, U1 - 1), generator=g, dtype=torch.int32)
    # labels in every tile of the vocabulary (utterance 0 walks through them), and targets equal to blank
    _, tiles = vocab_tiles(V)
    for k, (v0, n) in enumerate(tiles):
        if k + 1 < U1:
            tgt[0, k] = v0 + (k * 37) % n
    for (i, u) in c["blank_targets"]:
        if u + len(tiles) < U1 - 1:
            tgt[i, u + len(tiles)] = c["blank"]
    if rounded:
        enc, pred = enc.bfloat16().float(), pred.bfloat16().float()
    return enc, pred, w, b, tgt


def clamped_lengths(c):
    return [min(max(t, 0), c["T"]) for t in c["tl"]], [min(max(u, 0), c["U1"] - 1) for u in c["ul"]]


def oracle(enc, pred, w, b, tgt, tl, ul, blank, clamp, gc, act, dtype=torch.float64):
    D = enc.shape[-1]
    eye, zero = torch.eye(D, dtype=dtype), torch.zeros(D, dtype=dtype)
    ws = {"enc_ffn.weight": eye, "enc_ffn.bias": zero, "pred_ffn.weight": eye, "pred_ffn.bias": zero,
          "ffn_out.weight": w.to(dtype), "ffn_out.bias": b.to(dtype)}
    r = restated(enc, pred, ws, tgt, tl, ul, blank, clamp, gc, act, dtype)
    return dict(costs=r["costs"].double(), d_enc=r["d_enc"].double(), d_pred=r["d_pred"].double(),
                d_w=r["d_ffn_out.weight"].double(), d_b=r["d_ffn_out.bias"].double())


def log_probs64(enc, pred, w, b, tgt, blank, act):
    """fp64 lse / lp_blank / lp_label [B,T,U1] of every cell (lp_label of the last column: -inf)."""
    z = ACTS[act](enc.double()[:, :, None] + pred.double()[:, None])
    logits = z @ w.double().t() + b.double()
    lse = torch.logsumexp(logits, -1)
    lab = torch.where((tgt >= 0) & (tgt < w.shape[0]), tgt, torch.full_like(tgt, blank)).long()
    lpb = logits[..., blank] - lse
    lpl = torch.full_like(lse, -math.inf)
    lpl[:, :, :-1] = logits[:, :, :-1].gather(-1, lab[:, None, :, None].expand(-1, lse.shape[1], -1, 1))[..., 0] - \
        lse[:, :, :-1]
    return lse, lpb, lpl


# ------------------------------------------------------------------------------------------------------------- CPU
def test_tile_rule_and_case_coverage():
    """The tile rule gives tiles of at most 416 columns, multiples of 32, covering [0, V) with a non-empty last tile,
    for every V the entry points take; the case table reaches its edges."""
    for V in range(TILE_MAX + 1, V_CAP + 1):
        Vc, tiles = vocab_tiles(V)
        assert Vc <= TILE_MAX and Vc % 32 == 0, V
        assert all(v0 == k * Vc for k, (v0, _) in enumerate(tiles)), V
        assert all(n == Vc for _, n in tiles[:-1]) and 1 <= tiles[-1][1] <= Vc, V
        assert sum(n for _, n in tiles) == V, V
    assert vocab_tiles(417) == (224, [(0, 224), (224, 193)])
    assert vocab_tiles(832) == (416, [(0, 416), (416, 416)])
    assert len(vocab_tiles(V_CAP)[1]) == 79
    Vs = {c["V"] for c in CASES}
    assert {417, 832} <= Vs
    # the last tile has 1 - 16 real columns in its final 32-column group
    assert any(1 <= vocab_tiles(V)[1][-1][1] % 32 <= 16 for V in Vs)
    # blank at column 0, at the first and the last column of an inner tile, and at V - 1
    pos = set()
    for c in CASES:
        Vc, tiles = vocab_tiles(c["V"])
        k, col = divmod(c["blank"], Vc)
        pos.add("zero" if c["blank"] == 0 else "last" if c["blank"] == c["V"] - 1 else
                ("inner-first" if col == 0 else "inner-last" if col == Vc - 1 else "other") if 0 < k < len(tiles) - 1
                else "other")
    assert {"zero", "inner-first", "inner-last", "last"} <= pos, pos
    # labels in every tile, both backward kernels and both tile geometries
    for c in CASES:
        _, _, _, _, tgt = make_inputs(c)
        _, tiles = vocab_tiles(c["V"])
        assert all(bool(((tgt >= v0) & (tgt < v0 + n)).any()) for v0, n in tiles), c["name"]
    assert {c["D"] % 256 == 0 for c in CASES} == {True, False}
    geoms = {("21x6" if -(-c["U1"] // 21) * -(-c["T"] // 6) < -(-c["U1"] // 16) * -(-c["T"] // 8) else "16x8")
             for c in CASES}
    assert geoms == {"21x6", "16x8"}


def test_vt_shape_predicate_boundaries():
    from ctcvr_b200._lib import query
    for (U1, D, V), want in (((128, 512, V_CAP), 1), ((128, 512, V_CAP + 1), 0), ((128, 448, 1000), 0),
                             ((128, 640, 1000), 0), ((129, 512, 1000), 0), ((128, 384, 417), 1), ((1, 128, 1), 1),
                             ((128, 256, 0), 0)):
        assert query("ctcvr_joint_tc_vt_supported", U1, D, V) == want, (U1, D, V)
        assert vt_shape(U1, D, V) == bool(want), (U1, D, V)
    # the untiled predicate keeps its answer
    assert query("ctcvr_joint_tc_supported", 128, 512, 417) == 0
    assert query("ctcvr_joint_tc_supported", 128, 512, 416) == 1


def test_vt_ws_bytes_finite_and_independent_of_activation_bits():
    from ctcvr_b200._lib import query
    for q, plain in (("ctcvr_joint_rnnt_fwd_vt_ws_bytes", "ctcvr_joint_rnnt_fwd_ws_bytes"),
                     ("ctcvr_joint_rnnt_bwd_vt_ws_bytes", "ctcvr_joint_rnnt_bwd_ws_bytes")):
        for prec in (1, 2):
            for V in (100, 416, 417, 4096, V_CAP):
                base = query(q, 32, 250, 41, 512, V, prec)
                assert 256 < base < (1 << 40), (q, V, prec, base)
                for act in (0x100, 0x200):
                    assert query(q, 32, 250, 41, 512, V, prec | act) == base
            # one tile: the untiled entry point's workspace
            assert query(q, 4, 50, 11, 256, 300, prec) == query(plain, 4, 50, 11, 256, 300, prec)
        assert query(q, 4, 50, 11, 256, 1000, 2) > query(q, 4, 50, 11, 256, 1000, 1)


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def C():
    import ctcvr_b200
    assert torch.cuda.is_available()
    ctcvr_b200._lib.lib()
    return ctcvr_b200


def _tc_ok(C, what):
    torch.cuda.synchronize()
    flag = C._lib.lib().ctcvr_debug_tc_error()
    assert flag == 0, f"{what}: tcgen05 kernel hit a bounded mbarrier wait: 0x{flag:08x}"


def run(C, prec, act, enc, pred, w, b, tgt, tl, ul, blank, clamp, gc, vocab_tiling=True):
    e = enc.cuda().requires_grad_(True)
    p = pred.cuda().requires_grad_(True)
    wo, bo = w.cuda().requires_grad_(True), b.cuda().requires_grad_(True)
    i32 = lambda x: torch.as_tensor(x, dtype=torch.int32).cuda()
    costs = C.functional.fused_joint_rnnt_loss(e, p, wo, bo, i32(tgt), i32(tl), i32(ul), blank, clamp=clamp,
                                               reduction="none", precision=prec, activation=act,
                                               vocab_tiling=vocab_tiling)
    costs.backward(torch.tensor(gc, dtype=torch.float32, device="cuda"))
    _tc_ok(C, f"{prec} {act}")
    return dict(costs=costs.detach().double().cpu(), d_enc=e.grad.double().cpu(), d_pred=p.grad.double().cpu(),
                d_w=wo.grad.double().cpu(), d_b=bo.grad.double().cpu())


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[c["name"] for c in CASES])
def test_vocab_tiles_vs_fp64(C, c):
    """Every column, clamp off and biting, per utterance against the fp64 restatement, at the bars of
    tests/test_joint_edges.py.  All failures are gathered before asserting."""
    tl, ul = clamped_lengths(c)
    blank, gc, fails = c["blank"], c["gc"], []
    for clamp in (-1.0, BITE):
        for prec, act, rounded in COLUMNS:
            enc, pred, w, b, tgt = make_inputs(c, rounded)
            ref64 = oracle(enc, pred, w, b, tgt, tl, ul, blank, clamp, gc, act)
            ref32 = oracle(enc, pred, w, b, tgt, tl, ul, blank, clamp, gc, act, torch.float32) \
                if prec == "bf16x3" else None
            got = run(C, prec, act, enc, pred, w, b, tgt, tl, ul, blank, clamp, gc)
            f, worst = check(got, ref64, tl, ul, gc, *bars(prec, ref64, ref32, tl))
            tag = f"{c['name']} clamp={clamp} {prec} {act}{' bf16-valued inputs' if rounded else ''}"
            print(f"VT {tag}: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
            fails += [f"{tag}: {m}" for m in f]
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
def test_single_cta_backward_at_d512(C):
    """The D = 512 case with the bf16 backward forced onto its single-CTA kernel (ctcvr_debug_set_mode(3))."""
    c = CASES[2]
    tl, ul = clamped_lengths(c)
    enc, pred, w, b, tgt = make_inputs(c)
    ref64 = oracle(enc, pred, w, b, tgt, tl, ul, c["blank"], BITE, c["gc"], "tanh")
    C._lib.lib().ctcvr_debug_set_mode(3)
    try:
        got = run(C, "bf16", "tanh", enc, pred, w, b, tgt, tl, ul, c["blank"], BITE, c["gc"])
    finally:
        C._lib.lib().ctcvr_debug_set_mode(1)
    f, worst = check(got, ref64, tl, ul, c["gc"], *bars("bf16", ref64, None, tl))
    print("VT single-CTA bwd: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
    assert not f, f


@pytest.mark.gpu
def test_bad_lengths_and_labels_act_as_clamped(C):
    """At a tiled V, lengths outside [0, extent] and labels outside [0, V) give what their clamped values give: costs
    bit for bit, gradients up to the order of the fp32 atomics; and both agree with the fp64 oracle."""
    c = BAD
    enc, pred, w, b, tgt = make_inputs(c)
    tgt_bad = tgt.clone()
    for (i, u), lab in BAD_LABELS.items():
        tgt_bad[i, u] = lab
    tgt_ok = torch.where((tgt_bad >= 0) & (tgt_bad < c["V"]), tgt_bad, torch.full_like(tgt_bad, c["blank"]))
    tl, ul = clamped_lengths(c)
    blank, gc, fails = c["blank"], c["gc"], []
    for prec in ("bf16x3", "bf16"):
        ref64 = oracle(enc, pred, w, b, tgt_ok, tl, ul, blank, -1.0, gc, "tanh")
        ref32 = oracle(enc, pred, w, b, tgt_ok, tl, ul, blank, -1.0, gc, "tanh", torch.float32)
        bad = run(C, prec, "tanh", enc, pred, w, b, tgt_bad, c["tl"], c["ul"], blank, -1.0, gc)
        ok = run(C, prec, "tanh", enc, pred, w, b, tgt_ok, tl, ul, blank, -1.0, gc)
        if not torch.equal(bad["costs"], ok["costs"]):
            fails.append(f"{prec}: costs {bad['costs'].tolist()} against clamped {ok['costs'].tolist()}")
        for k in GRADS + SHARED:
            if not rel_l2(bad[k], ok[k]) <= 1e-6:
                fails.append(f"{prec}: {k} rel-L2 {rel_l2(bad[k], ok[k]):.2e} from the clamped run")
        f, worst = check(bad, ref64, tl, ul, gc, *bars(prec, ref64, ref32, tl))
        print(f"VT badvalues {prec}: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
        fails += [f"{prec}: {m}" for m in f]
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["bf16", "bf16x3"])
def test_small_vocabulary_is_unchanged(C, prec):
    """vocab_tiling=True at pad32(V) <= 416 runs the untiled kernels: costs and the forward's lse / lp_blank / lp_label
    bit-identical, gradients within the order of the fp32 atomics."""
    from ctcvr_b200.functional import ACT_TANH, _PREC, _joint_fwd
    c = _case("v412", 3, 30, 12, 256, 412, 5, tl=(30, 21, 9), ul=(11, 7, 4), gc=(1.7, -0.6, 0.25), seed=40)
    enc, pred, w, b, tgt = make_inputs(c)
    tl, ul = clamped_lengths(c)
    i32 = lambda x: torch.as_tensor(x, dtype=torch.int32).cuda()
    fw = [_joint_fwd(enc.cuda(), pred.cuda(), w.cuda(), b.cuda(), i32(tgt), i32(tl), i32(ul), 5, _PREC[prec], ACT_TANH,
                     vocab_tiling=vt)[2:] for vt in (False, True)]
    for x, y in zip(*fw):                              # the cells the forward writes (t < T_b, u <= U_b)
        for bi in range(c["B"]):
            assert torch.equal(x[bi, :tl[bi], :ul[bi] + 1], y[bi, :tl[bi], :ul[bi] + 1]), bi
    off = run(C, prec, "tanh", enc, pred, w, b, tgt, tl, ul, 5, -1.0, c["gc"], vocab_tiling=False)
    on = run(C, prec, "tanh", enc, pred, w, b, tgt, tl, ul, 5, -1.0, c["gc"], vocab_tiling=True)
    assert torch.equal(off["costs"], on["costs"])
    for k in GRADS + SHARED:
        assert rel_l2(on[k], off[k]) <= 1e-6, k


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["bf16", "bf16x3"])
def test_forward_log_probs_and_alignment_vs_fp64(C, prec):
    """The tiled forward's lse / lp_blank / lp_label against fp64 at V = 1000 (three tiles), and rnnt_forced_align's
    frames against the fp64 Viterbi wherever every decision margin on the oracle's path exceeds the arithmetic error."""
    from ctcvr_b200.functional import ACT_TANH, _PREC, _joint_fwd
    c = CASES[1]
    enc, pred, w, b, tgt = make_inputs(c)
    tl, ul = clamped_lengths(c)
    blank = c["blank"]
    i32 = lambda x: torch.as_tensor(x, dtype=torch.int32).cuda()
    args = (enc.cuda(), pred.cuda(), w.cuda(), b.cuda(), i32(tgt), i32(tl), i32(ul))
    _, _, lse, lpb, lpl = _joint_fwd(*args, blank, _PREC[prec], ACT_TANH, vocab_tiling=True)
    frames, tok, scores = C.functional.rnnt_forced_align(*args, blank, precision=prec, vocab_tiling=True)
    _tc_ok(C, prec)
    lse64, lpb64, lpl64 = log_probs64(enc, pred, w, b, tgt, blank, "tanh")
    tol = 2e-4 if prec == "bf16x3" else 3e-2           # absolute, in nats
    fails = []
    for bi in range(c["B"]):
        Tb, Ub = tl[bi], ul[bi]
        for name, got, ref in (("lse", lse, lse64), ("lp_blank", lpb, lpb64)):
            e = float((got[bi, :Tb, :Ub + 1].double().cpu() - ref[bi, :Tb, :Ub + 1]).abs().max())
            if not e <= tol:
                fails.append(f"b={bi} {name}: max error {e:.2e} > {tol:.0e}")
        if Ub > 0:
            e = float((lpl[bi, :Tb, :Ub].double().cpu() - lpl64[bi, :Tb, :Ub]).abs().max())
            if not e <= tol:
                fails.append(f"b={bi} lp_label: max error {e:.2e} > {tol:.0e}")
        if not bool((lpl[bi, :Tb, Ub].cpu() == -math.inf).all()):
            fails.append(f"b={bi}: lp_label of the last label column is not -inf")
        o = AO.rnnt_viterbi(lpb64[bi].numpy(), lpl64[bi].numpy(), Tb, Ub)
        bar = 2 * tol * (Tb + Ub)
        if o["margin"] > bar and not np.array_equal(frames[bi, :Ub].cpu().numpy(), o["frames"]):
            fails.append(f"b={bi}: frames {frames[bi, :Ub].tolist()} against {o['frames'].tolist()}")
        if not abs(float(scores[bi]) - o["score"]) <= tol * (Tb + Ub) + 1e-4 * abs(o["score"]):
            fails.append(f"b={bi}: score {float(scores[bi])} against {o['score']}")
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
def test_graphed_step(C):
    """GraphedJointRnntStep(..., precision='bf16', vocab_tiling=True) at V = 1000 replays to the eager result."""
    B, T, U, D, V, blank = 4, 20, 5, 256, 1000, 0
    torch.manual_seed(7)
    joint = C.TransducerJoint(V, D, D, D).cuda()
    g = torch.Generator().manual_seed(8)
    enc, pred = torch.randn(B, T, D, generator=g).cuda(), torch.randn(B, U + 1, D, generator=g).cuda()
    tgt = torch.randint(1, V, (B, U), generator=g, dtype=torch.int32).cuda()
    tl, ul = torch.tensor([20, 17, 9, 3], dtype=torch.int32).cuda(), torch.tensor([5, 2, 4, 0], dtype=torch.int32).cuda()
    step = C.GraphedJointRnntStep(joint, B, T, U, blank, precision="bf16", vocab_tiling=True)
    replays = []
    for _ in range(2):
        loss = step.step(enc, pred, tgt, tl, ul)
        torch.cuda.synchronize()
        replays.append((float(loss), {n: q.grad.clone() for n, q in step.joint.named_parameters()}, step.enc.grad.clone()))
    _tc_ok(C, "graphed step")
    e, p = enc.clone().requires_grad_(True), pred.clone().requires_grad_(True)
    for q in joint.parameters():
        q.grad = None
    eager = joint.rnnt_loss_fused(e, p, tgt, tl, ul, blank, reduction="sum", precision="bf16", vocab_tiling=True) / B
    eager.backward()
    _tc_ok(C, "eager step")
    rel = lambda a, b: float((a.double().cpu() - b.double().cpu()).norm() / max(float(b.double().norm()), 1e-30))
    for loss, grads, d_enc in replays:
        assert abs(loss - eager.item()) <= 1e-6 * abs(eager.item())
        for n, q in joint.named_parameters():
            assert rel(grads[n], q.grad) <= 1e-5, n
        assert rel(d_enc, e.grad) <= 1e-5


@pytest.mark.gpu
def test_patch_install_trains_v4096(C):
    """A reference-shaped Transducer with V = 4096 trains through patch.install(precision='bf16', vocab_tiling=True) and
    nothing else: the training seam returns the fp64 loss within the bf16 bars and every parameter gets a gradient."""
    from ctcvr_b200 import patch
    B, T, U, D, V, blank = 3, 16, 6, 256, 4096, 0
    torch.manual_seed(9)
    joint = C.TransducerJoint(V, D, D, D).cuda()
    emb = torch.nn.Embedding(V, D).cuda()

    class StubEncoder(torch.nn.Module):
        def forward(self, speech, lens, *a):
            mask = (torch.arange(speech.size(1), device=speech.device)[None, :] < lens[:, None]).unsqueeze(1)
            return speech, mask

    class Transducer(torch.nn.Module):                  # model/component/transducer.py, bodies absent on purpose
        def __init__(self):
            super().__init__()
            self.encoder, self.predictor, self.joint = StubEncoder(), emb, joint
            self.blank, self.ignore_id = blank, -1

    ns = {"transducer": types.SimpleNamespace(Transducer=Transducer)}
    done = patch.install(ns, precision="bf16", vocab_tiling=True)
    try:
        assert "Transducer.vocab_tiling = True" in done["transducer"]
        model = Transducer()
        g = torch.Generator().manual_seed(10)
        enc = torch.randn(B, T, D, generator=g)
        lens = torch.tensor([16, 11, 7])
        text = torch.randint(1, V, (B, U), generator=g)
        tlen = torch.tensor([6, 4, 2])
        loss = model._compute_rnnt_loss(enc.cuda(), lens.cuda(), text.cuda(), tlen.cuda())
        loss.backward()
        _tc_ok(C, "patched step")
        for n, q in list(joint.named_parameters()) + list(emb.named_parameters()):
            assert q.grad is not None and bool(torch.isfinite(q.grad).all()), n
        ys = torch.cat([torch.full((B, 1), blank), text], 1)
        pred = emb.weight.detach().cpu().double()[ys]
        ref = restated(enc, pred, joint_weights(joint), text.int(), lens.tolist(), tlen.tolist(), blank)
        r = ref["loss"].item()
        tol = max(BF16_COST * abs(r), BF16_COST_STEP * float((lens + tlen).double().mean()))
        assert abs(loss.item() - r) <= tol, (loss.item(), r)
    finally:
        patch.uninstall()


@pytest.mark.gpu
def test_cfg2_dims_v4096(C):
    """cfg2 dimensions (T = 250, U = 40, D = 512) at V = 4096 (ten tiles of 416 columns, 352 real in the last).

    Four utterances against fp64 per utterance, bf16x3 with vocab_tiling and the fp32 SIMT path alike, at the bars of
    tests/test_joint_edges.py: 1e-4 plus twice the error of an fp32 restatement of the reference, which is not small
    here (a d_enc element sums 41 x 4096 fp32 products).  Measured on a B200, the fp32 path itself is up to 4.6e-4
    rel-L2 from fp64 on one utterance's d_enc, bf16x3 with vocab tiles 3.6e-4 - each within its bar.

    Then the full batch of 32, bf16x3 against fp32, where no fp64 reference is computed: both are within their bars of
    fp64, so they may differ by the sum of the two (the triangle inequality), taken as the largest per-utterance bar of
    the four checked utterances.  A fixed 1e-4 between the two paths is not a property either of them has at this size
    (measured 1.9e-4 - 2.3e-4 on d_enc from run to run: both accumulate in fp32 atomics of varying order)."""
    T, U1, D, V, blank = 250, 41, 512, 4096, 0
    g = torch.Generator().manual_seed(11)
    B = 32
    enc = 0.5 * torch.randn(B, T, D, generator=g)
    pred = 0.5 * torch.randn(B, U1, D, generator=g)
    w = torch.randn(V, D, generator=g) / math.sqrt(D)
    b = 0.1 * torch.randn(V, generator=g)
    tgt = torch.randint(1, V, (B, U1 - 1), generator=g, dtype=torch.int32)
    tl = [T, 187, 250, 131] + torch.randint(T // 2, T + 1, (B - 4,), generator=g).tolist()
    ul = [U1 - 1, 33, 21, 40] + torch.randint(U1 // 2, U1, (B - 4,), generator=g).tolist()
    # four utterances against fp64
    sl, gc4 = slice(0, 4), [1.7, -0.6, 0.25, 3.0]
    args = (enc[sl], pred[sl], w, b, tgt[sl], tl[:4], ul[:4], blank, -1.0, gc4, "tanh")
    ref64, ref32 = oracle(*args), oracle(*args, torch.float32)
    fails, pair_bar = [], {}
    for prec in ("bf16x3", "fp32"):
        got = run(C, prec, "tanh", enc[sl], pred[sl], w, b, tgt[sl], tl[:4], ul[:4], blank, -1.0, gc4)
        tol = bars(prec, ref64, ref32, tl[:4])
        for i, k in enumerate(GRADS):
            pair_bar[k] = pair_bar.get(k, 0.0) + float(tol[2][:, i].max())
        for k in SHARED:
            pair_bar[k] = pair_bar.get(k, 0.0) + tol[3][k]
        f, worst = check(got, ref64, tl[:4], ul[:4], gc4, *tol)
        print(f"VT cfg2 V=4096 {prec} vs fp64: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
        fails += [f"{prec}: {m}" for m in f]
    assert not fails, "\n".join(fails)
    # the full batch, bf16x3 against fp32
    gc = [1.0 / B] * B
    x3 = run(C, "bf16x3", "tanh", enc, pred, w, b, tgt, tl, ul, blank, -1.0, gc)
    f32 = run(C, "fp32", "tanh", enc, pred, w, b, tgt, tl, ul, blank, -1.0, gc)
    cost = float(((x3["costs"] - f32["costs"]).abs() / f32["costs"].abs()).max())
    errs = {k: rel_l2(x3[k], f32[k]) for k in GRADS + SHARED}
    print(f"VT cfg2 V=4096 bf16x3 vs fp32: cost {cost:.2e} " +
          " ".join(f"{k}={v:.2e} (bar {pair_bar[k]:.1e})" for k, v in errs.items()))
    assert cost <= F32_TOL
    assert all(errs[k] <= pair_bar[k] for k in errs), (errs, pair_bar)


@pytest.mark.gpu
def test_vocabulary_cap(C):
    """V = 32768 (79 tiles) at a small lattice, bf16x3 against fp64; V = 32769 raises."""
    c = _case("cap", 2, 5, 3, 128, V_CAP, V_CAP - 1, tl=(5, 3), ul=(2, 1), gc=(1.7, -0.6), seed=50)
    enc, pred, w, b, tgt = make_inputs(c)
    tl, ul = clamped_lengths(c)
    ref64 = oracle(enc, pred, w, b, tgt, tl, ul, c["blank"], -1.0, c["gc"], "tanh")
    ref32 = oracle(enc, pred, w, b, tgt, tl, ul, c["blank"], -1.0, c["gc"], "tanh", torch.float32)
    got = run(C, "bf16x3", "tanh", enc, pred, w, b, tgt, tl, ul, c["blank"], -1.0, c["gc"])
    f, worst = check(got, ref64, tl, ul, c["gc"], *bars("bf16x3", ref64, ref32, tl))
    print("VT cap: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
    assert not f, f
    w2, b2 = torch.zeros(V_CAP + 1, 128), torch.zeros(V_CAP + 1)
    with pytest.raises(RuntimeError, match="vocab_tiling=True needs"):
        run(C, "bf16", "tanh", enc, pred, w2, b2, tgt, tl, ul, 0, -1.0, c["gc"])


@pytest.mark.gpu
def test_without_opt_in_large_vocabulary_still_raises(C):
    """V > 416 without vocab_tiling keeps the error of the tensor-core precisions (now naming the opt-in); fp32 ignores
    the flag; CTCVR_F32 is an error of the vt entry points that names the plain one."""
    from ctcvr_b200._lib import call, ptr, stream
    c = CASES[0]
    enc, pred, w, b, tgt = make_inputs(c)
    tl, ul = clamped_lengths(c)
    for prec in ("bf16", "bf16x3"):
        with pytest.raises(RuntimeError, match=f"precision='{prec}' needs.*vocab_tiling=True"):
            run(C, prec, "tanh", enc, pred, w, b, tgt, tl, ul, 0, -1.0, c["gc"], vocab_tiling=False)
    a = run(C, "fp32", "tanh", enc, pred, w, b, tgt, tl, ul, 0, -1.0, c["gc"], vocab_tiling=False)
    bb = run(C, "fp32", "tanh", enc, pred, w, b, tgt, tl, ul, 0, -1.0, c["gc"], vocab_tiling=True)
    assert torch.equal(a["costs"], bb["costs"])
    B, T, U1, D, V = 2, 5, 3, 128, 500
    f = lambda *s: torch.zeros(*s, device="cuda")
    i = lambda *s: torch.ones(*s, dtype=torch.int32, device="cuda")
    ws = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    with pytest.raises(RuntimeError, match="ctcvr_joint_rnnt_fwd"):
        call("ctcvr_joint_rnnt_fwd_vt", ptr(f(B, T, D)), ptr(f(B, U1, D)), ptr(f(V, D)), ptr(f(V)), ptr(i(B, U1 - 1)),
             ptr(i(B)), ptr(i(B)), ptr(f(B, T, U1)), ptr(f(B, T, U1)), ptr(f(B, T, U1)), B, T, U1, D, V, 0, 0, ptr(ws),
             ws.numel(), stream())
    for bad in (0x300, 0x400, 3):
        with pytest.raises(RuntimeError, match="unknown precision"):
            call("ctcvr_joint_rnnt_fwd_vt", ptr(f(B, T, D)), ptr(f(B, U1, D)), ptr(f(V, D)), ptr(f(V)),
                 ptr(i(B, U1 - 1)), ptr(i(B)), ptr(i(B)), ptr(f(B, T, U1)), ptr(f(B, T, U1)), ptr(f(B, T, U1)), B, T,
                 U1, D, V, 0, bad, ptr(ws), ws.numel(), stream())
    _tc_ok(C, "errors")
