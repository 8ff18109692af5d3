"""precision='bf16x3': the fused joint + RNN-T loss on the tcgen05 tensor cores at fp32 accuracy (every fp32 GEMM
operand split into bf16 hi + lo, three MMAs per product).  CPU cases check the arithmetic of the split (oracle/) and the
host-side surface; GPU cases (-m gpu) hold the kernels to the fp32 contract of 1e-4."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from conftest import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_TOL_F32 = 1e-4


def rel_l2(a, b):
    a = a.detach().double().cpu().numpy() if torch.is_tensor(a) else np.asarray(a, dtype=np.float64)
    b = b.detach().double().cpu().numpy() if torch.is_tensor(b) else np.asarray(b, dtype=np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


@pytest.fixture(scope="module")
def C():
    import ctcvr_b200
    assert torch.cuda.is_available()
    ctcvr_b200._lib.lib()
    return ctcvr_b200


def _tc_ok(C):
    flag = C._lib.lib().ctcvr_debug_tc_error()
    assert flag == 0, f"tcgen05 kernel hit a bounded mbarrier wait: 0x{flag:08x}"


def _run_fused(C, joint, enc, pred, tgt, tl, ul, blank, clamp, precision):
    enc = enc.clone().requires_grad_(True)
    pred = pred.clone().requires_grad_(True)
    for p in joint.parameters():
        p.grad = None
    loss = joint.rnnt_loss_fused(enc, pred, tgt, tl, ul, blank, clamp=clamp, reduction="mean", precision=precision)
    loss.backward()
    g = {"d_enc": enc.grad, "d_pred": pred.grad}
    g.update({"d_" + k: v.grad for k, v in joint.named_parameters()})
    return loss, g


# ------------------------------------------------------------------------------------------------------------- CPU
def test_split_product_restatement_within_contract_of_fp64():
    """The paper estimate of the split, checked before any kernel: the fused loss with the three joint GEMMs computed as
    hi*hi + hi*lo + lo*hi of bf16 splits is within 1e-4 of the fp64 restatement, loss and every gradient."""
    from oracle import bf16x3_oracle as X
    from oracle import transducer_oracle as TO
    torch.manual_seed(11)
    B, Tm, U, D, V, blank = 3, 17, 6, 128, 90, 5
    enc, pred = torch.randn(B, Tm, D), torch.randn(B, U + 1, D)
    w = {"ffn_out.weight": torch.randn(V, D) / D ** 0.5, "ffn_out.bias": torch.randn(V) * 0.1}
    tgt = torch.randint(6, V, (B, U), dtype=torch.int32)
    tl = torch.tensor([Tm, 11, 4], dtype=torch.int32)
    ul = torch.tensor([U, 2, 6], dtype=torch.int32)
    for clamp in (-1.0, 0.05):
        x3 = X.fused_joint_rnnt_bf16x3_restated(enc, pred, w, tgt, tl, ul, blank, clamp)
        eye = {"enc_ffn.weight": torch.eye(D), "enc_ffn.bias": torch.zeros(D), "pred_ffn.weight": torch.eye(D),
               "pred_ffn.bias": torch.zeros(D)}              # identity pre-projections: the fused op's inputs
        ref = TO.fused_joint_rnnt_restated(enc, pred, {**w, **eye}, tgt, tl, ul, blank, clamp, torch.float64)
        assert ref["loss"].item() > 0
        assert abs(x3["loss"].item() - ref["loss"].item()) <= 1e-5 * abs(ref["loss"].item())
        for k in ("d_enc_out", "d_pred_out", "d_ffn_out.weight", "d_ffn_out.bias"):
            assert rel_l2(x3[k], ref[k]) < ORACLE_TOL_F32, (clamp, k, rel_l2(x3[k], ref[k]))
        # one bf16 term alone is far outside the contract: the split is what buys the accuracy
        z = torch.tanh(enc[:, :, None] + pred[:, None]).reshape(-1, D)
        one = z.to(torch.bfloat16).double() @ w["ffn_out.weight"].t().to(torch.bfloat16).double()
        assert rel_l2(one, z.double() @ w["ffn_out.weight"].t().double()) > 1e-3


def test_split_product_is_exact_on_bf16_values():
    from oracle import bf16x3_oracle as X
    a = torch.randn(8, 32).to(torch.bfloat16).float()
    b = torch.randn(32, 5).to(torch.bfloat16).float()
    assert torch.equal(X.split_bf16_product(a, b), a.double() @ b.double())


def test_bf16x3_precision_value_and_workspace_queries():
    """_PREC knows 'bf16x3' (= CTCVR_BF16X3 = 2); the workspace queries need no GPU.  The backward of bf16x3 holds
    everything bf16's does plus hi / lo weight copies and the G_lo spill; its forward reads the fp32 activations in
    place and needs only the hi / lo weight tiles instead of bf16 copies of the activations."""
    sys.path.insert(0, ROOT)
    import ctcvr_b200 as C
    from ctcvr_b200._lib import query
    F = C.functional
    assert F._PREC["bf16x3"] == F.BF16X3 == 2
    with open(os.path.join(ROOT, "include", "ctcvr.h")) as f:
        assert "#define CTCVR_BF16X3 2" in f.read()
    for (B, Tm, U1, D, V) in ((32, 250, 41, 512, 412), (2, 9, 4, 128, 50), (3, 70, 28, 384, 416)):
        b16 = query("ctcvr_joint_rnnt_bwd_ws_bytes", B, Tm, U1, D, V, 1)
        x3 = query("ctcvr_joint_rnnt_bwd_ws_bytes", B, Tm, U1, D, V, 2)
        assert x3 >= b16 > 256
        Vp = (V + 31) // 32 * 32
        f3 = query("ctcvr_joint_rnnt_fwd_ws_bytes", B, Tm, U1, D, V, 2)
        assert f3 >= 2 * Vp * D * 2                       # hi and lo W_out tiles
    # outside the tiling the query answers the minimum and the call itself raises
    assert query("ctcvr_joint_rnnt_fwd_ws_bytes", 2, 9, 4, 64, 50, 2) == 256


def test_patch_install_bf16x3_default_and_uninstall():
    sys.path.insert(0, ROOT)
    import ctcvr_b200 as C

    class Transducer:
        def _compute_rnnt_loss(self, *a):
            return "reference"

    ns = types.SimpleNamespace(transducer=types.SimpleNamespace(Transducer=Transducer, basic_greedy_search=lambda *a: "ref"))
    done = C.patch.install(ns, precision="bf16x3")
    assert "Transducer._compute_rnnt_loss" in done["transducer"] and Transducer.precision == "bf16x3"
    C.patch.uninstall()
    assert not hasattr(Transducer, "precision") and Transducer()._compute_rnnt_loss() == "reference"
    assert ns.transducer.basic_greedy_search() == "ref"
    with pytest.raises(ValueError):
        C.patch.install(ns, precision="fp16")


def test_graphed_step_bf16x3_requires_fp32_inputs():
    sys.path.insert(0, ROOT)
    import ctcvr_b200 as C
    joint = C.TransducerJoint(40, 128, 128, 128)
    with pytest.raises(ValueError, match="bf16x3"):
        C.GraphedJointRnntStep(joint, 2, 8, 3, 5, precision="bf16x3", input_dtype=torch.bfloat16)


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_bf16x3_cfg2_full_size_vs_oracle(C):
    """cfg2 (B=32, T=250, U=40, D=512, V=412, ragged) with the bars of the fp32 path: loss within 1e-4 of the CPU
    reference call, gradients within 5e-4 rel-L2 of it (the reference is fp32 too), and on a 4-utterance slice every
    gradient within max(1e-4, 2x torchaudio's own fp32 noise) of the fp64 restatement."""
    from oracle import transducer_oracle as TO
    torch.manual_seed(1234)
    B, Tm, U, D, V, blank = 32, 250, 40, 512, 412, 5
    joint = C.TransducerJoint(V, D, D, D)
    enc, pred = torch.randn(B, Tm, D), torch.randn(B, U + 1, D)
    tgt = torch.randint(6, V, (B, U), dtype=torch.int32)
    tl = torch.randint(125, 251, (B,), dtype=torch.int32)
    ul = torch.randint(20, 41, (B,), dtype=torch.int32)
    tl[0], ul[0] = Tm, U
    w = {k: v.detach().clone() for k, v in joint.state_dict().items()}
    ref = TO.fused_joint_rnnt_reference_call(enc, pred, w, tgt, tl, ul, blank)
    joint = joint.cuda()
    keys = ("d_enc", "d_pred", "d_ffn_out.weight", "d_ffn_out.bias", "d_enc_ffn.weight", "d_pred_ffn.weight")
    rk = lambda k: {"d_enc": "d_enc_out", "d_pred": "d_pred_out"}.get(k, k)
    loss, g = _run_fused(C, joint, enc.cuda(), pred.cuda(), tgt.cuda(), tl.cuda(), ul.cuda(), blank, -1.0, "bf16x3")
    torch.cuda.synchronize()
    _tc_ok(C)
    assert abs(loss.item() - ref["loss"].item()) <= ORACLE_TOL_F32 * abs(ref["loss"].item())
    for k in keys:
        assert rel_l2(g[k], ref[rk(k)]) < 5e-4, (k, rel_l2(g[k], ref[rk(k)]))
    for b in range(B):
        assert torch.all(g["d_enc"][b, int(tl[b]):] == 0) and torch.all(g["d_pred"][b, int(ul[b]) + 1:] == 0)
    n = 4
    r64 = TO.fused_joint_rnnt_restated(enc[:n], pred[:n], w, tgt[:n], tl[:n], ul[:n], blank)
    r32 = TO.fused_joint_rnnt_reference_call(enc[:n], pred[:n], w, tgt[:n], tl[:n], ul[:n], blank)
    loss, g = _run_fused(C, joint, enc[:n].cuda(), pred[:n].cuda(), tgt[:n].cuda(), tl[:n].cuda(), ul[:n].cuda(), blank,
                         -1.0, "bf16x3")
    assert abs(loss.item() - r64["loss"].item()) <= ORACLE_TOL_F32 * abs(r64["loss"].item())
    for k in keys:
        ours, theirs = rel_l2(g[k], r64[rk(k)]), rel_l2(r32[rk(k)], r64[rk(k)])
        assert ours < max(ORACLE_TOL_F32, 2.0 * theirs), (k, ours, theirs)


@pytest.mark.gpu
def test_bf16x3_random_shapes_vs_fp32_kernels(C):
    """Shape fuzz against the fp32 SIMT kernels (pinned to the reference at 1e-4), at the fp32 tolerances: every joint
    width, vocabularies on both sides of the padding boundaries, tiny and odd T / U, ragged lengths, clamp on and off.
    Gradients of padded frames / label positions are exact zeros."""
    rng = np.random.default_rng(7)
    for it in range(24):
        D = int(rng.choice([128, 256, 384, 512]))
        V = int(rng.choice([7, 16, 31, 33, 48, 65, 100, 200, 257, 384, 400, 412, 416]))
        B, Tm, U = int(rng.integers(1, 6)), int(rng.integers(1, 70)), int(rng.integers(0, 28))
        blank = int(rng.integers(0, V))
        clamp = -1.0 if it % 3 else 0.5
        torch.manual_seed(100 + it)
        joint = C.TransducerJoint(V, D, D, D).cuda()
        enc, pred = torch.randn(B, Tm, D, device="cuda"), torch.randn(B, U + 1, D, device="cuda")
        tgt = torch.randint(0, V, (B, max(U, 1)), dtype=torch.int32, device="cuda")[:, :U]
        tl = torch.randint(1, Tm + 1, (B,), dtype=torch.int32, device="cuda")
        ul = torch.randint(0, U + 1, (B,), dtype=torch.int32, device="cuda")
        tl[0], ul[0] = Tm, U
        res = {}
        for prec in ("fp32", "bf16x3"):
            loss, g = _run_fused(C, joint, enc, pred, tgt, tl, ul, blank, clamp, prec)
            res[prec] = (loss.item(), {k: v.clone() for k, v in g.items()})
        torch.cuda.synchronize()
        _tc_ok(C)
        tag = f"it={it} B={B} T={Tm} U={U} D={D} V={V} blank={blank} clamp={clamp}"
        l32, g32 = res["fp32"]
        lx, gx = res["bf16x3"]
        assert np.isfinite(lx), tag
        assert abs(lx - l32) <= ORACLE_TOL_F32 * max(abs(l32), 1.0), (tag, lx, l32)
        for k in g32:
            assert torch.isfinite(gx[k]).all(), (tag, k)
            if float(g32[k].norm()) > 1e-6:
                assert rel_l2(gx[k], g32[k]) < ORACLE_TOL_F32, (tag, k, rel_l2(gx[k], g32[k]))
        for b in range(B):
            assert torch.all(gx["d_enc"][b, int(tl[b]):] == 0) and torch.all(gx["d_pred"][b, int(ul[b]) + 1:] == 0), tag


@pytest.mark.gpu
def test_bf16x3_compute_rnnt_loss_seam_cfg1(C):
    """`Transducer._compute_rnnt_loss` on cfg1 with precision='bf16x3' against the reference model's loss_rnnt and its
    predictor-output gradient, at the fp32 path's bars."""
    fx = load_golden("cfg1_example1.npz")
    blank = int(fx["blank"])
    joint = C.TransducerJoint(412, 256, 256, 256).cuda()
    joint.load_state_dict({k[len("joint."):]: torch.from_numpy(np.asarray(v)).cuda() for k, v in fx.items()
                           if k.startswith("joint.")})

    class Pred(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.out = torch.nn.Parameter(torch.from_numpy(fx["predictor_out"]).cuda().clone())

        def forward(self, ys_in):
            return self.out

    pred = Pred().cuda()
    model = C.Transducer(412, blank, torch.nn.Identity(), pred, joint, ctc=None, ctc_weight=0.0, transducer_weight=1.0,
                         precision="bf16x3")
    loss = model._compute_rnnt_loss(torch.from_numpy(fx["encoder_out"]).cuda(), torch.from_numpy(fx["encoder_out_lens"]).cuda(),
                                    torch.from_numpy(fx["texts"]).cuda(), torch.from_numpy(fx["text_lens"]).cuda())
    loss.backward()
    torch.cuda.synchronize()
    _tc_ok(C)
    assert abs(loss.item() - float(fx["loss_rnnt"])) <= ORACLE_TOL_F32 * float(fx["loss_rnnt"])
    assert rel_l2(0.7 * pred.out.grad, fx["d_predictor_out"]) < 2e-4


@pytest.mark.gpu
def test_bf16x3_graphed_and_bucketed_steps_match_eager(C):
    torch.manual_seed(3)
    B, Tm, U, D, V, blank = 4, 60, 12, 256, 100, 5
    joint = C.TransducerJoint(V, D, D, D).cuda()
    g = C.GraphedJointRnntStep(joint, B, Tm, U, blank, precision="bf16x3")
    stepper = C.BucketedJointRnntStep(joint, blank, t_bucket=16, u_bucket=8, precision="bf16x3")
    for seed, (Tb, Ubt) in enumerate([(Tm, U), (50, 9)]):
        torch.manual_seed(10 + seed)
        enc = torch.randn(B, Tb, D, device="cuda", requires_grad=True)
        pred = torch.randn(B, Ubt + 1, D, device="cuda", requires_grad=True)
        tgt = torch.randint(6, V, (B, Ubt), dtype=torch.int32, device="cuda")
        tl = torch.tensor([Tb, 41, Tb - 3, 17], dtype=torch.int32, device="cuda")
        ul = torch.tensor([Ubt, 5, Ubt, 1], dtype=torch.int32, device="cuda")
        joint.zero_grad(set_to_none=True)
        costs = joint.rnnt_loss_fused(enc, pred, tgt, tl, ul, blank, reduction="none", precision="bf16x3")
        loss = costs.sum() / B
        loss.backward()
        want = {n: p.grad.clone() for n, p in joint.named_parameters()}
        want_e, want_p, want_loss = enc.grad.clone(), pred.grad.clone(), loss.item()
        del costs, loss
        joint.zero_grad(set_to_none=True)
        if Tb == Tm:
            got = g.step(enc.detach(), pred.detach(), tgt, tl, ul)
            ge, gp = g.enc.grad, g.pred.grad
        else:
            got = stepper.step(enc.detach(), pred.detach(), tgt, tl, ul)
            ge, gp = stepper.enc_grad, stepper.pred_grad
        torch.cuda.synchronize()
        _tc_ok(C)
        # same kernels on the same data: equal up to the order of the fp32 atomics behind d_pred / d_bias
        assert abs(got.item() - want_loss) <= 1e-5 * abs(want_loss)
        for n, p in joint.named_parameters():
            assert rel_l2(p.grad, want[n]) < 1e-5, n
        assert rel_l2(ge, want_e) < 1e-5 and rel_l2(gp, want_p) < 1e-5


@pytest.mark.gpu
def test_bf16x3_unsupported_shapes_and_bad_values(C):
    torch.manual_seed(0)
    for D, V in ((64, 50), (640, 50), (128, 500)):
        joint = C.TransducerJoint(V, D, D, D).cuda()
        enc, pred = torch.randn(2, 9, D, device="cuda"), torch.randn(2, 4, D, device="cuda")
        tgt = torch.randint(0, V, (2, 3), dtype=torch.int32, device="cuda")
        tl = torch.tensor([9, 5], dtype=torch.int32, device="cuda")
        ul = torch.tensor([3, 1], dtype=torch.int32, device="cuda")
        with pytest.raises(RuntimeError, match="precision='bf16x3' needs"):
            joint.rnnt_loss_fused(enc, pred, tgt, tl, ul, 1, precision="bf16x3")
    B, Tm, U, D, V, blank = 3, 40, 6, 128, 50, 5
    joint = C.TransducerJoint(V, D, D, D).cuda()
    enc, pred = torch.randn(B, Tm, D, device="cuda"), torch.randn(B, U + 1, D, device="cuda")
    tgt = torch.randint(0, V, (B, U), dtype=torch.int32, device="cuda")
    tgt[0, 1], tgt[1, 0] = 10 ** 6, -7
    tl = torch.tensor([Tm, Tm + 50, 3], dtype=torch.int32, device="cuda")
    ul = torch.tensor([U, U + 9, 2], dtype=torch.int32, device="cuda")
    e = enc.clone().requires_grad_(True)
    loss = joint.rnnt_loss_fused(e, pred, tgt, tl, ul, blank, precision="bf16x3")
    loss.backward()
    torch.cuda.synchronize()
    _tc_ok(C)
    assert torch.isfinite(loss) and torch.isfinite(e.grad).all()
