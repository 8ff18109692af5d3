"""Joints other than add + tanh with pre-join linears: activation 'relu' / 'gelu' (nn.ReLU, exact nn.GELU()), a post-join
linear (joint.py:64-65) and prejoin_linear=False, through the fused RNN-T loss, the training seams and the decoders.

The restatement below extends the oracle's joint (oracle/transducer_oracle.py) to these configurations: the lattice, the
predictor and the decoder walks are the oracle's own; only the joint changes, so the decoder restatements run with
`joint_forward` swapped for `joint_forward_act`.  The per-utterance checker and its bars are those of
tests/test_joint_edges.py."""
import contextlib
import ctypes
import math
import os
import re
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import transducer_oracle as TO
from test_joint_edges import F32_TOL, GRADS, SHARED, bars, check, rel_l2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ACTS = {"tanh": torch.tanh, "relu": torch.relu, "gelu": lambda x: F.gelu(x, approximate="none")}


# --------------------------------------------------------------------------------------------------- restatement
def joint_forward_act(enc_out, pred_out, w, pre_project=True, activation="tanh"):
    """model/component/joint.py:48-69, joint_mode='add': pre-join linears when their keys are in `w`, the post-join
    linear when `post_ffn.weight` is, then `activation` and ffn_out."""
    if pre_project and "enc_ffn.weight" in w:
        enc_out = F.linear(enc_out, w["enc_ffn.weight"], w["enc_ffn.bias"])
        pred_out = F.linear(pred_out, w["pred_ffn.weight"], w["pred_ffn.bias"])
    out = enc_out.unsqueeze(2) + pred_out.unsqueeze(1)
    if "post_ffn.weight" in w:
        out = F.linear(out, w["post_ffn.weight"], w["post_ffn.bias"])
    act = ACTS[activation] if isinstance(activation, str) else activation
    return F.linear(act(out), w["ffn_out.weight"], w["ffn_out.bias"])


def restated(enc, pred, w, tgt, tl, ul, blank, clamp=-1.0, gc=None, activation="tanh", dtype=torch.float64):
    """fp64 loss and gradients of every input and weight (TO.fused_joint_rnnt_restated with joint_forward_act)."""
    ws = {k: v.detach().to(dtype).requires_grad_(True) for k, v in w.items()}
    e = enc.detach().cpu().to(dtype).requires_grad_(True)
    p = pred.detach().cpu().to(dtype).requires_grad_(True)
    logits = joint_forward_act(e, p, ws, True, activation)
    r = TO.rnnt_lattice_restated(logits, tgt.cpu(), torch.as_tensor(tl), torch.as_tensor(ul), blank, clamp, dtype)
    B = logits.size(0)
    scale = torch.full((B,), 1.0 / B, dtype=dtype) if gc is None else torch.as_tensor(gc, dtype=dtype)
    logits.backward(r["grads"] * scale.reshape(B, 1, 1, 1))
    out = dict(costs=r["costs"], loss=r["costs"].mean(), d_enc=e.grad, d_pred=p.grad)
    out.update({"d_" + k: v.grad for k, v in ws.items()})
    return out


@contextlib.contextmanager
def oracle_activation(activation):
    """The oracle's decoder walks with the joint of `activation` (and post_ffn.* / missing pre-join keys honoured)."""
    old = TO.joint_forward
    TO.joint_forward = lambda e, p, w, pre_project=True: joint_forward_act(e, p, w, pre_project, activation)
    try:
        yield
    finally:
        TO.joint_forward = old


def relu_kink_of_bf16_inputs(enc, pred):
    """relu whose derivative is taken where the bf16 path takes it: at the sum of the bf16-rounded inputs.  Rounding e
    and p to bf16 moves every h closer to 0 than their rounding error (~2^-9 |e|) to a random side of the kink, and each
    such element flips its derivative between 0 and 1.  The restatement with this mask (values unchanged, fp64
    otherwise) isolates that effect from the kernels' own bf16 arithmetic."""
    mask = ((enc.bfloat16().double().unsqueeze(2) + pred.bfloat16().double().unsqueeze(1)) > 0).double()
    return lambda h: torch.relu(h).detach() + (h - h.detach()) * mask


def joint_weights(joint, dtype=torch.float64):
    return {k: v.detach().cpu().to(dtype) for k, v in joint.state_dict().items()}


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("activation", ["tanh", "relu", "gelu"])
@pytest.mark.parametrize("layout", ["pre", "pre+post", "post", "none"])
def test_restatement_matches_module_composition(activation, layout):
    """joint_forward_act equals the nn.Linear / activation module composition of joint.py in fp64."""
    torch.manual_seed(1)
    D, V = 12, 7
    pre, post = layout in ("pre", "pre+post"), "post" in layout
    mods = dict(enc_ffn=torch.nn.Linear(D, D), pred_ffn=torch.nn.Linear(D, D), post_ffn=torch.nn.Linear(D, D),
                ffn_out=torch.nn.Linear(D, V))
    act = {"tanh": torch.nn.Tanh(), "relu": torch.nn.ReLU(), "gelu": torch.nn.GELU()}[activation]
    mods = {k: m.double() for k, m in mods.items()}
    e, p = torch.randn(2, 5, D, dtype=torch.float64), torch.randn(2, 3, D, dtype=torch.float64)
    x, y = (mods["enc_ffn"](e), mods["pred_ffn"](p)) if pre else (e, p)
    h = x.unsqueeze(2) + y.unsqueeze(1)
    ref = mods["ffn_out"](act(mods["post_ffn"](h) if post else h))
    w = {f"{n}.{k}": v for n, m in mods.items() for k, v in m.state_dict().items()
         if (pre or n not in ("enc_ffn", "pred_ffn")) and (post or n != "post_ffn")}
    assert set(k.split(".")[0] for k in w) == ({"enc_ffn", "pred_ffn"} if pre else set()) | \
        ({"post_ffn"} if post else set()) | {"ffn_out"}
    assert torch.allclose(joint_forward_act(e, p, w, True, activation), ref, rtol=0, atol=1e-13)


def test_post_join_fold_identity():
    """post(e + p) = (W_post e + b_post) + W_post p to 1e-12 in fp64, the gradients of e, p, W_post, b_post included: the
    identity the fused loss and the decoders fold the post-join linear with."""
    torch.manual_seed(2)
    D = 16
    e = torch.randn(3, 5, D, dtype=torch.float64, requires_grad=True)
    p = torch.randn(3, 4, D, dtype=torch.float64, requires_grad=True)
    W = torch.randn(D, D, dtype=torch.float64, requires_grad=True)
    b = torch.randn(D, dtype=torch.float64, requires_grad=True)
    g = torch.randn(3, 5, 4, D, dtype=torch.float64)
    a = F.linear(e.unsqueeze(2) + p.unsqueeze(1), W, b)
    f = F.linear(e, W, b).unsqueeze(2) + F.linear(p, W).unsqueeze(1)
    assert float((a - f).detach().abs().max()) <= 1e-12
    ga = torch.autograd.grad(a, (e, p, W, b), g)
    gf = torch.autograd.grad(f, (e, p, W, b), g)
    for x, y in zip(ga, gf):
        assert float((x - y).abs().max()) <= 1e-12 * max(1.0, float(x.abs().max()))


def test_decoder_weights_mirror_header():
    """`_lib.DecoderWeights` lists the fields of `ctcvr_decoder_weights` in the header's order, `activation` last."""
    import ctcvr_b200._lib as L
    src = open(os.path.join(ROOT, "include", "ctcvr.h")).read()
    body = re.search(r"typedef struct \{(.*?)\} ctcvr_decoder_weights;", src, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            names += [n.strip().lstrip("*") for n in re.sub(r"^(const\s+)?\w+\s*\*?", "", decl).split(",")]
    assert [n for n, _ in L.DecoderWeights._fields_] == names
    assert names[-1] == "activation" and L.DecoderWeights._fields_[-1][1] is ctypes.c_int
    defs = dict(re.findall(r"#define (CTCVR_ACT_\w+) (0x[0-9a-f]+)", src))
    from ctcvr_b200 import functional as CF
    assert {k: int(v, 16) for k, v in defs.items()} == {"CTCVR_ACT_TANH": CF.ACT_TANH, "CTCVR_ACT_RELU": CF.ACT_RELU,
                                                      "CTCVR_ACT_GELU": CF.ACT_GELU}


def test_ws_bytes_accept_activation_bits():
    """The workspace queries take the activation bits OR'ed into `precision`; they do not change the size."""
    from ctcvr_b200._lib import query
    for q in ("ctcvr_joint_rnnt_fwd_ws_bytes", "ctcvr_joint_rnnt_bwd_ws_bytes"):
        for prec in (0, 1, 2):
            base = query(q, 4, 50, 11, 256, 100, prec)
            assert base > 0
            for act in (0x100, 0x200):
                assert query(q, 4, 50, 11, 256, 100, prec | act) == base


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def C():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import ctcvr_b200
    return ctcvr_b200


def _case(name, B, T, U1, D, V, blank, tl, ul, gc, seed, columns=("fp32", "bf16x3", "bf16", "bf16in")):
    return dict(name=name, B=B, T=T, U1=U1, D=D, V=V, blank=blank, tl=list(tl), ul=list(ul), gc=list(gc), seed=seed,
                columns=columns)


CASES = [
    # D = 256: CTA-pair backward; V = 45 is off the 32-padding
    _case("pair_d256", 4, 70, 19, 256, 45, 7, tl=(70, 41, 9, 1), ul=(18, 11, 5, 0), gc=(1.7, -0.6, 0.0, 3.0), seed=1),
    # D = 384: single-CTA backward (D % 256 != 0); V = 130
    _case("single_d384", 3, 33, 30, 384, 130, 0, tl=(33, 20, 14), ul=(29, 7, 13), gc=(-0.6, 1.7, 0.25), seed=2),
    # outside the tensor-core tiling (U + 1 = 140, D = 96): fp32 only
    _case("fp32only", 2, 20, 140, 96, 37, 3, tl=(20, 11), ul=(139, 40), gc=(1.1, -0.4), seed=3, columns=("fp32",)),
]


def _inputs(c):
    g = torch.Generator().manual_seed(500 + c["seed"])
    B, T, U1, D, V = c["B"], c["T"], c["U1"], c["D"], c["V"]
    enc = 0.5 * torch.randn(B, T, D, generator=g)
    pred = 0.5 * torch.randn(B, U1, D, generator=g)
    # exact zeros of h = e + p: the relu derivative is 0 there (torch's convention), gelu's is 1/2
    for b in range(B):
        enc[b, 0, : D // 2] = -pred[b, 0, : D // 2]
        enc[b, 1, ::3] = -pred[b, 1, ::3]
    w = torch.randn(V, D, generator=g) / math.sqrt(D)
    bias = 0.1 * torch.randn(V, generator=g)
    tgt = torch.randint(0, V, (B, U1 - 1), generator=g, dtype=torch.int32)
    return enc, pred, w, bias, tgt


def _identity_weights(D, w, bias):
    eye, zero = torch.eye(D, dtype=torch.float64), torch.zeros(D, dtype=torch.float64)
    return {"enc_ffn.weight": eye, "enc_ffn.bias": zero, "pred_ffn.weight": eye, "pred_ffn.bias": zero,
            "ffn_out.weight": w.double(), "ffn_out.bias": bias.double()}


def _run(C, col, act, enc, pred, w, bias, tgt, tl, ul, blank, clamp, gc):
    dev = "cuda"
    prec = "bf16" if col == "bf16in" else col
    dt = torch.bfloat16 if col == "bf16in" else torch.float32
    e = enc.to(dev, dt).requires_grad_(True)
    p = pred.to(dev, dt).requires_grad_(True)
    W, b = w.to(dev).requires_grad_(True), bias.to(dev).requires_grad_(True)
    costs = C.fused_joint_rnnt_loss(e, p, W, b, tgt.to(dev), torch.tensor(tl, device=dev), torch.tensor(ul, device=dev),
                                    blank, clamp, "none", prec, activation=act)
    costs.backward(torch.tensor(gc, device=dev, dtype=torch.float32))
    assert e.grad.dtype == dt and p.grad.dtype == dt
    return dict(costs=costs.detach().double().cpu(), d_enc=e.grad.double().cpu(), d_pred=p.grad.double().cpu(),
                d_w=W.grad.double().cpu(), d_b=b.grad.double().cpu())


@pytest.mark.gpu
@pytest.mark.parametrize("act", ["relu", "gelu"])
@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_fused_loss_per_utterance(C, case, act):
    """Every column of every case, clamp off and on, against the fp64 restatement per utterance, with the bars of
    tests/test_joint_edges.py.  The bf16-input column is compared with a restatement of the bf16-rounded inputs.

    relu in bf16 on fp32 inputs: the kernels round the inputs to bf16 (as for tanh), and elements whose h is within the
    rounding error of 0 change side of the kink, i.e. their derivative flips between 0 and 1.  Those flips are a property
    of rounding the inputs, not of the kernels' arithmetic: their relative-L2 effect on a gradient is about
    sqrt(flipped fraction): 4.6e-4 of the elements flip in the D = 384 case, and the restatement with the flipped
    derivatives alone is 4.63e-2 off on one utterance's d_enc - what the kernels measured on a B200 (4.63e-2), while the
    bf16-input column, without the flips, is within 3e-3.  That column's gradient bar is therefore 3e-2 plus the error of an fp64 restatement that takes the
    derivative at the bf16-rounded sum (`relu_kink_of_bf16_inputs`), per utterance; the bf16-input column, whose
    reference is the rounded inputs, keeps the plain 3e-2."""
    enc, pred, w, bias, tgt = _inputs(case)
    tl, ul, gc, blank, D = case["tl"], case["ul"], case["gc"], case["blank"], case["D"]
    ws = _identity_weights(D, w, bias)
    report = []
    for clamp in (-1.0, 0.05):
        refs = {}
        for rounded in (False, True):
            e_, p_ = (enc.bfloat16().float(), pred.bfloat16().float()) if rounded else (enc, pred)
            r64 = restated(e_, p_, ws, tgt, tl, ul, blank, clamp, gc, act)
            r32 = restated(e_, p_, {k: v.float() for k, v in ws.items()}, tgt, tl, ul, blank, clamp, gc, act, torch.float32)
            refs[rounded] = ({"costs": r64["costs"], "d_enc": r64["d_enc"], "d_pred": r64["d_pred"],
                              "d_w": r64["d_ffn_out.weight"], "d_b": r64["d_ffn_out.bias"]},
                             {"costs": r32["costs"].double(), "d_enc": r32["d_enc"].double(), "d_pred": r32["d_pred"].double(),
                              "d_w": r32["d_ffn_out.weight"].double(), "d_b": r32["d_ffn_out.bias"].double()})
        for col in case["columns"]:
            ref64, ref32 = refs[col == "bf16in"]
            got = _run(C, col, act, enc, pred, w, bias, tgt, tl, ul, blank, clamp, gc)
            tol = bars(col, ref64, ref32, tl)
            if act == "relu" and col == "bf16":
                kink = restated(enc, pred, ws, tgt, tl, ul, blank, clamp, gc, relu_kink_of_bf16_inputs(enc, pred))
                kink = {"d_enc": kink["d_enc"], "d_pred": kink["d_pred"], "d_w": kink["d_ffn_out.weight"],
                        "d_b": kink["d_ffn_out.bias"]}
                grad = np.array([[tol[2] + (rel_l2(kink[k][b], ref64[k][b]) if tl[b] > 0 else 0.0) for k in GRADS]
                                 for b in range(len(tl))])
                tol = (tol[0], tol[1], grad, {k: tol[3][k] + rel_l2(kink[k], ref64[k]) for k in SHARED})
            fails, worst = check(got, ref64, tl, ul, gc, *tol)
            report.append((col, clamp, fails, {k: f"{v:.2e}" for k, v in worst.items()}))
    print(case["name"], act, [(c, cl, w_) for c, cl, _, w_ in report])
    bad = [(c, cl, f) for c, cl, f, _ in report if f]
    assert not bad, bad


def _make_joint(C, act, pre, post, D=128, V=29, seed=0):
    torch.manual_seed(seed)
    j = C.TransducerJoint(V, D, D, D, prejoin_linear=pre, postjoin_linear=post, activation=act)
    for prm in j.parameters():
        prm.data.mul_(1.5)
    return j.cuda()


LAYOUTS = [(True, True), (False, True), (False, False)]      # (prejoin_linear, postjoin_linear)


def _rel(a, b):
    return float((a.double().cpu() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


@pytest.mark.gpu
@pytest.mark.parametrize("act", ["tanh", "relu", "gelu"])
@pytest.mark.parametrize("pre,post", LAYOUTS)
def test_call_chain(C, act, pre, post):
    """rnnt_loss_fused and compute_rnnt_loss (the body of Transducer._compute_rnnt_loss) on every layout: the loss and the
    gradient of every joint parameter (post_ffn.* included) and of the inputs against the fp64 restatement."""
    from ctcvr_b200.transducer import compute_rnnt_loss
    B, T, U, D, V, blank = 3, 14, 6, 128, 29, 0
    joint = _make_joint(C, act, pre, post, D, V)
    w64 = joint_weights(joint)
    g = torch.Generator().manual_seed(9)
    enc = 0.7 * torch.randn(B, T, D, generator=g)
    text = torch.randint(1, V, (B, U), generator=g)
    tl, ul = [14, 9, 5], [6, 4, 1]
    emb = torch.nn.Embedding(V, D).cuda()
    ys = torch.cat([torch.full((B, 1), blank), text], 1)
    pred = emb(ys.cuda()).detach().cpu()
    ref = restated(enc, pred, w64, text.int(), tl, ul, blank, activation=act)
    for prec in ("fp32", "bf16x3"):
        for route in ("rnnt_loss_fused", "compute_rnnt_loss"):
            joint.zero_grad()
            e = enc.cuda().requires_grad_(True)
            if route == "rnnt_loss_fused":
                p = pred.cuda().requires_grad_(True)
                loss = joint.rnnt_loss_fused(e, p, text.int().cuda(), torch.tensor(tl).cuda(), torch.tensor(ul).cuda(), blank,
                                             precision=prec)
            else:
                model = types.SimpleNamespace(predictor=lambda y: emb(y).detach(), joint=joint, blank=blank, ignore_id=-1,
                                              precision=prec)
                loss = compute_rnnt_loss(model, e, torch.tensor(tl).cuda(), text.cuda(), torch.tensor(ul).cuda())
            loss.backward()
            assert abs(loss.item() - ref["loss"].item()) <= F32_TOL * abs(ref["loss"].item()), (prec, route)
            assert _rel(e.grad, ref["d_enc"]) <= F32_TOL, (prec, route)
            for n, prm in joint.named_parameters():
                assert _rel(prm.grad, ref["d_" + n]) <= F32_TOL, (prec, route, n)
    # bf16: the same seam at the bf16 bars (the pre- / post-projections run as bf16 GEMMs)
    joint.zero_grad()
    e = enc.cuda().requires_grad_(True)
    loss = joint.rnnt_loss_fused(e, pred.cuda(), text.int().cuda(), torch.tensor(tl).cuda(), torch.tensor(ul).cuda(), blank,
                                 precision="bf16")
    loss.backward()
    assert abs(loss.item() - ref["loss"].item()) <= 2e-2 * abs(ref["loss"].item())
    assert _rel(e.grad, ref["d_enc"]) <= 5e-2
    for n, prm in joint.named_parameters():
        assert _rel(prm.grad, ref["d_" + n]) <= 5e-2, n


def _decode_model(C, act, pre, post, D=48, V=23, seed=3):
    torch.manual_seed(seed)
    predictor = C.RNNPredictor(V, D, D, 0.0, D, 1, dropout=0.0).cuda().eval()
    for prm in predictor.parameters():
        prm.data.mul_(1.5)
    joint = C.TransducerJoint(V, D, D, D, prejoin_linear=pre, postjoin_linear=post, activation=act)
    for prm in joint.parameters():
        prm.data.mul_(2.0)
    with torch.no_grad():
        joint.ffn_out.bias[0] += 2.0                       # blank bias: hypotheses of a few tokens per utterance
    return types.SimpleNamespace(predictor=predictor, joint=joint.cuda().eval(), blank=0)


DEC_LAYOUTS = [("relu", True, False), ("gelu", True, False), ("relu", True, True), ("gelu", False, True),
               ("tanh", True, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("act,pre,post", DEC_LAYOUTS)
def test_decoders(C, act, pre, post):
    """Greedy (offline and streaming over chunks), online beam, prefix beam and the two batched beams return the oracle
    walks' token ids for relu, gelu and post-join joints."""
    m = _decode_model(C, act, pre, post)
    pw = {k: v.detach().cpu().float() for k, v in m.predictor.state_dict().items()}
    jw = {k: v.detach().cpu().float() for k, v in m.joint.state_dict().items()}
    g = torch.Generator().manual_seed(11)
    S, T, D, V = 3, 9, 48, 23
    enc = torch.randn(S, T, D, generator=g)
    lens = torch.tensor([9, 6, 4])
    ctc_logp = torch.log_softmax(torch.randn(S, T, V, generator=g), -1)
    with oracle_activation(act):             # the walks apply enc_ffn / pred_ffn / post_ffn of jw where present
        ref_greedy = TO.greedy_search_offline(pw, jw, 0, enc, lens, n_steps=5)
        st, last, ref_stream = None, 0, []
        for s in range(0, T, 4):
            toks, st, last = TO.greedy_chunk_streaming(pw, jw, 0, enc[0, s:s + 4], st, last, 5)
            ref_stream += toks
        ref_beam = [[h.tokens for h in TO.beam_chunk_online(pw, jw, 0, enc[s_, :int(lens[s_])], None, 3, 5)]
                    for s_ in range(S)]
        ref_pb = [[h for h, _ in TO.prefix_beam_search_wenet(pw, jw, 0, enc[s_, :int(lens[s_])],
                                                               ctc_logp[s_, :int(lens[s_])], 3)] for s_ in range(S)]
    ec = enc.cuda()
    assert C.basic_greedy_search(m, ec, lens.cuda(), n_steps=5) == ref_greedy
    toks, st, last = [], None, 0
    for s in range(0, T, 4):
        c, st, last = C.greedy_chunk(m, ec[:1, s:s + 4], st, last, n_steps=5)
        toks += c
    assert toks == ref_stream
    for s_ in range(S):
        hyps, _ = C.beam_chunk_online(m, ec[s_:s_ + 1, :int(lens[s_])], None, beam_size=3, n_steps=5)
        assert [h.tokens for h in hyps] == ref_beam[s_], s_
        pb = C.prefix_beam_search(m, ec[s_, :int(lens[s_])], ctc_logp[s_, :int(lens[s_])].cuda(), beam_size=3)
        assert [h for h, _ in pb] == ref_pb[s_], s_
    batched = C.beam_search_batch(m, ec, lens.cuda(), beam_size=3, n_steps=5)
    assert [[h.tokens for h in b] for b in batched] == ref_beam
    pbb = C.prefix_beam_search_batch(m, ec, lens.cuda(), ctc_logp.cuda(), beam_size=3)
    assert [[h for h, _ in b] for b in pbb] == ref_pb
    assert any(len(h) > 0 for h in ref_greedy)                # the walks emit tokens: the comparison has content


@pytest.mark.gpu
def test_patch_install_gelu_post_join(C):
    """patch.install() on reference-shaped stand-ins with a gelu + post-join joint: the training seam
    (Transducer._compute_rnnt_loss) returns the oracle loss and basic_greedy_search the oracle hypotheses."""
    from ctcvr_b200 import patch
    m = _decode_model(C, "gelu", True, True)
    blank, D, V = 0, 48, 23

    class StubEncoder(torch.nn.Module):
        def forward(self, speech, lens, *a):
            mask = (torch.arange(speech.size(1), device=speech.device)[None, :] < lens[:, None]).unsqueeze(1)
            return speech, mask

    class Transducer(torch.nn.Module):                  # model/component/transducer.py:73-189, bodies absent on purpose
        def __init__(self):
            super().__init__()
            self.encoder, self.predictor, self.joint = StubEncoder(), m.predictor, m.joint
            self.blank, self.ignore_id = blank, -1

    def basic_greedy_search(model, encoder_out, encoder_out_lens, n_steps=64):
        raise AssertionError("not patched")

    ns = {"transducer": types.SimpleNamespace(Transducer=Transducer, basic_greedy_search=basic_greedy_search)}
    done = patch.install(ns)
    try:
        assert "transducer" in done
        model = Transducer().cuda()
        g = torch.Generator().manual_seed(4)
        enc = torch.randn(2, 8, D, generator=g)
        lens = torch.tensor([8, 5])
        text = torch.randint(1, V, (2, 3), generator=g)
        tlen = torch.tensor([3, 2])
        loss = model._compute_rnnt_loss(enc.cuda(), lens.cuda(), text.cuda(), tlen.cuda())
        ys = torch.cat([torch.full((2, 1), blank), text], 1)
        pw64 = {k: v.detach().cpu().double() for k, v in m.predictor.state_dict().items()}
        pred = TO.predictor_forward(pw64, ys)
        ref = restated(enc, pred, joint_weights(m.joint), text.int(), lens.tolist(), tlen.tolist(), blank,
                       activation="gelu")
        assert abs(loss.item() - ref["loss"].item()) <= F32_TOL * abs(ref["loss"].item())
        hyps = ns["transducer"].basic_greedy_search(model, enc.cuda(), lens.cuda(), n_steps=5)
        pw = {k: v.detach().cpu().float() for k, v in m.predictor.state_dict().items()}
        jw = {k: v.detach().cpu().float() for k, v in m.joint.state_dict().items()}
        with oracle_activation("gelu"):
            assert hyps == TO.greedy_search_offline(pw, jw, blank, enc, lens, n_steps=5)
    finally:
        patch.uninstall()


@pytest.mark.gpu
def test_graphed_step_relu(C):
    """A GraphedJointRnntStep over a relu joint (pre- and post-join linears) replays to the eager result."""
    B, T, U, D, V, blank = 4, 20, 5, 128, 29, 0
    joint = _make_joint(C, "relu", True, True, D, V, seed=5)
    g = torch.Generator().manual_seed(6)
    enc, pred = torch.randn(B, T, D, generator=g).cuda(), torch.randn(B, U + 1, D, generator=g).cuda()
    tgt = torch.randint(1, V, (B, U), generator=g, dtype=torch.int32).cuda()
    tl, ul = torch.tensor([20, 17, 9, 3], dtype=torch.int32).cuda(), torch.tensor([5, 2, 4, 0], dtype=torch.int32).cuda()
    # the step is captured before any eager autograd graph over the joint exists (GraphedJointRnntStep's docstring)
    step = C.GraphedJointRnntStep(joint, B, T, U, blank)
    replays = []
    for _ in range(2):
        loss = step.step(enc, pred, tgt, tl, ul)
        torch.cuda.synchronize()
        replays.append((float(loss), {n: q.grad.clone() for n, q in step.joint.named_parameters()}, step.enc.grad.clone()))
    e, p = enc.clone().requires_grad_(True), pred.clone().requires_grad_(True)
    for q in joint.parameters():
        q.grad = None
    eager = joint.rnnt_loss_fused(e, p, tgt, tl, ul, blank, reduction="sum") / B
    eager.backward()
    for loss, grads, d_enc in replays:
        assert abs(loss - eager.item()) <= 1e-6 * abs(eager.item())
        for n, q in joint.named_parameters():
            assert _rel(grads[n], q.grad.cpu()) <= 1e-5, n
        assert _rel(d_enc, e.grad.cpu()) <= 1e-5


@pytest.mark.gpu
def test_unknown_activation_bit_is_an_error(C):
    """Bits of `precision` other than the precision and one CTCVR_ACT_* value make the entry points return non-zero
    (RuntimeError naming the value) before any launch; the decoders reject an unknown activation the same way."""
    from ctcvr_b200._lib import call, ptr, stream
    B, T, U1, D, V = 2, 5, 3, 128, 16
    f = lambda *s: torch.zeros(*s, device="cuda")
    i = lambda *s: torch.ones(*s, dtype=torch.int32, device="cuda")
    e, p, w, b, tg, tl, ul = f(B, T, D), f(B, U1, D), f(V, D), f(V), i(B, U1 - 1), i(B), i(B)
    lse, lpb, lpl = f(B, T, U1), f(B, T, U1), f(B, T, U1)
    ws = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    for bad in (0x300, 0x400, 0x1000, 0x10000, 3, 0x103, -1):
        with pytest.raises(RuntimeError, match="unknown precision"):
            call("ctcvr_joint_rnnt_fwd", ptr(e), ptr(p), ptr(w), ptr(b), ptr(tg), ptr(tl), ptr(ul), ptr(lse), ptr(lpb),
                 ptr(lpl), B, T, U1, D, V, 0, bad, ptr(ws), ws.numel(), stream())
        with pytest.raises(RuntimeError, match="unknown precision"):
            call("ctcvr_joint_rnnt_bwd", ptr(e), ptr(p), ptr(w), ptr(b), ptr(tg), ptr(tl), ptr(ul), ptr(lse), ptr(lpb),
                 ptr(lpl), ptr(lse), ptr(lse), ptr(f(B)), ptr(f(B)), -1.0, ptr(f(B, T, D)), ptr(f(B, U1, D)), ptr(f(V, D)),
                 ptr(f(V)), B, T, U1, D, V, 0, bad, ptr(ws), ws.numel(), stream())
    m = _decode_model(C, "relu", True, False)
    from ctcvr_b200.decode import _prepared
    wst = _prepared(m).get()
    wst.activation = 0x300
    try:
        with pytest.raises(RuntimeError, match="unknown activation"):
            call("ctcvr_rnnt_greedy", ctypes.byref(wst), ptr(f(1, 4, 48)), ptr(i(1)), ptr(f(1, 1, 48)), ptr(f(1, 1, 48)),
                 ptr(i(1)), ptr(i(1, 8)), ptr(i(1)), 1, 4, 8, 0, 2, None, 0, stream())
    finally:
        wst.activation = 0x100
    torch.cuda.synchronize()
