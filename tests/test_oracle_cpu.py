"""Pin the oracle: restatements vs the third-party ops called as the reference calls them,
and vs fixtures produced by the reference modules themselves (tests/golden/make_golden.py)."""
import numpy as np
import torch

from conftest import load_golden, predictor_case
from oracle import ctc_oracle as CO
from oracle import transducer_oracle as TO


def T(x):
    return torch.from_numpy(np.asarray(x))


def rel_l2(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


def _w(fx, prefix):
    return {k[len(prefix):]: T(v) for k, v in fx.items() if k.startswith(prefix)}


def test_lattice_restated_matches_torchaudio_and_golden():
    fx = load_golden("rnnt_small.npz")
    logits, tgt, tl, ul = T(fx["logits"]), T(fx["tgt"]), T(fx["tl"]), T(fx["ul"])
    blank = int(fx["blank"])
    for tag, clamp in (("n", -1.0), ("c", float(fx["clamp"]))):
        r = TO.rnnt_lattice_restated(logits, tgt, tl, ul, blank, clamp)
        np.testing.assert_allclose(r["costs"].numpy(), fx[f"{tag}_costs"], rtol=2e-6)
        np.testing.assert_allclose(r["costs"].mean().item(), fx[f"{tag}_loss"], rtol=2e-6)
        # reference gradient is d(mean)/dlogits = grads / B
        np.testing.assert_allclose(r["grads"].numpy() / logits.size(0), fx[f"{tag}_dlogits"], atol=2e-6)
        # padded cells carry exactly zero gradient
        assert np.all(r["grads"][1, 9:].numpy() == 0) and np.all(r["grads"][1, :, 4:].numpy() == 0)
    live = TO.rnnt_loss_reference_call(logits, tgt, tl, ul, blank, -1.0, "none")
    np.testing.assert_allclose(live.numpy(), fx["n_costs"], rtol=1e-6)


def test_fused_joint_rnnt_restated_matches_reference_grads():
    fx = load_golden("rnnt_small.npz")
    w = _w(fx, "w_")
    r = TO.fused_joint_rnnt_restated(T(fx["enc"]), T(fx["pred"]), w, T(fx["tgt"]), T(fx["tl"]), T(fx["ul"]),
                                     int(fx["blank"]))
    np.testing.assert_allclose(r["loss"].item(), fx["n_loss"], rtol=2e-6)
    np.testing.assert_allclose(r["d_enc_out"].numpy(), fx["n_d_enc"], atol=3e-6)
    np.testing.assert_allclose(r["d_pred_out"].numpy(), fx["n_d_pred"], atol=3e-6)
    for k in w:
        np.testing.assert_allclose(r["d_" + k].numpy(), fx["n_d_" + k], atol=1e-5, rtol=1e-4)


def test_cfg1_example1_loss():
    """BASELINE.json configs[0]: reference TransducerModel on example1.pt[:2]."""
    fx = load_golden("cfg1_example1.npz")
    jw = _w(fx, "joint.")
    enc, pred = T(fx["encoder_out"]), T(fx["predictor_out"])
    tl, ul = T(fx["encoder_out_lens"]), T(fx["text_lens"])
    r = TO.fused_joint_rnnt_restated(enc, pred, jw, T(fx["texts"]), tl, ul, int(fx["blank"]))
    np.testing.assert_allclose(r["loss"].item(), fx["loss_rnnt"], rtol=1e-5)
    loss_ctc, _ = CO.ctc_head_reference_call(enc, tl, T(fx["texts"]), ul, T(fx["ctc.ctc_lo.weight"]),
                                             T(fx["ctc.ctc_lo.bias"]), int(fx["blank"]), "offline")
    np.testing.assert_allclose(loss_ctc.item(), fx["loss_ctc"], rtol=1e-5)
    np.testing.assert_allclose(0.7 * r["loss"].item() + 0.3 * loss_ctc.item(), fx["loss"], rtol=1e-5)
    # d loss / d joint params = 0.7 * d rnnt / d params
    # (the reference is fp32: its own rounding noise vs this fp64 restatement is ~6e-5 rel-L2)
    for k in ("ffn_out.weight", "ffn_out.bias", "enc_ffn.weight", "pred_ffn.weight"):
        assert rel_l2(0.7 * r["d_" + k].numpy(), fx["d_" + k]) < 1e-4


def test_ctc_restated_matches_reference_heads():
    fx = load_golden("ctc_small.npz")
    hs, hl, ys, yl = T(fx["hs"]), T(fx["hl"]), T(fx["ys"]), T(fx["yl"])
    blank = int(fx["blank"])
    for mode, tag in (("offline", "off"), ("online", "on")):
        w, b = T(fx[f"{tag}_w"]), T(fx[f"{tag}_b"])
        loss, ys_hat = CO.ctc_head_reference_call(hs, hl, ys, yl, w, b, blank, mode)
        np.testing.assert_allclose(loss.item(), fx[f"{tag}_loss"], rtol=1e-6)
        np.testing.assert_allclose(ys_hat.numpy(), fx[f"{tag}_ys_hat"], atol=1e-6)
        nll, g = CO.ctc_loss_restated(ys_hat.numpy(), ys.numpy(), hl.numpy(), yl.numpy(), blank)
        B = hs.size(0)
        if mode == "offline":
            want = nll.sum() / B
            scale = np.full(B, 1.0 / B)
        else:
            want = (nll / np.maximum(yl.numpy(), 1)).mean()
            scale = 1.0 / np.maximum(yl.numpy(), 1) / B
        np.testing.assert_allclose(want, fx[f"{tag}_loss"], rtol=1e-5)
        dlogits = g * scale[:, None, None]
        d_hs = dlogits @ w.numpy().astype(np.float64)
        np.testing.assert_allclose(d_hs, fx[f"{tag}_d_hs"], atol=2e-6)
        assert nll[2] == 0.0 and np.all(g[2] == 0)            # infeasible -> zero_infinity


def test_ctc_restated_matches_aten_with_blank_targets():
    """The restatement against torch's ctc_loss in fp64 on targets equal to blank, where l' has odd states labelled
    blank: ATen allows the skip into such a state from the label two states back (and out of it two states on), and
    the gradient's blank column gathers them with the even states.  Also repeats, an empty target, an infeasible one.

    One exception: on the last frame ATen sets, rather than adds, the entry of the last target ("a blank and a
    non-blank"), so when that target is blank its gradient drops the final blank state.  There the restatement is held
    to central differences of ATen's cost instead."""
    g = torch.Generator().manual_seed(8)
    B, Tm, V, blank = 5, 9, 6, 2
    logits = 2.0 * torch.randn(B, Tm, V, generator=g, dtype=torch.float64)
    ys = torch.tensor([[2, 4, 1, 2], [4, 2, 2, 1], [2, 2, 2, 2], [3, 3, 0, 0], [1, 5, 1, 4]])
    hl, yl = torch.tensor([9, 7, 9, 9, 3]), torch.tensor([4, 4, 4, 0, 4])

    def aten(x):
        return torch.nn.functional.ctc_loss(x.log_softmax(2).transpose(0, 1), ys, hl, yl, blank=blank,
                                            reduction="none", zero_infinity=True)
    x = logits.clone().requires_grad_(True)
    want = aten(x)
    want.sum().backward()
    nll, grad = CO.ctc_loss_restated(logits.log_softmax(2).numpy(), ys.numpy(), hl.numpy(), yl.numpy(), blank)
    assert want[4].item() == 0.0 and nll[4] == 0.0 and np.all(grad[4] == 0)      # 3 frames for 4 labels
    np.testing.assert_allclose(nll, want.detach().numpy(), rtol=1e-12)
    ag = x.grad.numpy().copy()
    for b in (0, 2):                                  # last target blank: central differences on the last frame
        t = int(hl[b]) - 1
        for v in range(V):
            e = torch.zeros_like(logits)
            e[b, t, v] = 1e-6
            ag[b, t, v] = float(aten(logits + e)[b] - aten(logits - e)[b]) / 2e-6
    np.testing.assert_allclose(grad, ag, rtol=1e-6, atol=1e-9)


def test_example2_known_answers():
    """3.ipynb:87,159 and 3_v2.ipynb:150 record the frame argmax / collapsed ids of utts 0,1."""
    fx = load_golden("example2.npz")
    pre, lens, blank = T(fx["pre"]), fx["lens"], int(fx["blank"])
    hyps = CO.ctc_greedy_search(pre, lens, blank)
    res = CO.ctc_prefix_beam_search(pre, lens, int(fx["beam"]), blank)
    # collapsed sequences recorded in the notebooks (utt 0: 3_v2.ipynb:150, utt 1: 3.ipynb:159)
    assert hyps[0] == [2, 40, 188, 227, 247, 243, 375, 360, 32, 87, 251, 291, 282, 32, 141, 243, 55, 317, 3]
    assert hyps[1] == [2, 323, 296, 75, 243, 278, 394, 51, 247, 360, 364, 57, 238, 122, 65, 167, 271, 142, 68, 3]
    for i, r in enumerate(res):
        assert r["tokens"] == fx[f"best_{i}"].tolist()
        np.testing.assert_allclose(r["score"], fx[f"score_{i}"], rtol=1e-9, atol=1e-9)
        assert r["times"] == fx[f"times_{i}"].tolist()
        np.testing.assert_allclose(r["nbest_scores"], fx[f"nbest_scores_{i}"], rtol=1e-9, atol=1e-9)
        assert [t for x in r["nbest"] for t in x] == fx[f"nbest_flat_{i}"].tolist()
        assert [t for x in r["nbest_times"] for t in x] == fx[f"nbest_times_flat_{i}"].tolist()
    assert res[0]["tokens"] == hyps[0] and res[1]["tokens"] == hyps[1]


def test_decoders_match_reference():
    fx = load_golden("decode_small.npz")
    pw, jw = _w(fx, "predictor."), _w(fx, "joint.")
    enc, elens, blank = T(fx["enc"]), T(fx["elens"]), int(fx["blank"])
    hy = TO.greedy_search_offline(pw, jw, blank, enc, elens, 64)
    for b in range(3):
        assert hy[b] == fx[f"a5_hyp_{b}"].tolist()
    hy = TO.greedy_search_offline(pw, jw, blank, enc, elens, 2)
    for b in range(3):
        assert hy[b] == fx[f"a5cap2_hyp_{b}"].tolist()
    assert TO.greedy_search_offline(pw, jw, blank, enc[:1], elens[:1], 64)[0] == fx["a6w_hyp_0"].tolist()
    toks, st, last = [], None, blank
    for s in range(0, 37, 8):
        c, st, last = TO.greedy_chunk_streaming(pw, jw, blank, enc[0, s:s + 8], st, last, 10)
        toks += c
    assert toks == fx["a6_hyp_0"].tolist() and last == int(fx["a6_last"])
    np.testing.assert_allclose(st[0].numpy(), fx["a6_h"], atol=1e-5)
    for beam in (4, 10):
        hyps = None
        for s in range(0, 37, 8):
            hyps = TO.beam_chunk_online(pw, jw, blank, enc[0, s:s + 8], hyps, beam, 10)
        assert len(hyps) == int(fx[f"a7_b{beam}_n"])
        for i, h in enumerate(hyps):
            assert h.tokens == fx[f"a7_b{beam}_tok_{i}"].tolist()
            np.testing.assert_allclose(h.log_prob, fx[f"a7_b{beam}_lp_{i}"], atol=1e-4)
    ctc_logp = torch.log_softmax(enc[0] @ T(fx["ctc.ctc_lo.weight"]).T + T(fx["ctc.ctc_lo.bias"]), dim=-1)
    for beam in (5, 10):
        out = TO.prefix_beam_search_wenet(pw, jw, blank, enc[0], ctc_logp, beam)
        assert len(out) == int(fx[f"a8_b{beam}_n"])
        for i, (hyp, sc) in enumerate(out):
            assert hyp == fx[f"a8_b{beam}_tok_{i}"].tolist()
            np.testing.assert_allclose(sc, fx[f"a8_b{beam}_sc_{i}"], atol=1e-4)


def test_decoders_match_reference_at_config_sizes():
    """The oracle against the reference's hypotheses at BASELINE.json cfg3 / cfg5 sizes (decode_cfg.npz; H=256, V=412).
    Bounded to keep the CPU suite short: A5 on the 180-frame utterance, A6 over all 249 frames, A9 on four of the 32
    utterances of 500 frames.  A7 / A8 need minutes per 500-frame utterance in the Python oracle: the oracle's beam
    decoders are pinned on the small fixture above, the CUDA ones against this fixture at full length (-m gpu)."""
    from conftest import cfg_decoder_weights
    fx = load_golden("decode_cfg.npz")
    w = cfg_decoder_weights(fx)
    blank, V = int(fx["blank"]), int(fx["V"])
    pw = {k: T(v) for k, v in w["predictor"].items()}
    jw = {k: T(v) for k, v in w["joint"].items()}
    enc = T(w["enc"])
    hy = TO.greedy_search_offline(pw, jw, blank, enc[1:2, :180], torch.tensor([180]), 64)
    assert hy[0] == fx["a5_hyp_1"].tolist()
    toks, st, last = [], None, blank
    for s in range(0, 249, 16):
        c, st, last = TO.greedy_chunk_streaming(pw, jw, blank, enc[1, s:min(s + 16, 249)], st, last, 10)
        toks += c
    assert toks == fx["a6_hyp"].tolist() and last == int(fx["a6_last"])
    pick = [0, 1, 7, 31]
    lp = T(w["synth"].ctc_logp(32, 500, V, blank))[pick]
    res = CO.ctc_prefix_beam_search(lp, fx["a9_lens"][pick], 10, blank)
    for r, i in zip(res, pick):
        assert [t for x in r["nbest"] for t in x] == fx[f"a9_nbest_flat_{i}"].tolist()
        np.testing.assert_allclose(r["nbest_scores"], fx[f"a9_nbest_scores_{i}"], rtol=1e-9, atol=1e-9)
        assert r["times"] == fx[f"a9_times_{i}"].tolist()


def test_cer_restated_matches_reference_golden():
    """oracle calculate_cer vs the outputs of the reference's rnnt_eval.calculate_cer (tests/golden/cer_small.npz)."""
    fx = load_golden("cer_small.npz")
    for i in range(int(fx["n"])):
        cer, S, D, I, N = CO.calculate_cer(fx[f"hyp_{i}"].tolist(), fx[f"ref_{i}"].tolist())
        assert [S, D, I, N] == fx[f"res_{i}"].tolist(), i
        assert abs(cer - float(fx[f"cer_{i}"])) < 1e-12


def test_predictor_restated_matches_reference_golden():
    """Section 8f row 2: the restated predictor (embed -> LSTM cells -> projection) and its gradients against what
    the reference RNNPredictor (model/component/predictor.py:43-63) produced (predictor_small.npz), one and two
    layers; and against torch's own nn.LSTM on the same weights (the library call the reference makes)."""
    fx = load_golden("predictor_small.npz")
    for tag in ("p1", "p2"):
        (V, H, L, B, U1), st, ys, r = predictor_case(fx, tag)
        pw = {k: T(v).double() for k, v in st.items()}
        out, g = TO.predictor_forward_backward(pw, T(ys), T(r))
        assert rel_l2(out.numpy(), fx[f"{tag}_out"]) < 1e-6
        for k in st:
            assert rel_l2(g[k].numpy(), fx[f"{tag}_d_{k}"]) < 2e-6, (tag, k)
        lstm = torch.nn.LSTM(H, H, L, batch_first=True).double()
        lstm.load_state_dict({k[4:]: v for k, v in pw.items() if k.startswith("rnn.")})
        y, _ = lstm(pw["embed.weight"][T(ys)])
        y = y @ pw["projection.weight"].T + pw["projection.bias"]
        assert rel_l2(y.detach().numpy(), out.numpy()) < 1e-12


def test_lstm_numpy_restatement_forward_backward():
    """oracle/lstm_oracle.py (one layer, numpy, hand-derived backward with the kernels' decomposition) against torch's
    nn.LSTM autograd in fp64 - the library call the reference makes (model/component/predictor.py:58) - with a non-zero
    initial state and cotangents on out, h_n and c_n; and, composed with the embedding and the projection, against what
    the reference RNNPredictor produced (predictor_small.npz, case p1)."""
    from oracle import lstm_oracle as LO
    rng = np.random.default_rng(3)
    for B, U1, E, H in ((3, 6, 5, 7), (2, 1, 4, 4), (4, 9, 8, 8)):
        lstm = torch.nn.LSTM(E, H, 1, batch_first=True).double()
        x, h0, c0 = (T(rng.standard_normal(s)).requires_grad_(True) for s in ((B, U1, E), (1, B, H), (1, B, H)))
        r, rh, rc = (T(rng.standard_normal(s)) for s in ((B, U1, H), (1, B, H), (1, B, H)))
        y, (hn, cn) = lstm(x, (h0, c0))
        ((y * r).sum() + (hn * rh).sum() + (cn * rc).sum()).backward()
        w = [p.detach().numpy() for p in (lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0)]
        out, hn_o, cn_o, cache = LO.lstm_layer_forward(x.detach().numpy(), *w, h0[0].detach().numpy(), c0[0].detach().numpy())
        g = LO.lstm_layer_backward(cache, r.numpy(), rh[0].numpy(), rc[0].numpy())
        for got, want in ((out, y), (hn_o, hn[0]), (cn_o, cn[0]), (g["dx"], x.grad), (g["dW_ih"], lstm.weight_ih_l0.grad),
                          (g["dW_hh"], lstm.weight_hh_l0.grad), (g["db"], lstm.bias_ih_l0.grad), (g["db"], lstm.bias_hh_l0.grad),
                          (g["dh0"], h0.grad[0]), (g["dc0"], c0.grad[0])):
            assert rel_l2(got, want.detach().numpy()) < 1e-12
    fx = load_golden("predictor_small.npz")
    (V, H, L, B, U1), st, ys, r = predictor_case(fx, "p1")
    w = {k: v.astype(np.float64) for k, v in st.items()}
    emb = w["embed.weight"][ys]
    z = np.zeros((B, H))
    out, _, _, cache = LO.lstm_layer_forward(emb, w["rnn.weight_ih_l0"], w["rnn.weight_hh_l0"], w["rnn.bias_ih_l0"],
                                             w["rnn.bias_hh_l0"], z, z)
    proj = out @ w["projection.weight"].T + w["projection.bias"]
    assert rel_l2(proj, fx["p1_out"]) < 1e-6
    g = LO.lstm_layer_backward(cache, r.astype(np.float64) @ w["projection.weight"])
    assert rel_l2(g["dW_hh"], fx["p1_d_rnn.weight_hh_l0"]) < 2e-6 and rel_l2(g["dW_ih"], fx["p1_d_rnn.weight_ih_l0"]) < 2e-6
    assert rel_l2(g["db"], fx["p1_d_rnn.bias_ih_l0"]) < 2e-6
    d_emb = np.zeros_like(w["embed.weight"])
    np.add.at(d_emb, ys, g["dx"])
    assert rel_l2(d_emb, fx["p1_d_embed.weight"]) < 2e-6


def test_split_tf32_product_keeps_fp32_level_accuracy():
    """The operand split in front of the plain GEMMs around the LSTM recurrence (split_tf32_kernel): three TF32 terms
    stacked along K keep the product within ~2^-20 of the exact one, against ~2^-11 for a plain TF32 GEMM (what the
    library LSTM uses by default) - on a product of the bench's shape class (K = 512) and on badly scaled operands."""
    from oracle import lstm_oracle as LO
    rng = np.random.default_rng(11)
    for scale in (1.0, 1e-3):
        a = (rng.standard_normal((64, 512)) * scale).astype(np.float32)
        b = rng.standard_normal((512, 48)).astype(np.float32)
        exact = a.astype(np.float64) @ b.astype(np.float64)
        e3 = np.abs(LO.split_tf32_product(a, b, 3) - exact).max() / np.abs(exact).max()
        e1 = np.abs(LO.split_tf32_product(a, b, 1) - exact).max() / np.abs(exact).max()
        assert e3 < 4e-6 and e1 > 20 * e3, (scale, e3, e1)
    # the stacked operands reproduce hi + lo exactly: nothing is lost before the GEMM
    v = rng.standard_normal(1000).astype(np.float32)
    hi = LO._tf32_trunc(v)
    assert np.array_equal(hi + (v - hi), v) and np.all((hi.view(np.uint32) & np.uint32(0x1FFF)) == 0)
