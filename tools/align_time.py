"""Dev tool: GPU time of forced alignment (CUDA events, back-to-back calls after a warm-up), one JSON line per case.

    python tools/align_time.py [--iters N]

  * cfg2 RNN-T alignment (B=32, T=250, U=40, D=512, V=412) per precision: the fused joint forward
    (ctcvr_joint_rnnt_fwd, which writes lp_blank / lp_label) and the Viterbi (ctcvr_rnnt_viterbi) timed separately;
  * cfg5 CTC alignment (B=32, T=500, U=40, V=412): ctcvr_ctc_viterbi;
  * the baseline: torchaudio.functional.forced_align looped over the cfg5 batch, on the CPU and on the GPU (host clock
    around the loop, which ends in a device synchronise; torchaudio takes one utterance per call)."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ctcvr_b200._lib import call, ptr, query, stream  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--iters", type=int, default=50)
args = ap.parse_args()
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
card = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else torch.cuda.get_device_name()


def ev(f, n=args.iters):
    for _ in range(5):
        f()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        f()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n * 1e3


def emit(**kw):
    print(json.dumps(dict(card=card, **kw)), flush=True)


dev = "cuda"
torch.manual_seed(2)
B, T, U, D, V, BLANK = 32, 250, 40, 512, 412, 0
U1 = U + 1
enc = 0.5 * torch.randn(B, T, D, device=dev)
pred = 0.5 * torch.randn(B, U1, D, device=dev)
w = torch.randn(V, D, device=dev) / D ** 0.5
bias = 0.1 * torch.randn(V, device=dev)
tgt = torch.randint(1, V, (B, U), device=dev, dtype=torch.int32)
tl = torch.full((B,), T, dtype=torch.int32, device=dev)
ul = torch.full((B,), U, dtype=torch.int32, device=dev)
lse, lpb, lpl = (torch.empty(B, T, U1, device=dev) for _ in range(3))
frames = torch.empty(B, U, dtype=torch.int32, device=dev)
tok, scores = torch.empty(B, U, device=dev), torch.empty(B, device=dev)
vws = torch.empty(max(256, query("ctcvr_rnnt_viterbi_ws_bytes", B, T, U1)), dtype=torch.uint8, device=dev)
for name, prec in (("fp32", 0), ("bf16", 1), ("bf16x3", 2)):
    fws = torch.empty(max(256, query("ctcvr_joint_rnnt_fwd_ws_bytes", B, T, U1, D, V, prec)), dtype=torch.uint8, device=dev)
    fwd = lambda: call("ctcvr_joint_rnnt_fwd", ptr(enc), ptr(pred), ptr(w), ptr(bias), ptr(tgt), ptr(tl), ptr(ul), ptr(lse),
                       ptr(lpb), ptr(lpl), B, T, U1, D, V, BLANK, prec, ptr(fws), fws.numel(), stream())
    vit = lambda: call("ctcvr_rnnt_viterbi", ptr(lpb), ptr(lpl), ptr(tl), ptr(ul), ptr(frames), ptr(tok), ptr(scores),
                       B, T, U1, ptr(vws), vws.numel(), stream())
    t_fwd = ev(fwd, 10 if prec == 0 else args.iters)
    fwd()
    t_vit = ev(vit)
    emit(case="rnnt_align_cfg2", precision=name, B=B, T=T, U=U, D=D, V=V, forward_us=round(t_fwd, 1),
         viterbi_us=round(t_vit, 1), total_us=round(t_fwd + t_vit, 1), score0=float(scores[0]))

B, T, U, V, BLANK = 32, 500, 40, 412, 5
lp = torch.log_softmax(torch.randn(B, T, V, device=dev), -1)
ys = torch.randint(6, V, (B, U), device=dev)
hl = torch.full((B,), T, dtype=torch.int32, device=dev)
yl = torch.full((B,), U, dtype=torch.int32, device=dev)
labels = torch.empty(B, T, dtype=torch.int32, device=dev)
flp, cscores = torch.empty(B, T, device=dev), torch.empty(B, device=dev)
spans = torch.empty(B, U, 2, dtype=torch.int32, device=dev)
cws = torch.empty(max(256, query("ctcvr_ctc_viterbi_ws_bytes", B, T, U)), dtype=torch.uint8, device=dev)
t_ctc = ev(lambda: call("ctcvr_ctc_viterbi", ptr(lp), ptr(ys), ptr(hl), ptr(yl), ptr(labels), ptr(flp), ptr(cscores),
                        ptr(spans), B, T, V, U, BLANK, ptr(cws), cws.numel(), stream()))
emit(case="ctc_align_cfg5", B=B, T=T, U=U, V=V, viterbi_us=round(t_ctc, 1))

import torchaudio.functional as taf  # noqa: E402
for where in ("cpu", "cuda"):
    x, y = lp.to(where), ys.int().to(where)
    loop = lambda: [taf.forced_align(x[b:b + 1], y[b:b + 1], blank=BLANK) for b in range(B)]
    loop()
    torch.cuda.synchronize()
    reps = 3
    t0 = time.perf_counter()
    for _ in range(reps):
        out = loop()
    torch.cuda.synchronize()
    t_ta = (time.perf_counter() - t0) / reps * 1e6
    same = all(torch.equal(out[b][0][0].to(dev).int(), labels[b]) for b in range(B))
    emit(case="torchaudio_forced_align_loop_cfg5", device=where, threads=torch.get_num_threads(), B=B, T=T, U=U, V=V,
         us=round(t_ta, 1), speedup_of_ctc_viterbi=round(t_ta / t_ctc, 1), labels_equal_all=same)
