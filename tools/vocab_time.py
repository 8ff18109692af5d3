"""Step time of the fused joint + RNN-T loss against the vocabulary size at cfg2 dimensions (B=32, T=250, U=40, D=512):
the graphed fwd + bwd step (GraphedJointRnntStep, tanh joint) for V in {412, 1024, 4096, 8192} x bf16 / bf16x3 with
vocab_tiling=True (V = 412 is one tile: the untiled kernels), and fp32 at V = 1024 and 4096.  One seeded batch, seeded
weights and labels drawn over the whole vocabulary; all configurations alternated in one process, CUDA events around
each step, L2 flushed (256 MiB write) before every step, each timing window at least `--seconds` long.  Reports
ms/step, utt/s and the tensor-pipe share: the algorithmic FLOPs of the joint GEMMs, 6 B T (U+1) D V (SURVEY.md (d)),
over the step time.  Prints one JSON line and, with `--out`, appends it to that file.

    python tools/vocab_time.py [--rounds 3] [--seconds 1.0] [--out profiles/r5_vocab_time.jsonl]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from bench import CFG, make_inputs  # noqa: E402
from tools.precision_time import _card  # noqa: E402

VOCABS = (412, 1024, 4096, 8192)
CONFIGS = [(v, p) for v in VOCABS for p in ("bf16", "bf16x3")] + [(1024, "fp32"), (4096, "fp32")]


def tiles(V):
    """Vocabulary tiles of the tensor-core path (csrc/joint_tc.cu vocab_tiles)."""
    return -(-((V + 31) // 32 * 32) // 416)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--out", metavar="JSONL")
    args = ap.parse_args()
    import ctcvr_b200 as C
    dev = torch.device("cuda:0")
    B, T, U, D, blank = (CFG[k] for k in ("B", "T", "U", "D", "blank"))
    enc, pred, _, tl, ul = make_inputs(1234, dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    steps, joints = {}, {}
    for V in VOCABS:
        torch.manual_seed(V)
        joints[V] = C.TransducerJoint(V, D, D, D).to(dev)
    for V, prec in CONFIGS:
        g = torch.Generator().manual_seed(V)
        tgt = torch.randint(0, V, (B, U), generator=g, dtype=torch.int32)
        tgt[tgt == blank] = (blank + 1) % V
        s = C.GraphedJointRnntStep(joints[V], B, T, U, blank, precision=prec, vocab_tiling=True)
        s.load(enc, pred, tgt.to(dev), tl, ul)
        steps[(V, prec)] = s.step

    def window(fn, n):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for a, b in ev:
            flush.zero_()
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in ev) / n

    n_of = {}
    for key, fn in steps.items():                          # warm-up and window length
        for _ in range(3):
            fn()
        n_of[key] = max(3, int(args.seconds * 1e3 / window(fn, 3)) + 1)
    assert C._lib.lib().ctcvr_debug_tc_error() == 0
    res = {key: [] for key in steps}
    for _ in range(args.rounds):
        for key in CONFIGS:                                # alternated: drift hits every configuration alike
            res[key].append(window(steps[key], n_of[key]))
    assert C._lib.lib().ctcvr_debug_tc_error() == 0
    out = {"tool": "vocab_time", "config": {k: CFG[k] for k in ("B", "T", "U", "D", "blank")}, "card": _card(),
           "mode": "graphed fwd + bwd step, tanh joint, vocab_tiling=True",
           "l2": "flushed (256 MiB write) before each step", "rounds": args.rounds,
           "tensor_pipe_share": "6 B T (U+1) D V / step time, in TFLOP/s"}
    for V, prec in CONFIGS:
        v = sorted(res[(V, prec)])
        ms = v[len(v) // 2]
        flops = 6.0 * B * T * (U + 1) * D * V
        out[f"V{V}_{prec}"] = {"ms_per_step": round(ms, 4), "utt_per_s": round(B / ms * 1e3, 1),
                               "tflops": round(flops / ms * 1e-9, 1), "tiles": tiles(V) if prec != "fp32" else None,
                               "all_ms": [round(x, 4) for x in res[(V, prec)]], "steps_per_window": n_of[(V, prec)]}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
