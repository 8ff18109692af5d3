"""Step time of the fused joint + RNN-T loss per joint activation at cfg2 (B=32, T=250, U=40, D=512, V=412): the
graphed fwd + bwd step (GraphedJointRnntStep) for tanh / relu / gelu x bf16 / bf16x3, and fp32 once per activation.
One seeded batch with the weights as bench.py makes them; all configurations alternated in one process, CUDA events
around each step, L2 flushed (256 MiB write) before every step, each timing window at least `--seconds` long.  Prints
one JSON line and, with `--out`, appends it to that file.

    python tools/activation_time.py [--rounds 3] [--seconds 1.0] [--out profiles/activation_time.jsonl]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from bench import CFG, bench_weights, make_inputs  # noqa: E402
from tools.precision_time import _card  # noqa: E402

ACTS = ("tanh", "relu", "gelu")
CONFIGS = [(a, p) for a in ACTS for p in ("bf16", "bf16x3")] + [(a, "fp32") for a in ACTS]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--out", metavar="JSONL")
    args = ap.parse_args()
    import ctcvr_b200 as C
    dev = torch.device("cuda:0")
    B, T, U, D, V, blank = (CFG[k] for k in ("B", "T", "U", "D", "V", "blank"))
    enc, pred, tgt, tl, ul = make_inputs(1234, dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    steps, joints = {}, {}
    for act in ACTS:
        joint = C.TransducerJoint(V, D, D, D, activation=act)
        joint.load_state_dict(bench_weights())
        joints[act] = joint.to(dev)
    for act, prec in CONFIGS:
        g = C.GraphedJointRnntStep(joints[act], B, T, U, blank, precision=prec)
        g.load(enc, pred, tgt, tl, ul)
        steps[(act, prec)] = g.step

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
    res = {key: [] for key in steps}
    for _ in range(args.rounds):
        for key in CONFIGS:                                # alternated: drift hits every configuration alike
            res[key].append(window(steps[key], n_of[key]))
    out = {"tool": "activation_time", "config": dict(CFG), "card": _card(), "mode": "graphed fwd + bwd step",
           "l2": "flushed (256 MiB write) before each step", "rounds": args.rounds}
    for act, prec in CONFIGS:
        v = sorted(res[(act, prec)])
        out[f"{act}_{prec}"] = {"ms_per_step": round(v[len(v) // 2], 4), "all_ms": [round(x, 4) for x in res[(act, prec)]],
                                "steps_per_window": n_of[(act, prec)]}
    for prec in ("bf16", "bf16x3", "fp32"):
        base = out[f"tanh_{prec}"]["ms_per_step"]
        for act in ("relu", "gelu"):
            out[f"{act}_{prec}"]["vs_tanh"] = round(out[f"{act}_{prec}"]["ms_per_step"] / base, 3)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
