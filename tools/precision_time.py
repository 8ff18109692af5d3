"""Step time and accuracy of the three precisions of the fused joint + RNN-T loss at cfg2 (B=32, T=250, U=40, D=512,
V=412): one seeded batch with the weights as bench.py makes them, fwd + bwd timed eager and as a captured graph, the
three precisions alternated in one process, CUDA events around each step, L2 flushed (256 MiB write) before every step,
each timing window at least `--seconds` long.  Prints one JSON line.

    python tools/precision_time.py [--rounds 3] [--seconds 1.0] [--profile OUT.json]

`--profile` adds a torch.profiler pass (a few eager steps per precision) and writes the per-kernel CUDA time per step.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from bench import CFG, _peaks, bench_weights, make_inputs  # noqa: E402

PRECS = ("fp32", "bf16x3", "bf16")


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=10).stdout.strip().split(",")
        return {"name": out[0].strip(), "power_limit": out[1].strip()}
    except Exception:  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "power_limit": None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--profile", metavar="OUT")
    ap.add_argument("--no-parity", action="store_true")
    args = ap.parse_args()
    import ctcvr_b200 as C
    dev = torch.device("cuda:0")
    B, T, U, D, V, blank = (CFG[k] for k in ("B", "T", "U", "D", "V", "blank"))
    joint = C.TransducerJoint(V, D, D, D)
    joint.load_state_dict(bench_weights())
    joint = joint.to(dev)
    enc, pred, tgt, tl, ul = make_inputs(1234, dev)
    seed = torch.full((B,), 1.0 / B, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def eager(prec):
        e, p = enc.detach().requires_grad_(True), pred.detach().requires_grad_(True)

        def step():
            for q in joint.parameters():
                q.grad = None
            costs = joint.rnnt_loss_fused(e, p, tgt, tl, ul, blank, reduction="none", precision=prec)
            torch.autograd.backward(costs, grad_tensors=seed)
        return step

    steps = {}
    for prec in PRECS:
        steps[(prec, "eager")] = eager(prec)
        g = C.GraphedJointRnntStep(joint, B, T, U, blank, precision=prec)
        g.load(enc, pred, tgt, tl, ul)
        steps[(prec, "graph")] = g.step

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
        ms = window(fn, 3)
        n_of[key] = max(3, int(args.seconds * 1e3 / ms) + 1)
    res = {key: [] for key in steps}
    for _ in range(args.rounds):
        for mode in ("eager", "graph"):
            for prec in PRECS:                             # alternated: drift hits all three alike
                res[(prec, mode)].append(window(steps[(prec, mode)], n_of[(prec, mode)]))
    peaks = _peaks()
    cells = B * T * (U + 1)
    out = {"config": dict(CFG), "card": _card(), "l2": "flushed (256 MiB write) before each step",
           "rounds": args.rounds, "peak_tflops": peaks["tf_sust"], "peak_src": peaks["src"]}
    for prec in PRECS:
        mult = {"fp32": 0, "bf16": 1, "bf16x3": 3}[prec]
        for mode in ("eager", "graph"):
            ms = sorted(res[(prec, mode)])[len(res[(prec, mode)]) // 2]
            d = {"ms_per_step": round(ms, 4), "utt_per_s": round(B / ms * 1e3, 1), "steps_per_window": n_of[(prec, mode)],
                 "all_ms": [round(x, 4) for x in res[(prec, mode)]]}
            if mult:
                work = mult * 6.0 * cells * D * V           # tensor-core flops: logits, dZ and dW GEMMs
                d["tensor_tflops"] = round(work / ms / 1e9, 1)
                d["of_peak"] = round(work / ms / 1e9 / peaks["tf_sust"], 4)
            out[f"{prec}_{mode}"] = d
    out["speedup_bf16x3_vs_fp32"] = round(out["fp32_graph"]["ms_per_step"] / out["bf16x3_graph"]["ms_per_step"], 2)
    if not args.no_parity:
        from oracle import transducer_oracle as TO
        w = bench_weights()
        ref = TO.fused_joint_rnnt_reference_call(enc.cpu(), pred.cpu(), w, tgt.cpu(), tl.cpu(), ul.cpu(), blank)
        rk = {"enc": "d_enc_out", "pred": "d_pred_out"}
        for prec in ("bf16x3", "fp32"):
            e, p = enc.detach().requires_grad_(True), pred.detach().requires_grad_(True)
            for q in joint.parameters():
                q.grad = None
            loss = joint.rnnt_loss_fused(e, p, tgt, tl, ul, blank, reduction="mean", precision=prec)
            loss.backward()
            got = {"enc": e.grad, "pred": p.grad, **{n: q.grad for n, q in joint.named_parameters()}}
            rel = lambda a, b: float((a.double().cpu() - b.double()).norm() / b.double().norm().clamp_min(1e-30))
            out[f"parity_{prec}"] = {"loss_rel": abs(loss.item() - ref["loss"].item()) / abs(ref["loss"].item()),
                                     **{f"{k}_rel_l2": rel(v, ref[rk.get(k, "d_" + k)]) for k, v in got.items()}}
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        prof_out = {"card": out["card"], "config": dict(CFG), "note": "eager fwd+bwd, L2 flushed before each step"}
        for prec in PRECS:
            reps = 5
            with profile(activities=[ProfilerActivity.CUDA]) as pr:
                for _ in range(reps):
                    flush.zero_()
                    steps[(prec, "eager")]()
                torch.cuda.synchronize()
            k = {}
            for e_ in pr.key_averages():
                t = getattr(e_, "device_time_total", None) or getattr(e_, "cuda_time_total", 0)
                if t > 0 and "fill" not in e_.key.lower():
                    k[e_.key[:120]] = round(t / reps, 1)
            prof_out[prec] = dict(sorted(k.items(), key=lambda kv: -kv[1]))
        os.makedirs(os.path.dirname(os.path.abspath(args.profile)), exist_ok=True)
        with open(args.profile, "w") as f:
            json.dump(prof_out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
