"""Dev tool: GPU time (CUDA events, 50 back-to-back calls) of the CTC entry points at cfg5 (B=32, T=500, V=412, U=40).

    python tools/ctc_time.py [--against OTHER/libctcvr.so] [--rounds N]

With --against, the in-tree library and another build of it are timed in alternating rounds in one process, and their
costs and gradients on the same inputs are compared bit for bit."""
import argparse, ctypes, json, os, subprocess, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ctcvr_b200 import _lib
from ctcvr_b200._lib import ptr, stream
ap = argparse.ArgumentParser()
ap.add_argument("--against", default=None)
ap.add_argument("--rounds", type=int, default=1)
args = ap.parse_args()
libs = {"tree": _lib.lib()}
if args.against:
    other = ctypes.CDLL(os.path.abspath(args.against))
    for name, (res, argt) in _lib._SIGS.items():
        if hasattr(other, name):
            fn = getattr(other, name)
            fn.restype, fn.argtypes = res, argt
    libs["against"] = other
torch.manual_seed(5)
B, T, V, U, BLANK = 32, 500, 412, 40, 5
x = torch.randn(B, T, V, device="cuda"); lp = torch.empty_like(x)
ys = torch.randint(6, V, (B, U), device="cuda"); hl = torch.full((B,), T, dtype=torch.int32, device="cuda"); yl = torch.full((B,), U, dtype=torch.int32, device="cuda")
out = {k: (torch.empty(B, device="cuda"), torch.empty_like(x)) for k in libs}
ws = torch.empty(libs["tree"].ctcvr_ctc_loss_ws_bytes(B, T, U), dtype=torch.uint8, device="cuda")
def call(l, name, *a):
    if getattr(l, name)(*a) != 0:
        raise RuntimeError(f"{name}: {l.ctcvr_last_error().decode()}")
def ev(f, n=50):
    for _ in range(5): f()
    torch.cuda.synchronize(); a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n): f()
    b.record(); torch.cuda.synchronize(); return a.elapsed_time(b) / n * 1e3
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
card = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else torch.cuda.get_device_name()
for r in range(args.rounds):
    for k, l in libs.items():
        nll, grad = out[k]
        t_ls = ev(lambda: call(l, "ctcvr_log_softmax", ptr(x), ptr(lp), B * T, V, stream()))
        t_ab = ev(lambda: call(l, "ctcvr_ctc_loss", ptr(lp), ptr(ys), ptr(hl), ptr(yl), None, ptr(nll), None, B, T, V, U, BLANK, 1, ptr(ws), ws.numel(), stream()))
        t_all = ev(lambda: call(l, "ctcvr_ctc_loss", ptr(lp), ptr(ys), ptr(hl), ptr(yl), None, ptr(nll), ptr(grad), B, T, V, U, BLANK, 1, ptr(ws), ws.numel(), stream()))
        print(json.dumps({"lib": k, "round": r, "card": card, "log_softmax_us": round(t_ls, 1), "alpha_beta_us": round(t_ab, 1),
                          "alpha_beta_plus_grad_us": round(t_all, 1), "nll0": float(nll[0])}))
if args.against:
    print(json.dumps({"costs_bit_identical": torch.equal(out["tree"][0], out["against"][0]),
                      "grads_bit_identical": torch.equal(out["tree"][1], out["against"][1])}))
