#!/usr/bin/env python
"""bench.py — fused joint + RNN-T loss forward/backward throughput (BASELINE.json `metric`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision bf16|fp32] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload = BASELINE.json configs[1]: synthetic B=32, T=250 (post-subsampling), U=40, H=D=512, V=412 per
GPU ("weak" scaling: every rank holds its own 32 utterances; the only collective is the gradient
all-reduce of the data-parallel step).  A step = joint pre-projections + fused joint/log-softmax forward
+ lattice + fused backward (+ gradient all-reduce when N>1).  `value` is measured with inputs resident in
HBM; `e2e` goes through the same public API with HOST (pinned) inputs and a device->host read of the loss
inside the timed region.  L2 is flushed (256 MiB write) before every timed step.

Beside the contract keys the line carries (rank 0, N=1): `parity` - the CPU reference run on the SAME batch and
weights, per-utterance costs compared with the GPU step; `gpu_reference` - the reference's own data flow on this GPU
through the library kernels it would use (cuBLAS + torchaudio's rnnt_loss CUDA kernels, ATen ctc_loss); `fp32` - the
reference-precision path; `eager` - the ungraphed ragged-batch public API; `predictor` - the LSTM sequence kernels of
section 8f row 2 beside the library LSTM on the same GPU; `decode` - the A4-A10 rows with RTF.

`--dump-outputs DIR` writes what the last timed step handed its caller (rank 0): the loss and the gradients of the
inputs and of the joint's parameters, as DIR/<name>.npy in float32.  Inputs and weights are seeded, so two builds run
with the same arguments can be compared output for output; compare with a tolerance, since the summation order of
d_ffn_out.bias varies from run to run (two runs of the same build on one B200 differed by 6e-5 at a magnitude of 249).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DUMP_LIMIT_BYTES = 64 * 10**6

CFG = dict(B=32, T=250, U=40, D=512, V=412, blank=5)
METRIC = "fused joint+RNN-T loss fwd/bwd throughput"
# kernels of libctcvr.so inside one captured step (bf16 activations in place), as counted by ctcvr_launch_count() on
# an eager step:
UNIT = "utt/s"


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sust=p["bf16_tflops_sustained"], src="measured")
    except Exception:
        return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self.source = "nvidia-smi"
        self._stop = threading.Event()
        self._th = threading.Thread(target=self._run, daemon=True)

    def _nvml_handle(self):
        """NVML handle of CUDA device `index` (by PCI bus id: CUDA_VISIBLE_DEVICES may renumber), or None."""
        try:
            import pynvml
            pynvml.nvmlInit()
            pr = torch.cuda.get_device_properties(self.index)
            try:
                bus = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
                h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            return pynvml, h
        except Exception:
            return None, None

    def _run(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        nv, h = self._nvml_handle()
        if nv is not None:
            # NVML in-process: a query takes ~0.1 ms, so a timed region of a few ms still gets samples (nvidia-smi: ~100 ms)
            self.source = "nvml"
            bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
            try:
                self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            except Exception:
                pass
            while not self._stop.is_set():
                try:
                    self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                    get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                    mask = int(get(h))
                    for n, b_ in bits.items():
                        if mask & b_:
                            self.reasons.add(n)
                except Exception:
                    pass
                self._stop.wait(0.001)
            return
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                f = [x.strip() for x in out.split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for n, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._th.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._th.join(timeout=2)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_min_mhz": s[0] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s), "source": self.source}


def make_inputs(seed, device, pinned=False):
    g = torch.Generator().manual_seed(seed)
    B, T, U, D, V = CFG["B"], CFG["T"], CFG["U"], CFG["D"], CFG["V"]
    enc = torch.randn(B, T, D, generator=g)
    pred = torch.randn(B, U + 1, D, generator=g)
    tgt = torch.randint(6, V, (B, U), generator=g, dtype=torch.int32)
    tl = torch.full((B,), T, dtype=torch.int32)
    ul = torch.full((B,), U, dtype=torch.int32)
    ts = [enc, pred, tgt, tl, ul]
    if pinned:
        return [t.pin_memory() for t in ts]
    return [t.to(device) for t in ts]


def bench_weights(device=None):
    """The joint of the benchmark: seed 1234, default nn.Linear init (SURVEY.md 8d).  Built on the CPU so that the GPU arm,
    the CPU reference and the GPU reference all hold the same parameters."""
    torch.manual_seed(1234)
    D, V = CFG["D"], CFG["V"]
    lin = lambda o, i: torch.nn.Linear(i, o)
    mods = {"enc_ffn": lin(D, D), "pred_ffn": lin(D, D), "ffn_out": lin(V, D)}
    return {f"{k}.{n}": p.detach().clone() for k, m in mods.items() for n, p in m.named_parameters()}


def dump_outputs(path, outputs, limit=DUMP_LIMIT_BYTES):
    """Write {name: tensor} as path/<name>.npy in float32, at most `limit` bytes in all.  Smallest first, each output
    gets an equal share of what is left; one larger than its share is replaced by a seeded sample of its flattened
    elements (in index order), so that runs with the same arguments write the same elements."""
    os.makedirs(path, exist_ok=True)
    arrays = sorted(((n, t.detach().float().cpu().numpy()) for n, t in outputs.items()), key=lambda kv: kv[1].size)
    left = limit - 256 * len(arrays)                   # room for the .npy headers
    for i, (name, a) in enumerate(arrays):
        share = left // (len(arrays) - i) // a.itemsize
        if a.size > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)
        left -= a.nbytes


def cpu_reference_step(threads, seed=1234):
    """The reference's own PyTorch CPU path for this seam (joint.py:48-69 -> torchaudio rnnt_loss -> backward),
    restated in oracle/transducer_oracle.py, on the FULL batch of the benchmark (same inputs and weights as the GPU
    arm of rank 0).  step() -> (seconds, per-utterance costs)."""
    from oracle import transducer_oracle as TO
    torch.set_num_threads(threads)
    w = bench_weights()
    enc, pred, tgt, tl, ul = make_inputs(seed, "cpu")

    def step():
        t0 = time.perf_counter()
        ws = {k: v.clone().requires_grad_(True) for k, v in w.items()}
        e, p = enc.clone().requires_grad_(True), pred.clone().requires_grad_(True)
        logits = TO.joint_forward(e, p, ws)
        costs = TO.rnnt_loss_reference_call(logits, tgt, tl, ul, CFG["blank"], -1.0, "none")
        costs.mean().backward()
        return time.perf_counter() - t0, costs.detach()
    return step


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    step = cpu_reference_step(threads)
    for _ in range(max(1, min(args.warmup, 1))):
        step()
    ts = sorted(step()[0] for _ in range(args.steps))
    sec = ts[len(ts) // 2]
    val = CFG["B"] / sec
    sample = f"the full batch of {CFG['B']} utterances per step, median of {args.steps} timed steps after 1 warm-up, torch CPU + torchaudio"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[1]: B=32,T=250,U=40,H=D=512,V=412 joint+rnnt_loss fwd/bwd (reference on the host cores)"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def gpu_reference(dev, steps=5):
    """The kernel bar of SURVEY.md 2b / 8d: the reference's data flow for this seam on THIS GPU through the library
    kernels it would run with Config.device = "cuda" - cuBLAS GEMMs + elementwise add / tanh (joint.py:48-69), torchaudio's
    sm_100 rnnt_loss kernels, autograd backward - in fp32 and under bf16 autocast.  Same inputs and weights as the GPU
    arm.  Nothing of libctcvr.so and nothing of oracle/ runs here."""
    import torchaudio
    B, T, U, D, V, blank = (CFG[k] for k in ("B", "T", "U", "D", "V", "blank"))
    w = {k: v.to(dev).requires_grad_(True) for k, v in bench_weights().items()}
    enc, pred, tgt, tl, ul = make_inputs(1234, dev)
    enc.requires_grad_(True)
    pred.requires_grad_(True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    F = torch.nn.functional
    out = {}
    for name, ac in (("fp32", False), ("autocast_bf16", True)):
        def step():
            for t in list(w.values()) + [enc, pred]:
                t.grad = None
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=ac):
                e, p = F.linear(enc, w["enc_ffn.weight"], w["enc_ffn.bias"]), F.linear(pred, w["pred_ffn.weight"], w["pred_ffn.bias"])
                logits = F.linear(torch.tanh(e.unsqueeze(2) + p.unsqueeze(1)), w["ffn_out.weight"], w["ffn_out.bias"])
            costs = torchaudio.functional.rnnt_loss(logits.float(), tgt, tl, ul, blank=blank, reduction="none")
            costs.mean().backward()
            return costs
        for _ in range(2):
            step()
        ms = []
        for _ in range(steps):
            flush.zero_()
            torch.cuda.synchronize()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            costs = step()
            s1.record()
            torch.cuda.synchronize()
            ms.append(s0.elapsed_time(s1))
        ms.sort()
        out[name] = {"ms_per_step": ms[len(ms) // 2], "value": B / (ms[len(ms) // 2] * 1e-3), "unit": UNIT,
                     "loss": float(costs.mean())}
    out["what"] = "cuBLAS + elementwise joint, torchaudio rnnt_loss CUDA kernels, autograd backward; same batch and weights"
    del flush
    torch.cuda.empty_cache()
    return out


def run_ours(args):
    import torch.distributed as dist
    import ctcvr_b200 as C
    from ctcvr_b200 import _lib
    from ctcvr_b200.dist import GradAllReducer
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.global_batch:
        # BASELINE.json configs[3] read as a strong split: a fixed global batch sharded over the ranks
        assert args.global_batch % world == 0, "--global-batch must be divisible by the number of ranks"
        CFG["B"] = args.global_batch // world
    B, T, U, D, V, blank = (CFG[k] for k in ("B", "T", "U", "D", "V", "blank"))
    joint = C.TransducerJoint(V, D, D, D)
    joint.load_state_dict(bench_weights())
    joint = joint.to(dev)
    # N > 1: the gradient sum is the last kernel of the step graph (csrc/peer_reduce.cu over NVLink peer memory), checked
    # once here against NCCL on random data; `--allreduce nccl`, a node without peer access or a failed check fall back to
    # the NCCL all-reduce launched behind the graph
    reducer, exchange, allreduce_note = None, None, None
    if world > 1:
        from ctcvr_b200.dist import PeerGradExchange
        if args.allreduce == "peer":
            try:
                exchange = PeerGradExchange(sum(p.numel() for p in joint.parameters()) + 1)
                torch.manual_seed(77 + rank)
                probe = [torch.randn(n, device=dev) for n in (V * D, V, 1, 3 * D + 2)]
                want = [x.clone() for x in probe]
                for w_ in want:
                    dist.all_reduce(w_)
                try:
                    exchange.reduce(probe)
                    torch.cuda.synchronize()
                    good = all(torch.allclose(a_, b_, rtol=1e-5, atol=1e-5) for a_, b_ in zip(probe, want))
                except RuntimeError:
                    good = False
                ok = torch.tensor([float(good)], device=dev)
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
                if float(ok) != 1.0:
                    raise RuntimeError("sums differ from NCCL's on the probe tensors")
                allreduce_note = "parameter gradients + loss summed by ONE kernel over NVLink peer memory, captured as the last node of the step graph (checked against NCCL at start-up)"
            except RuntimeError as ex_err:
                if exchange is not None:
                    exchange.close()
                exchange = None
                allreduce_note = f"NCCL behind the step graph (peer exchange unavailable: {str(ex_err)[:160]})"
        if exchange is None:
            reducer = GradAllReducer(joint.parameters())
            allreduce_note = allreduce_note or "one grouped NCCL all-reduce of the parameter gradients behind the step graph"
    enc, pred, tgt, tl, ul = make_inputs(1234 + rank, dev)
    enc.requires_grad_(True)
    pred.requires_grad_(True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    gB = B * world

    # kernels of libctcvr.so per step, counted on one eager step through the same public API (graph replays do not pass
    # through the C ABI, so the captured launches are counted here)
    l_pre = _lib.lib().ctcvr_launch_count()
    joint.rnnt_loss_fused(enc, pred, tgt, tl, ul, blank, reduction="none", precision=args.precision).sum().backward()
    torch.cuda.synchronize()
    launches_per_step = int(_lib.lib().ctcvr_launch_count() - l_pre)
    joint.zero_grad(set_to_none=True)
    enc.grad = pred.grad = None

    use_graph = not args.no_graph
    # bf16 path: the captured input buffers (and the pinned host staging of the e2e loop) are bf16 - the first kernel of
    # the path rounds its inputs to bf16 anyway
    in_dtype = torch.bfloat16 if args.precision == "bf16" else torch.float32
    gkw = dict(global_batch=gB, precision=args.precision, input_dtype=in_dtype, grad_exchange=exchange)
    graphed = C.GraphedJointRnntStep(joint, B, T, U, blank, **gkw) if use_graph else None
    if graphed is not None:
        graphed.load(enc.detach(), pred.detach(), tgt, tl, ul)

    def step(e, p, tg, tl_, ul_):
        """One training step of the seam through the public API.  Graph mode: the whole step (pre-projections, fused
        forward, lattice, fused backward, projection backward) is one captured CUDA graph; inputs are copied into its
        resident buffers (e is None = already resident)."""
        if graphed is not None:
            loss = graphed.step(e, p, tg, tl_, ul_) if e is not None else graphed.step()
        else:
            joint.zero_grad(set_to_none=True)
            e.grad = p.grad = None
            costs = joint.rnnt_loss_fused(e, p, tg, tl_, ul_, blank, reduction="none", precision=args.precision)
            loss = costs.sum() / gB
            loss.backward()
            loss = loss.detach().clone()         # no live autograd graph over the parameters after the step (graph.py)
            del costs
            if exchange is not None:
                exchange.reduce_grads(joint.parameters(), extra=[loss.view(1)])
        if reducer is not None:
            reducer.reduce()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    resident = (None, None, None, None, None) if graphed is not None else (enc, pred, tgt, tl, ul)
    for _ in range(args.warmup):
        step(*resident)
    barrier()
    l0 = _lib.lib().ctcvr_launch_count()
    with ClockSampler(local) as clk:
        # K steps between one barrier + synchronize on each side.  Every step is bracketed by its own pair of events so
        # that the L2 flush in front of it is not counted; the host does not synchronise inside the region (at N > 1 the
        # ranks pace each other through the gradient exchange, as in a train loop).
        evs = []
        for _ in range(args.steps):
            flush.zero_()
            s, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            loss = step(*resident)
            e_.record()
            evs.append((s, e_))
        barrier()
        tot_ms = sum(s.elapsed_time(e_) for s, e_ in evs)
        launches = _lib.lib().ctcvr_launch_count() - l0
        if args.dump_outputs and rank == 0:
            e_in, p_in = (graphed.enc, graphed.pred) if graphed is not None else (enc, pred)
            outs = {"loss": loss, "d_enc_out": e_in.grad, "d_pred_out": p_in.grad}
            outs.update({f"d_{n}": p.grad for n, p in joint.named_parameters()})
            dump_outputs(args.dump_outputs, outs)
        if graphed is not None:      # replays do not pass through the C ABI: the captured launches, counted above
            launches = args.steps * launches_per_step
        # ---- e2e: host (pinned) inputs -> H2D -> step -> D2H of the loss, every step.  As in a real input pipeline the
        # H2D copy of step i+1 runs on a copy stream while step i computes (double-buffered staging) and the loss of
        # step i is read back while step i+1 runs; every step still pays its own copy and its own loss read-back, and
        # the K steps are timed as one region on the wall clock.
        h = make_inputs(1234 + rank, dev, pinned=False)
        if graphed is not None:
            h[0], h[1] = h[0].to(in_dtype), h[1].to(in_dtype)
        h = [t.cpu().pin_memory() for t in h]
        h2d = sum(t.numel() * t.element_size() for t in h)
        copy_stream = torch.cuda.Stream(device=dev)
        rb_stream = torch.cuda.Stream(device=dev)
        # graph mode: one captured step per staging slot, so the H2D copies land directly in the graph's own input
        # buffers (no device-to-device copy in front of the replay); eager mode: plain staging tensors
        graphs = None
        if graphed is not None:
            graphs = [graphed, C.GraphedJointRnntStep(joint, B, T, U, blank, **gkw)]
            staging = [g.input_buffers() for g in graphs]
        else:
            staging = [[torch.empty_like(t, device=dev) for t in h] for _ in range(2)]
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [torch.cuda.Event(), torch.cuda.Event()]

        @torch.no_grad()
        def prefetch(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[i % 2])
                for dst, src in zip(staging[i % 2], h):
                    dst.copy_(src, non_blocking=True)
                ready[i % 2].record(copy_stream)

        def e2e_run(nsteps):
            """K steps; step i's loss is copied to pinned host memory right behind the step and read by the host one
            step later (after step i+1 has been enqueued), so the device never waits for the host between steps."""
            for ev in consumed:
                ev.record(torch.cuda.current_stream())
            prefetch(0)
            host_loss = torch.empty(nsteps, dtype=torch.float32).pin_memory()
            done = [torch.cuda.Event() for _ in range(nsteps)]
            losses = []
            for i in range(nsteps):
                if i + 1 < nsteps:
                    prefetch(i + 1)
                torch.cuda.current_stream().wait_event(ready[i % 2])
                d = staging[i % 2]
                if graphs is not None:
                    lv = graphs[i % 2].step()
                    if reducer is not None:
                        reducer.reduce()
                else:
                    e_in, p_in = d[0].detach().requires_grad_(True), d[1].detach().requires_grad_(True)
                    lv = step(e_in, p_in, d[2], d[3], d[4])
                consumed[i % 2].record(torch.cuda.current_stream())
                # D2H read of the step's loss, on the read-back stream: the next step's graph does not queue behind the copy
                # (each graph writes its own loss buffer, which is not rewritten before step i + 2)
                rb_stream.wait_event(consumed[i % 2])
                lv.record_stream(rb_stream)
                with torch.cuda.stream(rb_stream):
                    host_loss[i:i + 1].copy_(lv.detach().reshape(1), non_blocking=True)
                    done[i].record(rb_stream)
                if i >= 1:
                    done[i - 1].synchronize()
                    losses.append(float(host_loss[i - 1]))
            done[nsteps - 1].synchronize()
            losses.append(float(host_loss[nsteps - 1]))
            torch.cuda.synchronize()
            return losses

        e2e_run(2)
        # the box's pinned-host -> device rate for this step's inputs (explains e2e when the copy, not the step, bounds it)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(copy_stream), torch.no_grad():
            c0.record(copy_stream)
            for dst, src in zip(staging[0], h):
                dst.copy_(src, non_blocking=True)
            c1.record(copy_stream)
        torch.cuda.synchronize()
        h2d_gbps = h2d / (c0.elapsed_time(c1) * 1e-3) / 1e9
        flush.zero_()
        barrier()
        t0 = time.perf_counter()
        e2e_losses = e2e_run(args.steps)
        e2e_ms = (time.perf_counter() - t0) * 1e3
        # every e2e step stages the same batch: each loss read back from the device must be the resident step's loss
        # (the all-reduced one when the exchange sums it) - a stale or torn read-back would show here
        want = float(loss.item())
        if not all(abs(x - want) <= 1e-3 * abs(want) for x in e2e_losses):
            raise RuntimeError(f"bench.py: e2e losses {e2e_losses[:4]}.. differ from the resident step's {want}")
    ms = torch.tensor([tot_ms / args.steps, e2e_ms / args.steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step, ms_e2e = float(ms[0]), float(ms[1])

    # ---- per-kernel roofline (rank 0): time the C-ABI entry points alone with CUDA events
    line = None
    if rank == 0:
        pk = _peaks()
        kern = time_kernels(C, joint, enc, pred, tgt, tl, ul, blank, args.precision, flush)
        M = B * T * (U + 1)
        flops_bwd = 4.0 * M * D * V
        flops_fwd = 2.0 * M * D * V
        ach_bwd = flops_bwd / (kern["bwd_ms"] * 1e-3) / 1e12
        ach_fwd = flops_fwd / (kern["fwd_ms"] * 1e-3) / 1e12
        step_tf = 6.0 * M * D * V / (ms_step * 1e-3) / 1e12
        # `frac` is against the sustained cuBLAS figure (the step is a long tensor-bound region); `frac_burst` against the
        # burst figure, the right denominator for the entry points timed alone between L2 flushes
        roof = {"bound": "tensor", "kernel": "joint_rnnt_bwd (dominant)", "achieved": ach_bwd,
                "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": ach_bwd / pk["tf_sust"],
                "frac_burst": ach_bwd / pk["tf_burst"], "peak_burst": pk["tf_burst"], "traffic": None,
                "peak_source": pk["src"] + " bf16 sustained / burst",
                "step_achieved": step_tf, "step_frac": step_tf / pk["tf_sust"], "step_frac_burst": step_tf / pk["tf_burst"],
                # for information only: the tensor work the step actually EXECUTES is 8 M D V (the backward recomputes the
                # logits); `frac` / `step_frac` above count the algorithmic 4 / 6 M D V as SURVEY.md 8(d) prescribes
                "step_executed_frac": (8.0 / 6.0) * step_tf / pk["tf_sust"],
                "fwd": {"achieved": ach_fwd, "frac": ach_fwd / pk["tf_sust"], "frac_burst": ach_fwd / pk["tf_burst"],
                        "ms": kern["fwd_ms"]},
                "bwd": {"achieved": ach_bwd, "frac": ach_bwd / pk["tf_sust"], "frac_burst": ach_bwd / pk["tf_burst"],
                        "ms": kern["bwd_ms"]},
                "lattice": {"ms": kern["lat_ms"], "achieved_GBps": 24.0 * M / (kern["lat_ms"] * 1e-3) / 1e9,
                            "frac_hbm": 24.0 * M / (kern["lat_ms"] * 1e-3) / 1e9 / pk["hbm"]}}
        roof.update(_ncu_traffic())
        line = {"metric": METRIC, "value": gB / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if args.global_batch else "weak",
                "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
                "config": {"workload": (f"configs[3] strong split: global B={gB} ({B}/GPU),T=250,U=40,H=D=512,V=412 fused joint+rnnt_loss fwd/bwd"
                                        if args.global_batch else
                                        "configs[1]: B=32/GPU,T=250,U=40,H=D=512,V=412 fused joint+rnnt_loss fwd/bwd"),
                           "global_batch": gB, "parallelism": f"dp{world}", "l2": "flushed (256 MiB write) before each step",
                           "precision": args.precision, "cuda_graph": bool(graphed is not None),
                           "allreduce": allreduce_note},
                "e2e": {"value": gB / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                        "loss_checked_every_step": True,
                        "input_dtype": str(in_dtype).replace("torch.", "") if graphed is not None else "float32",
                        "h2d_GBps_measured": h2d_gbps, "h2d_ms_per_step": h2d / (h2d_gbps * 1e9) * 1e3},
                "gpu_launches": int(launches), "gpu_launches_per_step": launches_per_step, "roofline": roof,
                "clocks": clk.summary(), "loss": float(loss.item()) * (1 if exchange is not None else world)}
        if world == 1 and not args.global_batch:
            # ---- the CPU reference on the SAME batch and weights: baseline timing (full batch, median of 3 after one
            # warm-up) and the parity check that rides in every record
            threads = os.cpu_count() or 1
            cstep = cpu_reference_step(threads)
            cstep()
            runs = sorted((cstep() for _ in range(3)), key=lambda r: r[0])
            csec, ccosts = runs[1]
            line["cpu_baseline"] = {"value": B / csec, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"the full batch of {B} utterances per step, median of 3 after 1 warm-up, torch CPU + torchaudio"}
            par = {"reference": "oracle: joint.py:48-69 + torchaudio.functional.rnnt_loss on the host, same batch and weights",
                   "tolerance": {"fp32": 1e-4, "bf16": 2e-3}}
            for prec in ("fp32", "bf16"):
                with torch.no_grad():
                    g = joint.rnnt_loss_fused(enc.detach(), pred.detach(), tgt, tl, ul, blank, reduction="none", precision=prec).cpu()
                rel = float(((g - ccosts).abs() / ccosts.abs()).max())
                par[prec] = {"max_rel_err_per_utterance_cost": rel, "loss": float(g.mean()), "ok": bool(rel <= par["tolerance"][prec])}
            par["reference_loss"] = float(ccosts.mean())
            par["step_loss_rel_err"] = abs(line["loss"] - par["reference_loss"]) / abs(par["reference_loss"])
            line["parity"] = par
            if not (par["fp32"]["ok"] and par["bf16"]["ok"]):
                raise RuntimeError(f"bench.py: the GPU costs disagree with the CPU reference on the benchmark batch: {par}")
            # ---- the reference-precision path (fp32 SIMT kernels, 1e-4): its own step time and denominator
            line["fp32"] = time_fp32_step(C, joint, B, T, U, blank, enc, pred, tgt, tl, ul, flush)
            # ---- the ungraphed public API on a ragged batch (what a train loop with varying shapes hits)
            line["eager"], line["bucketed"] = time_ragged(C, joint, enc, pred, tgt, blank, args.precision, flush, in_dtype)
            line["gpu_reference"] = gpu_reference(dev)
            line["gpu_reference"]["speedup_vs_fp32"] = line["value"] / line["gpu_reference"]["fp32"]["value"]
            line["gpu_reference"]["speedup_vs_autocast_bf16"] = line["value"] / line["gpu_reference"]["autocast_bf16"]["value"]
            try:        # a side row: it must not cost the record its headline
                line["predictor"] = time_predictor(C, B, U + 1, D)
                line["predictor"]["step_with_predictor"] = time_step_with_predictor(C, joint, B, T, U, D, V, blank, args.precision,
                                                                                     enc, tgt, tl, ul, flush)
            except Exception as e:  # noqa: BLE001
                line.setdefault("predictor", {})["error"] = f"{type(e).__name__}: {e}"[:300]
            if not args.no_decode:
                import bench_decode
                line["decode"] = bench_decode.run_rows(quick=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line))


def cpu_lstm_baseline(B, U1, H, reps=3):
    """The reference's own arithmetic for the predictor row: torch's nn.LSTM forward + backward on the host cores
    (model/component/predictor.py:58 runs exactly this call), all threads, median of `reps` after one warm-up."""
    import torch
    g = torch.Generator().manual_seed(4321)
    lstm = torch.nn.LSTM(H, H, 1, batch_first=True)
    x = torch.randn(B, U1, H, generator=g, requires_grad=True)
    r = torch.randn(B, U1, H, generator=g)
    ts = []
    for i in range(reps + 1):
        t0 = time.perf_counter()
        torch.autograd.backward(lstm(x)[0], r)
        dt = time.perf_counter() - t0
        x.grad = None
        lstm.zero_grad(set_to_none=True)
        if i:
            ts.append(dt)
    ts.sort()
    return {"ms": ts[len(ts) // 2] * 1e3, "cores": torch.get_num_threads(), "kind": "reference arithmetic (torch CPU nn.LSTM)",
            "sample": f"the full batch, median of {reps} after 1 warm-up"}


def time_predictor(C, B, U1, H, iters=20):
    """SURVEY.md section 8f row 2: the predictor's LSTM over the label sequence (model/component/predictor.py:58) at the
    bench shape, forward + backward with gradients of the input and of all four parameters.  `ours` = the persistent
    sequence kernels (csrc/lstm_seq.cu, fp32) + their four plain GEMMs; `library` = torch's nn.LSTM on this GPU (cuDNN,
    TF32 allowed by torch's default).  Both eager and replayed from a CUDA graph; CUDA events, median.  Parity: both
    outputs against torch's fp32 CPU LSTM - the arithmetic the reference runs - on the same weights and input."""
    import torch
    from ctcvr_b200 import functional as CF
    g = torch.Generator().manual_seed(4321)
    cpu = torch.nn.LSTM(H, H, 1, batch_first=True)
    x_c = torch.randn(B, U1, H, generator=g)
    with torch.no_grad():
        want = cpu(x_c)[0]
    lstm = torch.nn.LSTM(H, H, 1, batch_first=True).cuda()
    lstm.load_state_dict(cpu.state_dict())
    x = x_c.cuda().requires_grad_(True)
    h0 = torch.zeros(1, B, H, device="cuda")
    c0 = torch.zeros(1, B, H, device="cuda")
    r = torch.randn(B, U1, H, device="cuda")
    ps = [lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0]

    def clear():
        x.grad = None
        for p in ps:
            p.grad = None

    def ours():
        torch.autograd.backward(CF.lstm_sequence(x, *ps, h0[0], c0[0])[0], r)
        clear()

    def library():
        torch.autograd.backward(lstm(x, (h0, c0))[0], r)
        clear()

    def timed(fn):
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(iters + 1)]
        ev[0].record()
        for i in range(iters):
            fn()
            ev[i + 1].record()
        torch.cuda.synchronize()
        ts = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(iters))
        return ts[len(ts) // 2]

    with torch.no_grad():
        err_ours = float((CF.lstm_sequence(x, *ps, h0[0], c0[0])[0].cpu() - want).abs().max() / want.abs().max())
        err_lib = float((lstm(x, (h0, c0))[0].cpu() - want).abs().max() / want.abs().max())
    n0 = C._lib.lib().ctcvr_launch_count()
    ours()
    res = {"workload": f"LSTM layer fwd+bwd, B={B}, U+1={U1}, E=H={H}, fp32", "unit": "ms per fwd+bwd",
           "kernel_launches_per_call": int(C._lib.lib().ctcvr_launch_count() - n0),
           "max_abs_err_over_max_vs_cpu_fp32": {"ours": err_ours, "library_cudnn": err_lib}}
    if err_ours > 1e-4:
        raise RuntimeError(f"bench.py: the LSTM sequence kernels disagree with the CPU LSTM: {err_ours}")
    for name, fn in (("ours", ours), ("library_cudnn", library)):
        row = {"eager": round(timed(fn), 4)}
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            fn()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        try:
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                fn()
            row["graphed"] = round(timed(gr.replay), 4)
            del gr
        except Exception as e:  # noqa: BLE001
            row["graphed"] = None
            row["graph_error"] = type(e).__name__
            torch.cuda.synchronize()
        res[name] = row
    res["utt_per_s_ours_graphed"] = B / (res["ours"]["graphed"] * 1e-3) if res["ours"].get("graphed") else None
    res["cpu_baseline"] = cpu_lstm_baseline(B, U1, H)
    return res


def time_step_with_predictor(C, joint, B, T, U, D, V, blank, precision, enc, tgt, tl, ul, flush, reps=10):
    """The bench step with the label side inside the captured graph: add_blank -> RNNPredictor (embedding, LSTM sequence
    kernels, projection) -> fused joint / loss -> backward through all of it (13 parameter tensors, 13.2 MB of
    gradients: SURVEY.md section 8(e)'s data-parallel payload).  Same batch as the headline; L2 flushed before every
    timed replay; CUDA events, median."""
    import torch
    pr = C.RNNPredictor(V, D, D, 0.0, D, 1, dropout=0.0).to(enc.device)
    g = C.GraphedJointRnntStep(joint, B, T, U, blank, precision=precision, predictor=pr)
    g.load(enc.detach(), None, tgt, tl, ul)
    ts = []
    for i in range(reps + 2):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = g.step()
        e1.record()
        torch.cuda.synchronize()
        if i >= 2:
            ts.append(e0.elapsed_time(e1))
    ts.sort()
    ms = ts[len(ts) // 2]
    nbytes = sum(p.numel() for p in g.parameters()) * 4
    out = {"ms_per_step": ms, "value": B / (ms * 1e-3), "unit": UNIT, "loss": float(loss),
           "gradient_bytes": nbytes, "precision": precision}
    for p in pr.parameters():
        p.grad = None
    del g
    return out


def time_fp32_step(C, joint, B, T, U, blank, enc, pred, tgt, tl, ul, flush, reps=3):
    """precision='fp32': the SIMT kernels that meet the reference's 1e-4.  Denominator: the fp32 FMA peak of the chip
    (148 SMs x 128 lanes x 2 flop x max SM clock), since this path does not touch the tensor cores."""
    e, p = enc.detach().clone().requires_grad_(True), pred.detach().clone().requires_grad_(True)

    def step():
        joint.zero_grad(set_to_none=True)
        e.grad = p.grad = None
        joint.rnnt_loss_fused(e, p, tgt, tl, ul, blank, reduction="none", precision="fp32").sum().div(B).backward()
    step()
    ms = []
    for _ in range(reps):
        flush.zero_()
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        step()
        s1.record()
        torch.cuda.synchronize()
        ms.append(s0.elapsed_time(s1))
    ms.sort()
    med = ms[len(ms) // 2]
    joint.zero_grad(set_to_none=True)
    flops = 8.0 * B * T * (U + 1) * CFG["D"] * CFG["V"]          # executed: fwd 2 + bwd (recompute 2 + dZ 2 + dW 2)
    peak = 148 * 128 * 2 * 1.965e9 / 1e12
    return {"value": B / (med * 1e-3), "unit": UNIT, "ms_per_step": med, "tolerance": 1e-4,
            "roofline": {"bound": "fp32 FMA pipe", "achieved": flops / (med * 1e-3) / 1e12, "peak": peak, "unit": "TFLOP/s",
                         "frac": flops / (med * 1e-3) / 1e12 / peak, "peak_source": "nominal 148 SM x 128 FMA x 2 x 1.965 GHz",
                         "flops": "executed (incl. the logits recompute)"}}


def time_ragged(C, joint, enc, pred, tgt, blank, precision, flush, in_dtype, reps=3):
    """A train loop whose batches change shape: six ragged batches (T_b ~ U[Tmax/2, Tmax], U_b ~ U[Umax/2, Umax], the
    batch maxima Tmax in 229..250 and Umax in 36..40, element 0 at the maximum), stepped (a) through the ungraphed public
    op - new workspaces and ~40 launches per call - and (b) through BucketedJointRnntStep (T rounded up to 16 frames, U to
    8 labels: two captured graphs serve the six shapes).  Median step time over `reps` passes after one warm-up pass."""
    B, T = enc.shape[0], enc.shape[1]
    U = tgt.shape[1]
    g = torch.Generator().manual_seed(99)
    batches, cells = [], 0
    for Tm, Um in ((250, 40), (238, 37), (245, 39), (250, 40), (229, 36), (241, 38)):
        Tm, Um = min(Tm, T), min(Um, U)
        tl = torch.randint(Tm // 2, Tm + 1, (B,), generator=g, dtype=torch.int32)
        ul = torch.randint(Um // 2, Um + 1, (B,), generator=g, dtype=torch.int32)
        tl[0], ul[0] = Tm, Um
        cells += int(((tl.long()) * (ul.long() + 1)).sum())
        batches.append((enc.detach()[:, :Tm].contiguous(), pred.detach()[:, :Um + 1].contiguous(), tgt[:, :Um].contiguous(),
                        tl.to(enc.device), ul.to(enc.device)))

    def timed(step_fn):
        for b_ in batches:
            step_fn(*b_)
        ms = []
        for _ in range(reps):
            for b_ in batches:
                flush.zero_()
                torch.cuda.synchronize()
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record()
                step_fn(*b_)
                s1.record()
                torch.cuda.synchronize()
                ms.append(s0.elapsed_time(s1))
        ms.sort()
        return ms[len(ms) // 2]

    def eager_step(e, p, tg, tl, ul):
        joint.zero_grad(set_to_none=True)
        e, p = e.requires_grad_(True), p.requires_grad_(True)
        e.grad = p.grad = None
        joint.rnnt_loss_fused(e, p, tg, tl, ul, blank, reduction="mean", precision=precision).backward()

    med_e = timed(eager_step)
    for e, p, *_ in batches:
        e.requires_grad_(False)
        p.requires_grad_(False)
        e.grad = p.grad = None
    joint.zero_grad(set_to_none=True)
    stepper = C.BucketedJointRnntStep(joint, blank, t_bucket=16, u_bucket=8, precision=precision, input_dtype=in_dtype)
    med_b = timed(stepper.step)
    joint.zero_grad(set_to_none=True)
    frac = cells / float(len(batches) * B * T * (U + 1))
    common = {"unit": UNIT, "lattice_cells_per_step": cells // len(batches), "cells_vs_full_batch": frac}
    return ({"value": B / (med_e * 1e-3), "ms_per_step": med_e, "what": "ungraphed rnnt_loss_fused + backward, six ragged batch shapes", **common},
            {"value": B / (med_b * 1e-3), "ms_per_step": med_b, "graphs_captured": stepper.captures,
             "what": "BucketedJointRnntStep (shape-bucketed CUDA graph cache, input copy included), same six ragged batch shapes", **common})


def _ncu_traffic():
    """DRAM bytes (read + write) per call of the backward entry point's tensor-core kernels, from the newest committed
    `ncu --set full` capture (profiles/r*_traffic.json: it names the commit it was taken at).  ncu cannot run inside a
    timed benchmark, so this is a recorded measurement of the same code, not a live one."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
    for path in reversed(files):
        try:
            d = json.load(open(path))
            k = d["kernels"]
            names = [n for n in k if n.startswith("joint_bwd") or n.startswith("dw_gemm")]
            return {"traffic": float(sum(k[n]["dram_read_bytes"] + k[n]["dram_write_bytes"] for n in names)),
                    "traffic_source": os.path.basename(path) + " (" + str(d.get("commit", "?")) + "): " + ", ".join(names)}
        except (OSError, KeyError, ValueError):
            continue
    return {"traffic": None}


def time_kernels(C, joint, enc, pred, tgt, tl, ul, blank, precision, flush, reps=5):
    from ctcvr_b200._lib import call, ptr, query, stream
    prec = {"fp32": 0, "bf16": 1}[precision]
    with torch.no_grad():
        e, p = joint.project(enc.detach(), pred.detach())
        e, p = e.contiguous(), p.contiguous()
        w, b = joint.ffn_out.weight.detach().contiguous(), joint.ffn_out.bias.detach().contiguous()
    B, T, D = e.shape
    U1, V = p.shape[1], w.shape[0]
    dev = e.device
    lse = torch.empty(B, T, U1, device=dev)
    lpb, lpl, al, be = (torch.empty_like(lse) for _ in range(4))
    costs = torch.empty(B, device=dev)
    gc = torch.full((B,), 1.0 / B, device=dev)
    d_e, d_p, d_w, d_b = torch.empty_like(e), torch.empty_like(p), torch.empty_like(w), torch.empty_like(b)
    wsf = torch.empty(max(256, query("ctcvr_joint_rnnt_fwd_ws_bytes", B, T, U1, D, V, prec)), dtype=torch.uint8, device=dev)
    wsb = torch.empty(max(256, query("ctcvr_joint_rnnt_bwd_ws_bytes", B, T, U1, D, V, prec)), dtype=torch.uint8, device=dev)

    def fwd():
        call("ctcvr_joint_rnnt_fwd", ptr(e), ptr(p), ptr(w), ptr(b), ptr(tgt), ptr(tl), ptr(ul), ptr(lse), ptr(lpb),
             ptr(lpl), B, T, U1, D, V, blank, prec, ptr(wsf), wsf.numel(), stream())

    def lat():
        call("ctcvr_rnnt_lattice", ptr(lpb), ptr(lpl), ptr(tl), ptr(ul), ptr(al), ptr(be), ptr(costs), B, T, U1, stream())

    def bwd():
        call("ctcvr_joint_rnnt_bwd", ptr(e), ptr(p), ptr(w), ptr(b), ptr(tgt), ptr(tl), ptr(ul), ptr(lse), ptr(lpb), ptr(lpl), ptr(al),
             ptr(be), ptr(costs), ptr(gc), -1.0, ptr(d_e), ptr(d_p), ptr(d_w), ptr(d_b), B, T, U1, D, V, blank, prec,
             ptr(wsb), wsb.numel(), stream())

    out = {}
    for name, fn in (("fwd_ms", fwd), ("lat_ms", lat), ("bwd_ms", bwd)):
        fn()
        tot = 0.0
        for _ in range(reps):
            flush.zero_()
            s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            t.record()
            torch.cuda.synchronize()
            tot += s.elapsed_time(t)
        out[name] = tot / reps
    return out


def main():
    sys.dont_write_bytecode = True      # the tree may be read-only: the benchmark writes nothing into it
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-graph", action="store_true", help="eager step instead of the captured CUDA graph")
    ap.add_argument("--precision", default=os.environ.get("CTCVR_PRECISION", "bf16"), choices=["bf16", "fp32"])
    ap.add_argument("--global-batch", type=int, default=0,
                    help="strong scaling (configs[3]): fixed global batch split over the ranks; the headline extras are skipped")
    ap.add_argument("--allreduce", default="peer", choices=["peer", "nccl"],
                    help="N>1: gradient sum by the in-graph NVLink peer kernel (default) or by NCCL behind the graph")
    ap.add_argument("--no-decode", action="store_true", help="skip the A4-A10 rows (bench_decode.py) in the JSON line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and gradients of the last timed step as DIR/<name>.npy (float32, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        args.warmup = max(args.warmup, 3)
        run_ours(args)


if __name__ == "__main__":
    main()
