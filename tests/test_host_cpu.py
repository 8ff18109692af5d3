"""CPU-side checks: the C-ABI library loads and exports every symbol include/ctcvr.h declares, the
host shims fail loudly without a GPU (no silent fallback), and the data-parallel step's host logic
(utterance sharding + gradient all-reduce) reproduces the single-process gradients under gloo."""
import os
import re
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import ctcvr_b200
    from ctcvr_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "ctcvr.h")).read()
    declared = set(re.findall(r"\b(ctcvr_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    l = _lib.lib()
    for name in sorted(declared):
        assert hasattr(l, name), f"libctcvr.so does not export {name}"
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    assert l.ctcvr_version() >= 100
    assert ctcvr_b200.__version__


def test_header_is_plain_c(tmp_path):
    """include/ctcvr.h is the drop-in boundary: it must compile as C99 (no C++ types, no torch) and as C++."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "hdr.c"
    src.write_text('#include "ctcvr.h"\nint main(void) { int (*f)(void) = ctcvr_version; return f == (int (*)(void))0; }\n')
    inc = os.path.join(ROOT, "include")
    for cmd in (["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I", inc, str(src)],
                ["g++", "-std=c++17", "-Wall", "-fsyntax-only", "-I", inc, "-x", "c++", str(src)]):
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr


def test_ws_queries_need_no_gpu():
    from ctcvr_b200._lib import query
    assert query("ctcvr_rnnt_loss_dense_ws_bytes", 2, 10, 5) == 5 * 2 * 10 * 5 * 4
    assert query("ctcvr_ctc_loss_ws_bytes", 2, 10, 5) > 0
    assert query("ctcvr_joint_rnnt_bwd_ws_bytes", 32, 250, 41, 512, 412, 0) > 0
    assert query("ctcvr_joint_rnnt_bwd_ws_bytes", 32, 250, 41, 512, 412, 1) > 0


def test_no_cpu_fallback():
    import ctcvr_b200 as C
    j = C.TransducerJoint(11, 8, 8, 8)
    e, p = torch.randn(1, 3, 8), torch.randn(1, 2, 8)
    with pytest.raises(RuntimeError):
        j(e, p)
    with pytest.raises(RuntimeError):
        j.rnnt_loss_fused(e, p, torch.zeros(1, 1, dtype=torch.int32), torch.tensor([3]), torch.tensor([1]), 5)
    with pytest.raises(RuntimeError):
        C.rnnt_loss(torch.randn(1, 3, 2, 11), torch.zeros(1, 1, dtype=torch.int32), torch.tensor([3], dtype=torch.int32),
                    torch.tensor([1], dtype=torch.int32), blank=5)
    with pytest.raises(RuntimeError):
        C.ctc_loss_from_logits(torch.randn(1, 3, 11), torch.zeros(1, 1, dtype=torch.long), torch.tensor([3]),
                               torch.tensor([1]), 5)
    with pytest.raises(RuntimeError):
        C.ctc_prefix_beam_search(torch.randn(1, 3, 11), torch.tensor([3]), 2, blank_id=5)
    # argument errors of the C ABI surface as RuntimeError with the library's message
    from ctcvr_b200._lib import call
    with pytest.raises(RuntimeError, match="bad dims"):
        call("ctcvr_rnnt_lattice", None, None, None, None, None, None, None, 0, 0, 0, None)


def test_module_surface_matches_reference_names():
    import ctcvr_b200 as C
    j = C.TransducerJoint(412, 256, 256, 256)
    assert list(j.state_dict()) == ["enc_ffn.weight", "enc_ffn.bias", "pred_ffn.weight", "pred_ffn.bias",
                                    "ffn_out.weight", "ffn_out.bias"]
    assert list(C.CTC(412, 256, 0.1, True, 5).state_dict()) == ["ctc_lo.weight", "ctc_lo.bias"]
    assert list(C.OnlineCTC(412, 256, 0.1, 5).state_dict()) == ["ctc_lo.weight", "ctc_lo.bias"]
    p = C.RNNPredictor(412, 256, 256, 0.1, 256, 1)
    assert list(p.state_dict()) == ["embed.weight", "rnn.weight_ih_l0", "rnn.weight_hh_l0", "rnn.bias_ih_l0",
                                    "rnn.bias_hh_l0", "projection.weight", "projection.bias"]
    ys = C.add_blank(torch.tensor([[7, 8, 0]]), 5, -1)
    assert ys.tolist() == [[5, 7, 8, 0]]


def test_bucketed_step_host_logic_and_peer_exchange_fail_loudly():
    """Host logic that needs no GPU: the bucket rounding of BucketedJointRnntStep, its refusal to run on a CPU joint,
    and PeerGradExchange / the peer entry points failing loudly (no fallback) without a process group or a device."""
    import ctypes
    import ctcvr_b200 as C
    from ctcvr_b200 import _lib
    from ctcvr_b200.dist import PeerGradExchange
    joint = C.TransducerJoint(40, 128, 128, 128)
    st = C.BucketedJointRnntStep(joint, 5, t_bucket=16, u_bucket=8)
    assert st.bucket_of(4, 1, 1) == (4, 16, 8) and st.bucket_of(4, 16, 8) == (4, 16, 8) and st.bucket_of(4, 17, 9) == (4, 32, 16)
    assert st.bucket_of(32, 250, 40) == (32, 256, 40)
    with pytest.raises(ValueError):
        C.BucketedJointRnntStep(joint, 5, t_bucket=0)
    x = torch.zeros(4, 10, 128)
    with pytest.raises(RuntimeError):                       # capture needs the joint on a CUDA device
        st.step(x, torch.zeros(4, 4, 128), torch.zeros(4, 3, dtype=torch.int32), torch.full((4,), 10, dtype=torch.int32),
                torch.full((4,), 3, dtype=torch.int32))
    with pytest.raises(RuntimeError):                       # one process per GPU: needs an initialised process group
        PeerGradExchange(1024)
    ctx, handle = ctypes.c_void_p(), ctypes.create_string_buffer(64)
    with pytest.raises(RuntimeError):                       # bad rank / world are rejected before any CUDA call
        _lib.call("ctcvr_peer_create", 3, 2, 1024, ctypes.byref(ctx), handle)
    with pytest.raises(RuntimeError):
        _lib.call("ctcvr_peer_create", 0, 9, 1024, ctypes.byref(ctx), handle)
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):                   # no device: cudaMalloc fails -> error, not a host buffer
            _lib.call("ctcvr_peer_create", 0, 2, 1024, ctypes.byref(ctx), handle)


def test_patch_install_precision_default_and_uninstall():
    """patch.install(namespace, precision=...) on stand-in modules: the patched Transducer class gets the precision
    default, uninstall restores everything; an unknown precision is rejected."""
    import types
    import ctcvr_b200 as C

    class Transducer:
        def _compute_rnnt_loss(self, *a):
            return "reference"

    ns = types.SimpleNamespace(transducer=types.SimpleNamespace(Transducer=Transducer, basic_greedy_search=lambda *a: "ref"))
    done = C.patch.install(ns, precision="bf16")
    assert "Transducer._compute_rnnt_loss" in done["transducer"] and Transducer.precision == "bf16"
    assert Transducer._compute_rnnt_loss is not None and ns.transducer.basic_greedy_search is C.basic_greedy_search
    C.patch.uninstall()
    assert not hasattr(Transducer, "precision") and Transducer()._compute_rnnt_loss() == "reference"
    assert ns.transducer.basic_greedy_search() == "ref"
    with pytest.raises(ValueError):
        C.patch.install(ns, precision="fp16")


def test_shard_bounds():
    from ctcvr_b200.dist import shard_bounds
    for n, w in ((256, 8), (10, 4), (3, 8)):
        cover = []
        for r in range(w):
            lo, hi = shard_bounds(n, w, r)
            cover += list(range(lo, hi))
        assert cover == list(range(n))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from ctcvr_b200.dist import GradAllReducer, dp_loss_and_backward, shard_bounds
    from oracle import transducer_oracle as TO
    torch.manual_seed(0)
    B, T, U, D, V, blank = 5, 9, 4, 12, 17, 5          # uneven shards: 3 + 2
    lin = {k: torch.nn.Linear(i, o) for k, (i, o) in {"enc_ffn": (D, D), "pred_ffn": (D, D), "ffn_out": (D, V)}.items()}
    params = {f"{k}.{n}": p for k, m in lin.items() for n, p in m.named_parameters()}
    enc, pred = torch.randn(B, T, D), torch.randn(B, U + 1, D)
    tgt = torch.randint(6, V, (B, U), dtype=torch.int32)
    tl = torch.tensor([9, 7, 5, 9, 3], dtype=torch.int32)
    ul = torch.tensor([4, 0, 2, 4, 1], dtype=torch.int32)
    lo, hi = shard_bounds(B, world, rank)

    def costs_fn():      # stand-in for the CUDA op: same math through the oracle's differentiable call
        logits = TO.joint_forward(enc[lo:hi], pred[lo:hi], params)
        return TO.rnnt_loss_reference_call(logits, tgt[lo:hi], tl[lo:hi], ul[lo:hi], blank, -1.0, "none")

    red = GradAllReducer(params.values())
    total = dp_loss_and_backward(costs_fn, B, red)
    if rank == 0:
        q.put((total.item(), {k: p.grad.numpy().tolist() for k, p in params.items()}))
    dist.barrier()
    dist.destroy_process_group()


def test_dp_step_matches_single_process_gloo():
    """N-rank loss/grad == 1-rank loss/grad on the concatenated batch (SURVEY.md §4 item 4)."""
    from oracle import transducer_oracle as TO
    ctx = mp.get_context("spawn")
    q = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    import time
    deadline = time.time() + 120
    while q.empty() and time.time() < deadline and any(p.is_alive() for p in procs):
        time.sleep(0.2)
    if q.empty():
        for p in procs:
            p.kill()
        pytest.fail("data-parallel workers died or timed out")
    total, grads = q.get()
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    torch.manual_seed(0)
    B, T, U, D, V, blank = 5, 9, 4, 12, 17, 5
    lin = {k: torch.nn.Linear(i, o) for k, (i, o) in {"enc_ffn": (D, D), "pred_ffn": (D, D), "ffn_out": (D, V)}.items()}
    params = {f"{k}.{n}": p for k, m in lin.items() for n, p in m.named_parameters()}
    enc, pred = torch.randn(B, T, D), torch.randn(B, U + 1, D)
    tgt = torch.randint(6, V, (B, U), dtype=torch.int32)
    tl = torch.tensor([9, 7, 5, 9, 3], dtype=torch.int32)
    ul = torch.tensor([4, 0, 2, 4, 1], dtype=torch.int32)
    loss = TO.rnnt_loss_reference_call(TO.joint_forward(enc, pred, params), tgt, tl, ul, blank, -1.0, "mean")
    loss.backward()
    assert abs(total - loss.item()) < 1e-5 * abs(loss.item())
    for k, p in params.items():
        torch.testing.assert_close(torch.tensor(grads[k]), p.grad, rtol=1e-4, atol=1e-6)


def test_predictor_lstm_host_logic_without_gpu():
    """Section 8f row 2 on a box without a GPU: the LSTM entry points are exported and validate their arguments before any
    CUDA call, the shape predicate answers from the SM-count fallback, and the Python layer refuses CPU tensors loudly
    (there is no library-LSTM fallback behind RNNPredictor)."""
    import ctcvr_b200 as C
    from ctcvr_b200 import functional as CF
    from ctcvr_b200._lib import call, query
    assert query("ctcvr_lstm_seq_supported", 32, 512) == 1 and query("ctcvr_lstm_seq_supported", 2, 256) == 1
    assert query("ctcvr_lstm_seq_supported", 1, 1184) == 1
    assert query("ctcvr_lstm_seq_supported", 32, 100000) == 0 and query("ctcvr_lstm_seq_supported", 0, 256) == 0
    # exchange buffer: 2 x [4H][roundup(B, 8)] 8-byte {value, tag} words
    assert query("ctcvr_lstm_seq_ws_bytes", 32, 512) == 2 * 4 * 512 * 32 * 8
    assert query("ctcvr_lstm_seq_ws_bytes", 2, 256) == 2 * 4 * 256 * 8 * 8
    assert query("ctcvr_lstm_seq_ws_bytes", 0, 256) == 0
    with pytest.raises(RuntimeError, match="bad dims"):
        call("ctcvr_lstm_seq_fwd", None, None, None, None, None, None, None, None, None, 0, 1, 8, None, 0, None)
    with pytest.raises(RuntimeError, match="NULL pointer"):
        call("ctcvr_lstm_seq_bwd", None, None, None, None, None, None, None, None, None, None, 2, 3, 8, None, 0, None)
    with pytest.raises(RuntimeError, match="bad arguments"):
        call("ctcvr_split_tf32", None, None, 4, 4, 1, 0, None)
    pr = C.RNNPredictor(20, 16, 16, 0.0, 16, 2, dropout=0.0)
    assert [k for k in pr.state_dict() if k.startswith("rnn.")] == [
        "rnn.weight_ih_l0", "rnn.weight_hh_l0", "rnn.bias_ih_l0", "rnn.bias_hh_l0",
        "rnn.weight_ih_l1", "rnn.weight_hh_l1", "rnn.bias_ih_l1", "rnn.bias_hh_l1"]
    with pytest.raises(RuntimeError, match="CUDA"):
        pr(torch.zeros(2, 3, dtype=torch.long))
    with pytest.raises(RuntimeError, match="CUDA"):
        pr.forward_step(torch.zeros(2, 1, dtype=torch.long), torch.zeros(2, 1), pr.init_state(2, torch.device("cpu")))
    z = torch.zeros(2, 16)
    with pytest.raises(RuntimeError, match="CUDA"):
        CF.lstm_sequence(torch.zeros(2, 3, 16), pr.rnn.weight_ih_l0, pr.rnn.weight_hh_l0, pr.rnn.bias_ih_l0,
                         pr.rnn.bias_hh_l0, z, z)
    with pytest.raises(RuntimeError):                       # the graphed step with a predictor needs a CUDA joint too
        C.GraphedJointRnntStep(C.TransducerJoint(20, 16, 16, 16), 2, 4, 3, 5, predictor=pr)
    # patch.install covers the reference predictor's forward / forward_step (model/component/predictor.py:43-63,79-98)
    import types

    class RNNPredictor(torch.nn.Module):
        def forward(self, input_tensor, cache=None):
            return "reference body"

    ns = {"predictor": types.SimpleNamespace(RNNPredictor=RNNPredictor)}
    done = C.patch.install(ns)
    try:
        assert done == {"predictor": ["RNNPredictor.forward/forward_step"]}
        assert RNNPredictor.forward is not None and RNNPredictor.forward.__name__ == "_predictor_forward"
    finally:
        C.patch.uninstall()
    assert RNNPredictor().forward(None) == "reference body" and not hasattr(RNNPredictor, "forward_step")


def test_mm3_fallback_and_precision_switch_restored(monkeypatch):
    """functional._mm3: when torch's cuBLAS precision switch cannot be set (a script that drives the legacy allow_tf32
    flag), the product falls back to a plain fp32 matmul of the UNSPLIT operands with the same transposition
    conventions; and the switch is restored after a normal block."""
    from ctcvr_b200 import functional as CF
    before = torch.backends.cuda.matmul.fp32_precision
    with CF._tf32_matmul() as t:
        assert t.ok and torch.backends.cuda.matmul.fp32_precision == "tf32"
    assert torch.backends.cuda.matmul.fp32_precision == before

    def broken_enter(self):
        self.ok, self.old = False, None
        return self

    monkeypatch.setattr(CF._tf32_matmul, "__enter__", broken_enter)
    g = torch.Generator().manual_seed(0)
    a, b = torch.randn(5, 7, generator=g), torch.randn(7, 3, generator=g)
    assert torch.allclose(CF._mm3(a, b), a @ b)
    assert torch.allclose(CF._mm3(a.t().contiguous(), b, a_t=True), a @ b)            # a given as [K, M]
    assert torch.allclose(CF._mm3(a, b.t().contiguous(), b_t=True), a @ b)            # b given as [N, K]
    out = torch.empty(5, 3)
    CF._mm3(a.t().contiguous(), b.t().contiguous(), out=out, a_t=True, b_t=True)
    assert torch.allclose(out, a @ b)
    assert torch.backends.cuda.matmul.fp32_precision == before


def test_bench_dump_outputs_float32_bounded_and_repeatable(tmp_path):
    """bench.py --dump-outputs: every output lands as float32 <name>.npy; over the byte limit the large outputs are
    cut to a seeded sample of their elements, the same one on every run, and the files stay within the limit."""
    import numpy as np
    import bench
    g = torch.Generator().manual_seed(0)
    outs = {"loss": torch.tensor(1.5), "d_w": torch.randn(40, 30, generator=g).bfloat16(),
            "d_x": torch.randn(100, 100, generator=g)}
    bench.dump_outputs(str(tmp_path / "all"), outs)
    for n, t in outs.items():
        a = np.load(tmp_path / "all" / f"{n}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, t.float().numpy())
    limit = 20000
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), outs, limit=limit)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["d_w.npy", "d_x.npy", "loss.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= limit
    a, b = np.load(tmp_path / "a" / "d_x.npy"), np.load(tmp_path / "b" / "d_x.npy")
    assert 0 < a.size < 100 * 100 and np.array_equal(a, b)
    assert np.isin(a, outs["d_x"].numpy().ravel()).all()
    assert np.array_equal(np.load(tmp_path / "a" / "loss.npy"), np.float32(1.5))
