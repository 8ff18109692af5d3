"""On-device RNN-T decoders behind the reference's decode call surface.

  basic_greedy_search(model, encoder_out, encoder_out_lens, n_steps=64) -> List[List[int]]
      model/component/transducer.py:22-70 (and wenet/transducer/search/greedy_search.py:6-54)
  greedy_chunk(model_parts, encoder_out_chunk, states, prev_token, n_steps=10)
      the loop of OnlineRNNTModel._decode_chunk_streaming_logic (model/online_rnnt_model.py:193-222)
  beam_chunk_online(...)   model/online_rnnt_model.py:389-522        (A7)
  prefix_beam_search(...)  wenet/transducer/search/prefix_beam_search.py:42-148  (A8)

`model` only needs `.predictor` (embed, rnn, projection), `.joint` (enc_ffn, pred_ffn, ffn_out) and
`.blank` / `.blank_id`, i.e. the reference's own modules work as well as the mirrors in this package.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Tuple

import torch

from . import _lib
from ._lib import DecoderWeights, call, ptr, query, stream
from .functional import _ACT
from .joint import joint_activation


class PreparedDecoder:
    """Device-side weight layouts of `ctcvr_decoder_weights` (include/ctcvr.h), derived once per
    parameter version (re-derived automatically after an optimizer step / load_state_dict)."""

    def __init__(self, predictor, joint):
        self.predictor, self.joint = predictor, joint
        self._key = None
        self._keep = None
        self.struct = None

    def _version_key(self):
        ps = list(self.predictor.parameters()) + list(self.joint.parameters())
        return tuple((p.data_ptr(), p._version) for p in ps)

    @torch.no_grad()
    def get(self) -> DecoderWeights:
        key = self._version_key()
        if key == self._key:
            return self.struct
        p, j = self.predictor, self.joint
        rnn = p.rnn
        L, H = rnn.num_layers, rnn.hidden_size
        f = lambda t: t.detach().float().contiguous()
        emb = f(p.embed.weight)
        if not emb.is_cuda:
            raise RuntimeError("ctcvr_b200 decoders run on CUDA (B200) only; move the model to the GPU")
        bias = lambda l, n: (f(getattr(rnn, f"{n}_l{l}")) if rnn.bias else torch.zeros(4 * H, device=emb.device))
        gate_tok = torch.addmm(bias(0, "bias_ih") + bias(0, "bias_hh"), emb, f(rnn.weight_ih_l0).t()).contiguous()
        w_hh_t = torch.stack([f(getattr(rnn, f"weight_hh_l{l}")).t().contiguous() for l in range(L)]).contiguous()
        if L > 1:
            w_ih_t = torch.stack([f(getattr(rnn, f"weight_ih_l{l}")).t().contiguous() for l in range(1, L)]).contiguous()
            b_gate = torch.stack([bias(l, "bias_ih") + bias(l, "bias_hh") for l in range(1, L)]).contiguous()
        else:
            w_ih_t = b_gate = None
        proj_t, proj_b = f(p.projection.weight).t().contiguous(), f(p.projection.bias)
        if j.pred_ffn is not None:
            pf_t, pf_b = f(j.pred_ffn.weight).t().contiguous(), f(j.pred_ffn.bias)
        else:   # prejoin_linear=False: identity
            P = proj_t.shape[1]
            pf_t, pf_b = torch.eye(P, device=emb.device), torch.zeros(P, device=emb.device)
        post = _post_ffn(j)
        if post is not None:    # post(e + p) = post(e) + W_post p: the prediction side takes W_post without its bias
            wp = f(post.weight)
            pf_t, pf_b = (pf_t @ wp.t()).contiguous(), (wp @ pf_b).contiguous()
        out_t, out_b = f(j.ffn_out.weight).t().contiguous(), f(j.ffn_out.bias)
        self._keep = (gate_tok, w_hh_t, w_ih_t, b_gate, proj_t, proj_b, pf_t, pf_b, out_t, out_b)
        s = DecoderWeights()
        for name, t in zip(("gate_tok", "w_hh_t", "w_ih_t", "b_gate", "proj_t", "proj_b", "pred_ffn_t",
                            "pred_ffn_b", "out_t", "out_b"), self._keep):
            setattr(s, name, None if t is None else t.data_ptr())
        s.V, s.H, s.L, s.P, s.D = out_t.shape[1], H, L, proj_t.shape[1], out_t.shape[0]
        s.activation = _ACT[joint_activation(j)]
        self.struct, self._key = s, key
        return s


def _prepared(model) -> PreparedDecoder:
    pd = getattr(model, "_ctcvr_prepared", None)
    if pd is None or pd.predictor is not model.predictor or pd.joint is not model.joint:
        pd = PreparedDecoder(model.predictor, model.joint)
        try:
            object.__setattr__(model, "_ctcvr_prepared", pd)
        except Exception:
            pass
    return pd


def _blank_of(model) -> int:
    return int(model.blank if hasattr(model, "blank") else model.blank_id)


def _post_ffn(joint):
    """The post-join linear of a joint that applies one (joint.py:64-65), else None."""
    return joint.post_ffn if getattr(joint, "postjoin_linear", False) and getattr(joint, "post_ffn", None) is not None \
        else None


def _enc_proj(model, encoder_out):
    j = model.joint
    x = encoder_out.float()
    if getattr(j, "enc_ffn", None) is not None:
        x = torch.nn.functional.linear(x, j.enc_ffn.weight, j.enc_ffn.bias)
    post = _post_ffn(j)
    if post is not None:    # the encoder side of the folded post-join linear keeps its bias
        x = torch.nn.functional.linear(x, post.weight.float(), post.bias.float())
    return x.contiguous()


@torch.no_grad()
def greedy_batch(model, encoder_out, encoder_out_lens, n_steps: int, h=None, c=None, last_token=None):
    """Run the greedy walk for N utterances/streams at once.  Returns (hyps, h, c, last_token) with the
    predictor state after the walk ([L,N,H]) and the last emitted token per stream."""
    w = _prepared(model).get()
    blank = _blank_of(model)
    ep = _enc_proj(model, encoder_out)
    N, T, D = ep.shape
    dev = ep.device
    lens = encoder_out_lens.to(device=dev, dtype=torch.int32).contiguous()
    if h is None:
        h = torch.zeros((w.L, N, w.H), dtype=torch.float32, device=dev)
        c = torch.zeros_like(h)
    else:
        h, c = h.detach().float().contiguous().clone(), c.detach().float().contiguous().clone()
    if last_token is None:
        last_token = torch.full((N,), blank, dtype=torch.int32, device=dev)
    else:
        last_token = last_token.to(device=dev, dtype=torch.int32).contiguous().clone()
    max_out = T * n_steps
    toks = torch.empty((N, max_out), dtype=torch.int32, device=dev)
    nout = torch.empty((N,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        call("ctcvr_rnnt_greedy", ctypes.byref(w), ptr(ep), ptr(lens), ptr(h), ptr(c), ptr(last_token), ptr(toks),
             ptr(nout), N, T, max_out, blank, int(n_steps), None, 0, stream())
    nh = nout.cpu().tolist()
    width = max(nh) if N > 0 else 0
    th = toks[:, :max(width, 1)].cpu().numpy()          # numpy rows: per-utterance slicing of a torch tensor costs ~5 us each
    hyps = [th[i, :nh[i]].tolist() for i in range(N)]
    return hyps, h, c, last_token


def basic_greedy_search(model, encoder_out: torch.Tensor, encoder_out_lens: torch.Tensor,
                        n_steps: int = 64) -> List[List[int]]:
    """Drop-in for model/component/transducer.py:22-70: all utterances decoded by one kernel launch,
    one device->host copy of the hypotheses at the end (the reference syncs once per step)."""
    return greedy_batch(model, encoder_out, encoder_out_lens, n_steps)[0]


@torch.no_grad()
def greedy_chunk(model, encoder_out_chunk: torch.Tensor, predictor_states: Optional[List[torch.Tensor]],
                 prev_token: int, n_steps: int = 10) -> Tuple[List[int], List[torch.Tensor], int]:
    """The search loop of model/online_rnnt_model.py:193-222 for one encoder chunk [1,Tc,H]:
    returns (tokens, [h,c], last_token)."""
    dev = encoder_out_chunk.device
    Tc = encoder_out_chunk.size(1)
    if predictor_states is None:
        predictor_states = model.predictor.init_state(batch_size=1, device=dev)
    if Tc == 0:
        return [], predictor_states, prev_token
    lens = torch.tensor([Tc], dtype=torch.int32, device=dev)
    last = torch.tensor([prev_token], dtype=torch.int32, device=dev)
    hyps, h, c, last = greedy_batch(model, encoder_out_chunk, lens, n_steps, predictor_states[0],
                                    predictor_states[1], last)
    return hyps[0], [h, c], int(last.item())


# ------------------------------------------------------------------------------------------------ A7
class BeamHypothesis:
    """model/online_rnnt_model.py:41-55."""

    def __init__(self, tokens: List[int], log_prob: float, predictor_states):
        self.tokens = tokens
        self.log_prob = log_prob
        self.predictor_states = predictor_states

    def copy(self):
        st = [s.clone() for s in self.predictor_states] if self.predictor_states is not None else None
        return BeamHypothesis(list(self.tokens), self.log_prob, st)

    def __lt__(self, other):
        return self.log_prob < other.log_prob


class OnlineBeamState:
    """Device-resident beam of one stream, carried across chunks (the reference keeps a Python list of
    BeamHypothesis on the module, model/online_rnnt_model.py:138-143)."""

    def __init__(self, model, beam_size: int, n_steps: int, max_out: int = 4096):
        self.w = _prepared(model).get()
        self.beam, self.n_steps, self.max_out = int(beam_size), int(n_steps), int(max_out)
        dev = next(model.joint.parameters()).device
        with torch.cuda.device(dev):
            nbytes = query("ctcvr_rnnt_beam_state_bytes", ctypes.byref(self.w), self.beam, self.n_steps, self.max_out)
            self.buf = torch.zeros(int(nbytes), dtype=torch.uint8, device=dev)
            call("ctcvr_rnnt_beam_reset", ptr(self.buf), ctypes.byref(self.w), self.beam, self.n_steps, self.max_out,
                 stream())


@torch.no_grad()
def beam_chunk_online(model, encoder_out_chunk: torch.Tensor, state: Optional[OnlineBeamState], beam_size: int = 4,
                      n_steps: int = 10) -> Tuple[List[BeamHypothesis], OnlineBeamState]:
    """The search of OnlineRNNTModel._decode_chunk_beam_search (model/online_rnnt_model.py:425-522) for one
    encoder chunk [1,Tc,H] (or [Tc,H]): one kernel launch per chunk, the beam stays on the device between
    chunks.  Returns (hypotheses ordered as the reference's list, state)."""
    if state is None:
        state = OnlineBeamState(model, beam_size, n_steps)
    w = _prepared(model).get()
    blank = _blank_of(model)
    x = encoder_out_chunk if encoder_out_chunk.dim() == 3 else encoder_out_chunk.unsqueeze(0)
    ep = _enc_proj(model, x)[0].contiguous()
    Tc = ep.shape[0]
    dev = ep.device
    beam, LH = state.beam, w.L * w.H
    out_n = torch.zeros((1,), dtype=torch.int32, device=dev)
    out_tok = torch.zeros((beam, state.max_out), dtype=torch.int32, device=dev)
    out_len = torch.zeros((beam,), dtype=torch.int32, device=dev)
    out_sc = torch.zeros((beam,), dtype=torch.float64, device=dev)
    out_h = torch.zeros((beam, w.L, w.H), dtype=torch.float32, device=dev)
    out_c = torch.zeros_like(out_h)
    with torch.cuda.device(dev):
        call("ctcvr_rnnt_beam_chunk", ctypes.byref(w), ptr(ep), Tc, ptr(state.buf), beam, state.n_steps, state.max_out,
             blank, ptr(out_n), ptr(out_tok), ptr(out_len), ptr(out_sc), ptr(out_h), ptr(out_c), stream())
    n = int(out_n.item())
    lens, toks, sc = out_len.cpu(), out_tok.cpu(), out_sc.cpu()
    hyps = [BeamHypothesis(toks[i, :int(lens[i])].tolist(), float(sc[i]),
                           [out_h[i].unsqueeze(1).clone(), out_c[i].unsqueeze(1).clone()]) for i in range(n)]
    return hyps, state


@torch.no_grad()
def beam_search_batch(model, encoder_out: torch.Tensor, encoder_out_lens: torch.Tensor, beam_size: int = 4,
                      n_steps: int = 10, max_out: Optional[int] = None) -> List[List[BeamHypothesis]]:
    """The search of `_decode_chunk_beam_search` (model/online_rnnt_model.py:425-522) over whole utterances, for S
    utterances in ONE kernel launch (one CTA per utterance; `ctcvr_rnnt_beam_chunk_batch`).  The reference decodes one
    stream at a time (batch 1 is asserted, online_rnnt_model.py:277-278); chunk boundaries only matter to the encoder, so
    utterance s gets exactly the hypotheses (tokens, order, scores) of feeding its frames through `beam_chunk_online`.
    encoder_out [S,T,H], encoder_out_lens [S].  Returns, per utterance, the beam as a list of BeamHypothesis."""
    w = _prepared(model).get()
    blank = _blank_of(model)
    ep = _enc_proj(model, encoder_out).contiguous()
    S, T = ep.shape[0], ep.shape[1]
    dev = ep.device
    beam = int(beam_size)
    lens = encoder_out_lens.to(device=dev, dtype=torch.int32).contiguous()
    mo = int(max_out) if max_out is not None else max(16, T * int(n_steps) + 1)      # a frame appends at most n_steps tokens
    LH = w.L * w.H
    with torch.cuda.device(dev):
        nbytes = int(query("ctcvr_rnnt_beam_state_bytes", ctypes.byref(w), beam, int(n_steps), mo))
        states = torch.zeros(S * nbytes, dtype=torch.uint8, device=dev)
        out_n = torch.zeros((S,), dtype=torch.int32, device=dev)
        out_tok = torch.zeros((S, beam, mo), dtype=torch.int32, device=dev)
        out_len = torch.zeros((S, beam), dtype=torch.int32, device=dev)
        out_sc = torch.zeros((S, beam), dtype=torch.float64, device=dev)
        out_h = torch.zeros((S, beam, w.L, w.H), dtype=torch.float32, device=dev)
        out_c = torch.zeros_like(out_h)
        call("ctcvr_rnnt_beam_reset_batch", ptr(states), ctypes.byref(w), S, beam, int(n_steps), mo, stream())
        call("ctcvr_rnnt_beam_chunk_batch", ctypes.byref(w), ptr(ep), ptr(lens), S, T, ptr(states), beam, int(n_steps), mo,
             blank, ptr(out_n), ptr(out_tok), ptr(out_len), ptr(out_sc), ptr(out_h), ptr(out_c), stream())
    ns, ls, sc = out_n.cpu().tolist(), out_len.cpu().numpy(), out_sc.cpu().numpy()
    width = max(int(ls.max()), 1)                           # only the used part of the token arrays crosses PCIe
    toks = out_tok[:, :, :width].contiguous().cpu().numpy()
    res = []
    for s_ in range(S):
        res.append([BeamHypothesis(toks[s_, i, :ls[s_, i]].tolist(), float(sc[s_, i]),
                                   [out_h[s_, i].unsqueeze(1), out_c[s_, i].unsqueeze(1)]) for i in range(ns[s_])])
    return res


# ------------------------------------------------------------------------------------------------ A8
@torch.no_grad()
def prefix_beam_search(model, encoder_out: torch.Tensor, ctc_logp: torch.Tensor, beam_size: int = 5,
                       ctc_weight: float = 0.3, transducer_weight: float = 0.7) -> List[Tuple[List[int], float]]:
    """wenet/transducer/search/prefix_beam_search.py:42-148 below the encoder call: encoder_out [T,H] (or
    [1,T,H]), ctc_logp [T,V] = ctc.log_softmax(encoder_out).  Returns [(hyp tokens incl. the leading blank, score)]
    best first."""
    w = _prepared(model).get()
    blank = _blank_of(model)
    x = encoder_out if encoder_out.dim() == 3 else encoder_out.unsqueeze(0)
    ep = _enc_proj(model, x)[0].contiguous()
    T = ep.shape[0]
    dev = ep.device
    cl = ctc_logp.reshape(-1, ctc_logp.shape[-1]).detach().float().contiguous().to(dev)
    beam = int(beam_size)
    out_n = torch.zeros((1,), dtype=torch.int32, device=dev)
    out_tok = torch.zeros((beam, T + 1), dtype=torch.int32, device=dev)
    out_len = torch.zeros((beam,), dtype=torch.int32, device=dev)
    out_sc = torch.zeros((beam,), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        nbytes = query("ctcvr_rnnt_prefix_beam_ws_bytes", ctypes.byref(w), beam, T)
        ws = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=dev)
        call("ctcvr_rnnt_prefix_beam", ctypes.byref(w), ptr(ep), ptr(cl), T, beam, blank, float(ctc_weight),
             float(transducer_weight), ptr(out_n), ptr(out_tok), ptr(out_len), ptr(out_sc), ptr(ws), ws.numel(), stream())
    n = int(out_n.item())
    lens, toks, sc = out_len.cpu(), out_tok.cpu(), out_sc.cpu()
    return [(toks[i, :int(lens[i])].tolist(), float(sc[i])) for i in range(n)]


@torch.no_grad()
def prefix_beam_search_batch(model, encoder_out: torch.Tensor, encoder_out_lens: torch.Tensor, ctc_logp: torch.Tensor,
                             beam_size: int = 5, ctc_weight: float = 0.3,
                             transducer_weight: float = 0.7) -> List[List[Tuple[List[int], float]]]:
    """`prefix_beam_search` (wenet/transducer/search/prefix_beam_search.py:42-148 below the encoder call) for S
    utterances in ONE launch (one CTA per utterance; `ctcvr_rnnt_prefix_beam_batch`): encoder_out [S,T,H],
    encoder_out_lens [S], ctc_logp [S,T,V].  Per utterance the same [(hyp incl. the leading blank, score)] list, best
    first, as the single-utterance call on its first encoder_out_lens[s] frames."""
    w = _prepared(model).get()
    blank = _blank_of(model)
    ep = _enc_proj(model, encoder_out).contiguous()
    S, T = ep.shape[0], ep.shape[1]
    dev = ep.device
    cl = ctc_logp.detach().float().contiguous().to(dev)
    if cl.shape[0] != S or cl.shape[1] != T:
        raise RuntimeError("prefix_beam_search_batch: ctc_logp must be [S,T,V] for encoder_out [S,T,H]")
    lens = encoder_out_lens.to(device=dev, dtype=torch.int32).contiguous()
    beam = int(beam_size)
    out_n = torch.zeros((S,), dtype=torch.int32, device=dev)
    out_tok = torch.zeros((S, beam, T + 1), dtype=torch.int32, device=dev)
    out_len = torch.zeros((S, beam), dtype=torch.int32, device=dev)
    out_sc = torch.zeros((S, beam), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        nbytes = int(query("ctcvr_rnnt_prefix_beam_ws_bytes", ctypes.byref(w), beam, T))
        ws = torch.empty(max(S * nbytes, 256), dtype=torch.uint8, device=dev)
        call("ctcvr_rnnt_prefix_beam_batch", ctypes.byref(w), ptr(ep), ptr(cl), ptr(lens), S, T, beam, blank,
             float(ctc_weight), float(transducer_weight), ptr(out_n), ptr(out_tok), ptr(out_len), ptr(out_sc), ptr(ws),
             ws.numel(), stream())
    ns, ls, sc = out_n.cpu().tolist(), out_len.cpu().numpy(), out_sc.cpu().numpy()
    width = max(int(ls.max()), 1)
    toks = out_tok[:, :, :width].contiguous().cpu().numpy()
    return [[(toks[s_, i, :ls[s_, i]].tolist(), float(sc[s_, i])) for i in range(ns[s_])] for s_ in range(S)]
