"""`install()` - swap the bodies of the reference's hot-path seams (SURVEY.md section 8b) for the kernels of this
package, IN PLACE, so that the reference's own train / eval / decode scripts run unchanged:

    import ctcvr_b200.patch as patch
    patch.install()             # imports model.* / wenet.* of the reference from sys.path
    # or patch.install(ns) with ns = {"model.online_rnnt_model": <module>, ...} / an object with those attributes

Every replacement keeps the reference's signature, argument meaning and return tuple (file:line in each docstring).
Classes are patched, not instances, so models built before or after the call are both covered; `uninstall()` restores
the originals.  Nothing here computes on the CPU: the patched methods raise RuntimeError on CPU tensors like the rest
of the package.
"""
from __future__ import annotations

import importlib
from typing import Dict, List, Optional

import torch

from . import decode as D
from . import functional as CF
from .predictor import lstm_stack
from .transducer import compute_rnnt_loss

_SAVED: List[tuple] = []

_MODULES = {
    "joint": "model.component.joint",
    "predictor": "model.component.predictor",
    "transducer": "model.component.transducer",
    "rnnt_model": "model.rnnt_model",
    "online": "model.online_rnnt_model",
    "prefix_beam": "wenet.transducer.search.prefix_beam_search",
    "search": "wenet.transformer.search",
}


def _resolve(ns, key):
    """ns may be None (import from sys.path), a dict keyed by the short names of _MODULES or the dotted module names,
    or any object carrying those attributes."""
    dotted = _MODULES[key]
    if ns is None:
        try:
            return importlib.import_module(dotted)
        except Exception:
            return None
    if isinstance(ns, dict):
        return ns.get(key, ns.get(dotted))
    return getattr(ns, key, None)


def _set(obj, name, value):
    _SAVED.append((obj, name, getattr(obj, name, None), hasattr(obj, name)))
    setattr(obj, name, value)


class _BeamList(list):
    """The hypotheses list handed back to the reference's drivers (model/online_rnnt_model.py:534-645 store it on the
    module and pass it into the next chunk): it carries the device-resident beam it was read from."""
    state = None


# ------------------------------------------------------------------------------------------------ replacements
def _joint_forward(self, enc_out: torch.Tensor, pred_out: torch.Tensor, pre_project: bool = True) -> torch.Tensor:
    """TransducerJoint.forward (model/component/joint.py:48-69): dense logits [B,T,U,V].  The add/tanh configuration
    both reference models build runs `ctcvr_joint_logits`; other configurations keep the reference's data flow."""
    fusable = isinstance(getattr(self, "activation", None), torch.nn.Tanh) and not getattr(self, "postjoin_linear", False) \
        and getattr(self, "joint_mode", "add") == "add"
    if pre_project and getattr(self, "prejoin_linear", True) and self.enc_ffn is not None and self.pred_ffn is not None:
        enc_out, pred_out = self.enc_ffn(enc_out), self.pred_ffn(pred_out)
    if fusable and enc_out.dim() == 3 and pred_out.dim() == 3:
        return CF.joint_logits(enc_out, pred_out, self.ffn_out.weight, self.ffn_out.bias)
    if enc_out.ndim != 4:
        enc_out = enc_out.unsqueeze(2)
    if pred_out.ndim != 4:
        pred_out = pred_out.unsqueeze(1)
    out = enc_out + pred_out
    if getattr(self, "postjoin_linear", False) and self.post_ffn is not None:
        out = self.post_ffn(out)
    return self.ffn_out(self.activation(out))


def _predictor_forward(self, input_tensor: torch.Tensor, cache: Optional[List[torch.Tensor]] = None) -> torch.Tensor:
    """RNNPredictor.forward (model/component/predictor.py:43-63): embed -> dropout -> LSTM -> projection with the
    recurrence in the sequence kernels (csrc/lstm_seq.cu) instead of the library LSTM."""
    embed = self.dropout(self.embed(input_tensor))
    if cache is None:
        st = self.init_state(batch_size=input_tensor.size(0), device=input_tensor.device)
        h0, c0 = st[0], st[1]
    else:
        assert len(cache) == 2
        h0, c0 = cache[0], cache[1]
    out, _, _ = lstm_stack(self.rnn, embed, h0, c0, self.training)
    return self.projection(out)


def _predictor_forward_step(self, input_tensor: torch.Tensor, padding: torch.Tensor, cache: List[torch.Tensor]):
    """RNNPredictor.forward_step (model/component/predictor.py:79-98)."""
    assert len(cache) == 2
    state_m, state_c = cache[0], cache[1]
    embed = self.dropout(self.embed(input_tensor.to(self.embed.weight.device)))
    out, m, c = lstm_stack(self.rnn, embed, state_m, state_c, self.training)
    out = self.projection(out)
    pad = padding.unsqueeze(0)
    return out, [pad * state_m + m * (1 - pad), pad * state_c + c * (1 - pad)]


def _transducer_compute_rnnt_loss(self, encoder_out, encoder_out_lens, text, text_lengths):
    """Transducer._compute_rnnt_loss (model/component/transducer.py:161-189): the fused seam."""
    return compute_rnnt_loss(self, encoder_out, encoder_out_lens, text, text_lengths)


def _ctc_forward_offline(self, hs_pad, hlens, ys_pad, ys_lens):
    """CTC.forward (model/rnnt_model.py:40-60): reduction 'sum' / batch; F.dropout without `training=` is kept."""
    logits = self.ctc_lo(torch.nn.functional.dropout(hs_pad, p=self.dropout_rate))
    loss, ys_hat = CF.ctc_loss_from_logits(logits, ys_pad, hlens, ys_lens, self.blank_id,
                                           "sum" if getattr(self, "reduce", True) else "none", True)
    return loss / logits.size(0), ys_hat


def _ctc_forward_online(self, hs_pad, hlens, ys_pad, ys_lens):
    """OnlineCTC.forward (model/online_rnnt_model.py:25-32): reduction 'mean'."""
    logits = self.ctc_lo(torch.nn.functional.dropout(hs_pad, p=self.dropout_rate))
    return CF.ctc_loss_from_logits(logits, ys_pad, hlens, ys_lens, self.blank_id, "mean", True)


def _ctc_log_softmax(self, hs_pad):
    """CTC.log_softmax (model/rnnt_model.py:62-70, model/online_rnnt_model.py:34-35)."""
    return CF.log_softmax_rows(self.ctc_lo(hs_pad))


def _ctc_greedy_offline(self, audios, audio_lens):
    """TransducerModel.ctc_greedy_search (model/rnnt_model.py:188-210): argmax + collapse on the device, one
    device->host copy instead of one `.item()` per frame."""
    encoder_out, encoder_mask = self.encoder(audios, audio_lens)
    lens = encoder_mask.squeeze(1).sum(1)
    return CF.ctc_greedy_search(self.ctc.ctc_lo(encoder_out), lens, int(self.transducer.blank))


def _ctc_greedy_online(self, audios, audio_lens):
    """OnlineRNNTModel.ctc_greedy_search (model/online_rnnt_model.py:647-671)."""
    if not self.ctc_head:
        return [[] for _ in range(audios.size(0))]
    encoder_out, encoder_mask = self.encoder(audios, audio_lens)
    lens = encoder_mask.reshape(encoder_mask.size(0), -1).sum(1)
    return CF.ctc_greedy_search(self.ctc_head.ctc_lo(encoder_out), lens, int(self.blank_id))


def _decode_chunk_streaming_logic(self, chunk_xs, offset, required_cache_size, att_cache_in, cnn_cache_in,
                                  predictor_states_in, prev_token_in, n_steps: int = 10):
    """OnlineRNNTModel._decode_chunk_streaming_logic (model/online_rnnt_model.py:166-222):
    -> (chunk tokens, att_cache, cnn_cache, [h, c], last token).  The encoder chunk stays the reference's; the search
    loop (one launch, no per-step host sync) is `ctcvr_rnnt_greedy` with the carried state."""
    encoder_out, att_cache_out, cnn_cache_out = self.encoder.forward_chunk(
        xs=chunk_xs, offset=offset, required_cache_size=required_cache_size, att_cache=att_cache_in,
        cnn_cache=cnn_cache_in)
    toks, states, last = D.greedy_chunk(self, encoder_out, predictor_states_in, int(prev_token_in), n_steps=n_steps)
    return toks, att_cache_out, cnn_cache_out, states, last


def _make_decode_chunk_beam_search(hyp_cls):
    def _decode_chunk_beam_search(self, chunk_xs, offset, required_cache_size, att_cache_in, cnn_cache_in,
                                  beam_hypotheses_in, beam_size: int = 4, n_steps: int = 10):
        """OnlineRNNTModel._decode_chunk_beam_search (model/online_rnnt_model.py:389-522):
        -> (List[BeamHypothesis] best first, att_cache, cnn_cache).  The beam lives on the device between chunks; the
        returned list (what the reference's drivers store and pass back in) carries it."""
        encoder_out, att_cache_out, cnn_cache_out = self.encoder.forward_chunk(
            xs=chunk_xs, offset=offset, required_cache_size=required_cache_size, att_cache=att_cache_in,
            cnn_cache=cnn_cache_in)
        if beam_hypotheses_in is None:
            state = None
        elif isinstance(beam_hypotheses_in, _BeamList) and beam_hypotheses_in.state is not None \
                and beam_hypotheses_in.state.beam == int(beam_size):
            state = beam_hypotheses_in.state
        else:
            raise RuntimeError("ctcvr_b200: _decode_chunk_beam_search continues the beam it returned for the previous "
                               "chunk (or starts from None); a hand-built hypothesis list cannot be resumed")
        if encoder_out.size(1) == 0:
            out = _BeamList(beam_hypotheses_in or [])
            out.state = state
            return out, att_cache_out, cnn_cache_out
        hyps, state = D.beam_chunk_online(self, encoder_out, state, beam_size=beam_size, n_steps=n_steps)
        out = _BeamList(hyp_cls(tokens=h.tokens, log_prob=h.log_prob, predictor_states=h.predictor_states) for h in hyps)
        out.state = state
        return out, att_cache_out, cnn_cache_out
    return _decode_chunk_beam_search


def _make_prefix_beam_search(seq_cls):
    def prefix_beam_search(self, speech, speech_lengths, decoding_chunk_size: int = -1, beam_size: int = 5,
                           num_decoding_left_chunks: int = -1, simulate_streaming: bool = False,
                           ctc_weight: float = 0.3, transducer_weight: float = 0.7):
        """PrefixBeamSearch.prefix_beam_search (wenet/transducer/search/prefix_beam_search.py:42-148):
        -> (List[Sequence] best first, encoder_out).  `Sequence.hyp` starts with blank as in the reference;
        `Sequence.cache` is None (the predictor caches stay on the device)."""
        assert speech.shape[0] == speech_lengths.shape[0]
        assert decoding_chunk_size != 0
        assert speech.shape[0] == 1
        encoder_out, _ = self.encoder(speech, speech_lengths, decoding_chunk_size, num_decoding_left_chunks)
        ctc_probs = self.ctc.log_softmax(encoder_out).squeeze(0)
        out = D.prefix_beam_search(self, encoder_out[0], ctc_probs, beam_size=beam_size, ctc_weight=ctc_weight,
                                   transducer_weight=transducer_weight)
        return [seq_cls(hyp=h, score=s, cache=None) for h, s in out], encoder_out
    return prefix_beam_search


# ------------------------------------------------------------------------------------------------ install
def install(namespace=None, precision: Optional[str] = None, vocab_tiling: Optional[bool] = None) -> Dict[str, List[str]]:
    """Patch whatever of the reference is present in `namespace` (None: import it).  Returns what was patched.
    `precision` ("fp32" | "bf16" | "bf16x3") becomes the class default of the patched `Transducer` (the fused loss
    reads `self.precision`, fp32 when absent), so an unchanged train script opts into the tcgen05 path with
    `install(precision="bf16")`, or into the tcgen05 path at fp32 accuracy with `install(precision="bf16x3")`; a model
    instance can still override it with its own `precision` attribute.  `vocab_tiling` (bool) becomes the class default of
    `Transducer.vocab_tiling` the same way: `install(precision="bf16", vocab_tiling=True)` trains a vocabulary beyond 416
    on the tensor cores."""
    if precision not in (None, "fp32", "bf16", "bf16x3"):
        raise ValueError("precision must be None, 'fp32', 'bf16' or 'bf16x3'")
    done: Dict[str, List[str]] = {}

    def note(mod, name):
        done.setdefault(mod, []).append(name)

    m = _resolve(namespace, "joint")
    if m is not None and hasattr(m, "TransducerJoint"):
        _set(m.TransducerJoint, "forward", _joint_forward)
        note("joint", "TransducerJoint.forward")
    m = _resolve(namespace, "predictor")
    if m is not None and hasattr(m, "RNNPredictor"):
        _set(m.RNNPredictor, "forward", _predictor_forward)
        _set(m.RNNPredictor, "forward_step", _predictor_forward_step)
        note("predictor", "RNNPredictor.forward/forward_step")
    m = _resolve(namespace, "transducer")
    if m is not None:
        if hasattr(m, "Transducer"):
            _set(m.Transducer, "_compute_rnnt_loss", _transducer_compute_rnnt_loss)
            note("transducer", "Transducer._compute_rnnt_loss")
            if precision is not None:
                _set(m.Transducer, "precision", precision)
                note("transducer", f"Transducer.precision = {precision}")
            if vocab_tiling is not None:
                _set(m.Transducer, "vocab_tiling", bool(vocab_tiling))
                note("transducer", f"Transducer.vocab_tiling = {bool(vocab_tiling)}")
        if hasattr(m, "basic_greedy_search"):
            _set(m, "basic_greedy_search", D.basic_greedy_search)
            note("transducer", "basic_greedy_search")
    m = _resolve(namespace, "rnnt_model")
    if m is not None:
        if hasattr(m, "CTC"):
            _set(m.CTC, "forward", _ctc_forward_offline)
            _set(m.CTC, "log_softmax", _ctc_log_softmax)
            note("rnnt_model", "CTC.forward/log_softmax")
        if hasattr(m, "TransducerModel"):
            _set(m.TransducerModel, "ctc_greedy_search", _ctc_greedy_offline)
            note("rnnt_model", "TransducerModel.ctc_greedy_search")
    m = _resolve(namespace, "online")
    if m is not None:
        if hasattr(m, "OnlineCTC"):
            _set(m.OnlineCTC, "forward", _ctc_forward_online)
            _set(m.OnlineCTC, "log_softmax", _ctc_log_softmax)
            note("online", "OnlineCTC.forward/log_softmax")
        if hasattr(m, "basic_greedy_search"):              # imported by name at model/online_rnnt_model.py:10
            _set(m, "basic_greedy_search", D.basic_greedy_search)
            note("online", "basic_greedy_search")
        if hasattr(m, "OnlineRNNTModel"):
            cls = m.OnlineRNNTModel
            _set(cls, "_decode_chunk_streaming_logic", _decode_chunk_streaming_logic)
            _set(cls, "_decode_chunk_beam_search", _make_decode_chunk_beam_search(getattr(m, "BeamHypothesis", D.BeamHypothesis)))
            _set(cls, "ctc_greedy_search", _ctc_greedy_online)
            note("online", "OnlineRNNTModel._decode_chunk_streaming_logic/_decode_chunk_beam_search/ctc_greedy_search")
    m = _resolve(namespace, "prefix_beam")
    if m is not None and hasattr(m, "PrefixBeamSearch"):
        _set(m.PrefixBeamSearch, "prefix_beam_search", _make_prefix_beam_search(m.Sequence))
        note("prefix_beam", "PrefixBeamSearch.prefix_beam_search")
    m = _resolve(namespace, "search")
    if m is not None and hasattr(m, "ctc_prefix_beam_search"):
        from . import search as S
        _set(m, "ctc_prefix_beam_search", S.ctc_prefix_beam_search)
        _set(m, "ctc_greedy_search", S.ctc_greedy_search)
        note("search", "ctc_prefix_beam_search/ctc_greedy_search")
    return done


def uninstall() -> None:
    while _SAVED:
        obj, name, old, had = _SAVED.pop()
        if had:
            setattr(obj, name, old)
        else:
            delattr(obj, name)
