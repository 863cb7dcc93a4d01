"""Windowed rendering loop around `perf_decoder.unmask_tokens` (reference inference/generators.py:23-443, SURVEY §8 f3).

`ScorePerformerGenerator` keeps the reference's constructor, methods, arguments, `PerformanceData` state and return values, so a
real-time player written against the reference runs unchanged.  What is different is where the bookkeeping lives.  The reference
keeps the growing note sequence on the device and decides everything with device-tensor expressions (`torch.all(a == b)` per chord
candidate, `torch.where(torch.diff(...))` per context check, `.clone()` / `torch.cat` per note group): each of those is a kernel
launch plus a blocking device->host read, a dozen per generated chord, next to a decoder step that takes ~0.2 ms on a B200.  Here the
note skeleton (everything except the sampled fields is known before rendering starts) lives in host numpy arrays:

* chord ends and bar starts are index arithmetic on the host copy of the notes;
* one call per chord uploads the window's two token arrays (<= 512 x 12 int64) and reads back only the chord's new tuples, which the
  messenger needs on the host anyway to decide whether the time window is full;
* the device keeps what is large: encoder embeddings, the decoder caches, the generated sequence the caller reads.

The decisions are the reference's, line for line in effect: chord grouping on (Bar, Position) (:159-165), the optional tempo-token
refresh (:168-172), bar-aligned truncation to `max_context_len` (:136-140, :182-200), bars shifted to zero for the model (:203-204,
241-243), the cache-length check (:222-226), the time-window stop and cut (:256-257, 266-271) and the cache cut (:289-293).
tests/test_inference_host.py replays whole renderings against logs produced by the unmodified reference class.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from types import SimpleNamespace
from typing import Callable, Dict, Optional, Union

import numpy as np
import torch
from torch import Tensor

from ..modules.sampling import top_k
from .messengers import IntermediateData, SPMuple2IntermediateData, SPMupleMessenger
from .token_tables import DEFAULT_TEMPO, EOS_TOKEN, SOS_TOKEN, find_closest, is_spmuple2


@dataclass
class PerformanceData:
    perf_seq: Optional[np.ndarray] = None                # the dataset's performance (target tokens, host)
    notes: Optional[Tensor] = None                       # SOS + notes with the rendered fields MASKed + EOS (device)
    embeddings: Optional[Tensor] = None                  # performance (style) embedding per note
    context: Optional[Tensor] = None                     # score-encoder embedding per note
    gen_seq: Optional[Tensor] = None                     # everything rendered and kept so far, SOS first
    intermediates: Optional[IntermediateData] = None     # the messenger's tempo state after `gen_seq`
    caches: Optional[object] = None                      # decoder caches covering the kept part of the context
    reached_eos: bool = False


def bar_starts(bars: np.ndarray) -> np.ndarray:
    """Indices i with bars[i + 1] != bars[i] (what `torch.where(torch.diff(x))[0]` returns in the reference)."""
    return np.flatnonzero(bars[1:] != bars[:-1])


def chord_end(notes: np.ndarray, i: int) -> int:
    """One past the last note that shares (Bar, Position) with note i (generators.py:159-163)."""
    end = i + 1
    while end < len(notes) and notes[end, 0] == notes[i, 0] and notes[end, 1] == notes[i, 1]:
        end += 1
    return end


def resume_start(kept_bars: np.ndarray, n_kept: int, max_context_len: int) -> int:
    """Where the context of a new call starts inside the kept sequence (`kept_bars` = its Bar column without the SOS row): at the
    first bar start that leaves fewer than `max_context_len` notes, else 0 (generators.py:135-140)."""
    if n_kept < max_context_len - 1:
        return 0
    nb = bar_starts(kept_bars)
    fits = np.flatnonzero(n_kept - (nb + 1) < max_context_len)
    return 0 if len(nb) == 0 or len(fits) == 0 else int(nb[fits[0]]) + 2


def overflow_shift(bars: np.ndarray, first_note: int, max_context_len: int) -> int:
    """How many leading notes a full window drops: up to the first bar start that makes it fit, unless that would leave only the
    newest note; otherwise one (generators.py:185-190).  `bars` is the window's Bar column."""
    n = len(bars)
    nb = bar_starts(bars[first_note:])
    fits = np.flatnonzero(n - (nb + first_note) < max_context_len)
    if len(nb) and len(fits):
        cand = int(nb[fits[0]]) + 1 + first_note
        if cand != n - 1:
            return cand
    return 1


class ScorePerformerGenerator:
    def __init__(self, model, dataset, collator, messenger: SPMupleMessenger, device: Optional[Union[str, torch.device]] = None):
        assert model.perf_decoder is not None
        self.model, self.dataset, self.collator, self.messenger, self.device = model, dataset, collator, messenger, device
        self.tokenizer = dataset.tokenizer
        self.sos_token_id = self.tokenizer[0, SOS_TOKEN]
        self.eos_token_id = self.tokenizer[0, EOS_TOKEN]
        self._spm2 = is_spmuple2(self.tokenizer)
        self._init_variables()
        self.reset()

    def _init_variables(self):
        fields = range(len(self.tokenizer.sizes))
        self._mask_cols = sorted(set(fields).difference(self.collator.mask_ignore_token_dims))
        self.mask_dims = torch.tensor(self._mask_cols)

    def reset(self):
        self.perf_data = PerformanceData()
        self._mirrors: Dict[str, tuple] = {}

    # ------------------------------------------------------------------ host mirrors of the small token tensors
    def _mirror(self, name: str, t: Tensor) -> np.ndarray:
        """Host copy of `perf_data.<name>`, fetched once per tensor object: the caller may REPLACE the tensor between calls (a new
        object is fetched again); edits made in place to the same tensor object are not seen -- assign a new tensor instead."""
        src, arr = self._mirrors.get(name, (None, None))
        if src is not t:
            arr = t.detach().cpu().numpy().copy()
            self._mirrors[name] = (t, arr)
        return arr

    def _set_mirror(self, name: str, t: Tensor, arr: np.ndarray):
        self._mirrors[name] = (t, arr)

    # ------------------------------------------------------------------ preparation
    def prepare_performance_notes(self, perf_idx: int, score_embeddings: Optional[Tensor] = None,
                                  perf_embeddings: Optional[Tensor] = None, overlay_bars: float = 0.5):
        perf_seq = self.dataset.performances[perf_idx]
        self.perf_data.perf_seq = perf_seq
        initial_tempo = DEFAULT_TEMPO
        if self._spm2 and hasattr(self.dataset, "initial_tempos"):
            initial_tempo = self.dataset.initial_tempos[self.dataset.performance_names[perf_idx]]

        seq = self.dataset.processor.add_eos_token(self.dataset.processor.add_sos_token(perf_seq))
        need_perf = self.model.perf_encoder is not None and perf_embeddings is None
        need_score = self.model.score_encoder is not None and score_embeddings is None
        if need_perf or need_score:
            score_embeddings, perf_embeddings, _ = self.encode_embeddings(perf_idx, overlay_bars=overlay_bars)

        notes = np.array(seq, copy=True)
        notes[1:-1, self._mask_cols] = self.collator.mask_token_id
        self.perf_data.notes = torch.from_numpy(notes).to(self.device)
        self._set_mirror("notes", self.perf_data.notes, notes.copy())
        self.perf_data.embeddings, self.perf_data.context = perf_embeddings, score_embeddings
        if self._spm2:
            self.perf_data.intermediates = SPMuple2IntermediateData(initial_tempo=initial_tempo)
        return self.perf_data

    # ------------------------------------------------------------------ the window loop
    def generate_performance_notes(self, start_time: float = 0., time_window: float = 0.2, time_window_overflow: float = 0.1,
                                   delta_embedding: Optional[Tensor] = None, max_context_len: int = 512,
                                   group_chord_notes: bool = True, time_messages: bool = True, sort_messages: bool = False,
                                   filter_logits_fn: Callable = top_k, filter_kwargs: Optional[Dict[str, object]] = None,
                                   disable_tqdm: bool = True, disable_caches: bool = False, lookahead_notes: int = 0):
        """One time window of the rendering (generators.py:106-295); arguments and results as in the reference.

        `lookahead_notes` (an addition; 0 = the reference's call pattern, one decoder call per chord): render up to that many notes of
        the following chords in the SAME decoder call, then walk the chords on the host exactly as if they had been rendered one by
        one -- messenger, time-window test, cut -- and slice the returned caches back to the chord the reference would have stopped
        at.  A decoder call has a fixed cost (weight staging, prepared terms) that dwarfs a note-step, so a window of several chords
        costs one call instead of one per chord.  The kept tuples, messages, tempo state and caches are the same as without
        lookahead whenever a note's rendering depends on earlier notes only (greedy decoding; with sampling the random draws of
        notes beyond the window are simply discarded instead of never made).  Switched off where the call pattern matters:
        when the Tempo field is an input refreshed from the messenger between chords, and wherever the window would reach
        `max_context_len` (truncation decisions are the reference's, chord by chord)."""
        pd, tok = self.perf_data, self.tokenizer
        notes = self._mirror("notes", pd.notes)
        style_all = pd.embeddings.clone().detach() if pd.embeddings is not None else None
        score_all = pd.context.clone().detach() if pd.context is not None else None
        if pd.gen_seq is None:
            pd.gen_seq = pd.notes[:1]
        kept = self._mirror("gen_seq", pd.gen_seq)
        device = pd.gen_seq.device

        cur = kept.shape[0]                                # index of the next note to render
        start = resume_start(kept[1:, 0], cur, max_context_len)
        window = kept[start:].copy()                       # context + notes of this call, host
        known = window.shape[0]
        first = int(window[0, 0] == self.sos_token_id)
        delta = None if delta_embedding is None else delta_embedding.to(self.device)
        tempo_col = tok.vocab_types_idx.get("Tempo") if self._spm2 else None
        refresh_tempo = tempo_col is not None and tempo_col not in self._mask_cols

        caches, state = pd.caches, pd.intermediates
        times, rendered, ran = [], [], False
        while not pd.reached_eos:
            end = chord_end(notes, cur) if group_chord_notes else cur + 1
            k = end - cur
            if refresh_tempo:                              # tempo is an input, not rendered: follow the messenger's estimate
                bpm = state.tempos[-1, 0] if state.tempos is not None else state.initial_tempo
                token = find_closest(tok.tempos, bpm) + tok.zero_token
                notes[cur:end, tempo_col] = token
                pd.notes[cur:end, tempo_col] = int(token)
            if notes[end - 1, 0] == self.eos_token_id:
                pd.reached_eos = True
                break

            # further whole chords for the same decoder call, as long as the window stays below the context limit without them
            bounds = [cur, end]
            room = max_context_len - 1 - (window.shape[0] + k)
            while lookahead_notes > 0 and not refresh_tempo and bounds[-1] - cur < lookahead_notes:
                nxt = chord_end(notes, bounds[-1]) if group_chord_notes else bounds[-1] + 1
                if notes[nxt - 1, 0] == self.eos_token_id or nxt - end > room:
                    break
                bounds.append(nxt)
            run_end = bounds[-1]

            window = np.concatenate([window, notes[cur:end]], axis=0)
            if window.shape[0] >= max_context_len:
                shift = overflow_shift(window[:, 0], first, max_context_len)
                window, known, start, first, caches = window[shift:], known - shift, start + shift, 0, None
                if known < max_context_len / 8:
                    break                                  # more notes inside the time window than the context can hold
            if run_end > end:
                window = np.concatenate([window, notes[end:run_end]], axis=0)
            n, k = window.shape[0], run_end - cur

            # what the model sees: bars counted from the window's first note, every rendered field of every note MASKed in the
            # second stream
            to_zero = window[first, 0] - tok.zero_token
            tokens = window.copy()
            tokens[first:, 0] -= to_zero
            masked = tokens.copy()
            masked[first:, self._mask_cols] = self.collator.mask_token_id

            if style_all is not None and delta is not None:
                style_all[cur:run_end] += delta
            context = score_all[start:run_end].unsqueeze(0) if score_all is not None else None
            style = style_all[start:run_end].unsqueeze(0) if style_all is not None else None
            if caches is not None and (n - 1 - k != caches.token_emb.shape[1] or caches.token_emb.shape[1] == 0
                                       or len(caches.transformer.attention) == 0):
                caches = None

            with torch.inference_mode():
                out, caches = self.model.perf_decoder.unmask_tokens(
                    torch.from_numpy(tokens).to(self.device), torch.from_numpy(masked).to(self.device),
                    context=context, style_embeddings=style, caches=None if disable_caches else caches, return_caches=True,
                    filter_logits_fn=filter_logits_fn, filter_kwargs=filter_kwargs, disable_tqdm=disable_tqdm)
                fresh = out[n - k:n].cpu().numpy().copy()  # the one device->host read of the call
            ran = True
            fresh[:, 0] += to_zero
            full = False
            for a, b in zip(bounds[:-1], bounds[1:]):      # the chords of the call, one by one as the reference meets them
                chord = fresh[a - cur:b - cur]
                chord_times, state = self.messenger.tokens_to_messages(chord, note_attributes=False, note_off_events=False,
                                                                       intermediates=state, return_intermediates=True, sort=False)
                times.extend(chord_times.tolist())
                rendered.append(chord)
                if chord_times.max() >= start_time + time_window + time_window_overflow:
                    full = True
                    if b < run_end and caches is not None:  # chords rendered ahead of the one that filled the window never happened
                        caches = self.cut_caches(caches, right_idx=n - 1 - (run_end - b))
                    break
                window[n - k + (a - cur):n - k + (b - cur)] = chord
            if full:
                break
            cur = run_end

        if not ran:
            return None, []
        inside = np.flatnonzero(np.array(times) <= start_time + time_window)
        n_keep = 0 if len(inside) == 0 else int(inside[-1]) + 1
        if n_keep == 0:
            return None, []

        new_tokens = np.concatenate(rendered, axis=0)[:n_keep]
        messages, pd.intermediates = self.messenger.tokens_to_messages(new_tokens, intermediates=pd.intermediates,
                                                                       return_intermediates=True, to_times=time_messages,
                                                                       sort=sort_messages)
        if style_all is not None and delta is not None:   # keep the shifted style of the notes that stay
            total = pd.gen_seq.shape[0]
            pd.embeddings[total:total + n_keep] = style_all[total:total + n_keep]

        gen_seq = torch.from_numpy(new_tokens).to(device=device)
        pd.gen_seq = torch.cat([pd.gen_seq, gen_seq])
        self._set_mirror("gen_seq", pd.gen_seq, np.concatenate([kept, new_tokens], axis=0))
        if caches is not None:                             # drop the cache rows of rendered notes that fell outside the window
            caches = self.cut_caches(caches, right_idx=caches.token_emb.shape[1] - (len(times) - n_keep))
        pd.caches = caches
        return gen_seq, messages

    def predict_number_of_notes(self, start_time: float = 0., time_window: float = 0.2, max_notes: int = 32):
        """How many of the next target notes start inside the window at the current tempo (generators.py:297-318).  Works on a
        copy: the reference shifts the Tempo column of the dataset's array in place."""
        pd = self.perf_data
        done = len(pd.gen_seq) - 1 if pd.gen_seq is not None else 0
        ahead = np.array(pd.perf_seq[done:done + max_notes], copy=True)
        if len(ahead) == 0:
            return 0.
        if pd.intermediates is not None and pd.intermediates.tempos is not None:
            col = self.tokenizer.vocab_types_idx["Tempo"]
            token = self.tokenizer[col, f"Tempo_{int(pd.intermediates.tempos[-1, 0])}"]
            ahead[:, col] += token - pd.perf_seq[done - 1, col]
        at = self.messenger.tokens_to_messages(ahead, note_attributes=False, note_off_events=False,
                                               intermediates=pd.intermediates, sort=False)
        return (at <= start_time + time_window).sum()

    # ------------------------------------------------------------------ encoders over a whole piece
    def encode_embeddings(self, perf_idx: int, compute_latents: bool = False, overlay_bars: float = 0., augmentations=None):
        """Score / performance embeddings of every note of a piece from overlapping `max_seq_len` windows of whole bars
        (generators.py:320-426).  The dataset supplies the windows (`dataset.get(meta=...)`), this loop moves the bars to zero,
        runs `forward_encoders` and keeps, from every window after the first, the notes of bars not yet covered."""
        ds, tok = self.dataset, self.tokenizer
        score_name, _ = ds._performance_map[ds.performance_names[perf_idx]]
        score_idx = ds.scores._name_to_idx[score_name]
        if ds._score_indices[score_idx] is None:
            ds._score_indices[score_idx] = ds.indexer.compute_bar_indices(ds.scores[score_idx])
        bar_index = ds._score_indices[score_idx]

        def last_bar_of_window(first_bar):                 # data/datasets/utils.py:56-58
            reach = np.flatnonzero(bar_index <= bar_index[first_bar] + ds.max_seq_len)[-1] - 1
            return min(max(first_bar, reach), first_bar + ds.max_bar - 1)

        bar_col, bar0 = tok.vocab_types_idx["Bar"], tok.zero_token
        total_bars = ds.scores[score_idx][-1, bar_col] - bar0
        first_bar, keep_from = 0, 0
        last_bar = last_bar_of_window(first_bar)
        meta = _sample_meta(score_idx=score_idx, perf_idx=perf_idx, start_bar=first_bar, end_bar=last_bar, augmentations=augmentations)
        score_parts, perf_parts = [], []
        while True:
            sample = ds.get(meta=meta)
            sos = int(sample.score[0, 0] == self.sos_token_id)
            eos = int(sample.score[-1, 0] == self.eos_token_id)
            if sample.score[sample.score.shape[0] - eos - 1, bar_col] - bar0 > total_bars:
                break
            inputs = self.model.allocate_inputs(self.model.prepare_inputs(self.collator((sample,))), self.device)
            to_zero = inputs["score"][:, sos, bar_col] - bar0
            inputs["score"][:, sos:sample.score.shape[0] - eos, bar_col] -= to_zero
            inputs["perf"][:, sos:sample.perf.shape[0] - eos, bar_col] -= to_zero
            with torch.inference_mode():
                enc = self.model.forward_encoders(score=inputs["score"], score_mask=inputs["score_mask"], perf=inputs["perf"],
                                                  perf_mask=inputs["perf_mask"], bars=inputs["bars"], beats=inputs["beats"],
                                                  onsets=inputs["onsets"], deadpan_mask=inputs["deadpan_mask"], compute_loss=False)
            cut = 0
            if overlay_bars:
                cut = int(np.flatnonzero(sample.score[:, bar_col] - bar0 >= keep_from)[0]) - sos
            if enc.score_embeddings is not None:
                score_parts.append(enc.score_embeddings[0, cut:])
            if enc.perf_embeddings is not None:
                perf_parts.append(enc.perf_embeddings[0, cut:])
            if eos:
                break
            if overlay_bars:
                first_bar = sample.score[int(sample.score.shape[0] * (1 - overlay_bars)), 0] - bar0
                keep_from = last_bar + 1
            else:
                keep_from = first_bar = last_bar + 1
            last_bar = last_bar_of_window(first_bar)
            meta.start_bar, meta.end_bar = first_bar, last_bar

        score_emb = torch.cat(score_parts, dim=0) if score_parts else None
        perf_emb = torch.cat(perf_parts, dim=0) if perf_parts else None
        latents = None
        if perf_emb is not None and compute_latents:
            pad = lambda s: torch.from_numpy(np.concatenate([[s[0]], s, [s[-1]]]))[None].to(self.device)
            latents = self.model.perf_encoder.embeddings_to_latents(
                embeddings=perf_emb[None], bars=pad(ds.scores[score_idx][:, 0]), beats=pad(ds._beat_maps[score_idx]),
                onsets=pad(ds._onset_maps[score_idx]))
        return score_emb, perf_emb, latents

    # ------------------------------------------------------------------ caches
    @staticmethod
    def cut_caches(caches, left_idx=0, right_idx=None):
        """Keep positions [left_idx, right_idx) of every cached tensor (time is dim -2).  Views, no copies; the container types
        are taken from the object itself so that the reference's and this package's cache classes both work."""
        right_idx = caches.token_emb.shape[-1] if right_idx is None else right_idx      # (sic: the reference's default, :430)
        cut = lambda t: t[..., left_idx:right_idx, :]
        tr = caches.transformer
        caches.token_emb = caches.token_emb[:, left_idx:right_idx]
        caches.transformer = type(tr)(hiddens=[cut(h) for h in tr.hiddens],
                                      attention=[type(a)(cut(a.keys), cut(a.values), None) for a in tr.attention])
        return caches


# the reference's logit filters (modules/sampling.py) and the keyword arguments each takes, with its defaults
_BATCH_FILTERS = {"top_k": {"thres": 0.9, "k": None}, "top_p": {"thres": 0.9}, "top_a": {"min_p_pow": 2.0, "min_p_ratio": 0.02}}


def _batch_sampling(filter_logits_fn: Callable, filter_kwargs: Optional[Dict[str, object]], model, cols) -> Dict[str, object]:
    """`render_batch` keyword arguments for a reference filter function and its kwargs; raises on anything else.  top-k's `thres`
    gives k = ceil((1 - thres) V) per rendered field, V the vocabulary of the field's head."""
    from ..modules import sampling
    name = next((n for n in _BATCH_FILTERS if filter_logits_fn is getattr(sampling, n)), None)
    if name is None and getattr(filter_logits_fn, "__module__", "").endswith("modules.sampling"):
        name = getattr(filter_logits_fn, "__name__", None)              # the same functions of the original package
    if name not in _BATCH_FILTERS:
        raise ValueError(f"render_performances samples with top_k, top_p or top_a of modules.sampling, not {filter_logits_fn!r}")
    kw = dict(filter_kwargs or {})
    unknown = set(kw) - set(_BATCH_FILTERS[name])
    if unknown:
        raise ValueError(f"{name} takes {sorted(_BATCH_FILTERS[name])}, not {sorted(unknown)}")
    args = {**_BATCH_FILTERS[name], **kw}
    if name == "top_p":
        return {"top_p": float(args["thres"])}
    if name == "top_a":
        return {"top_a": (float(args["min_p_pow"]), float(args["min_p_ratio"]))}
    if args["k"] is not None or "thres" not in kw:
        return {"top_k": args["k"]}                                      # None: render_batch's ceil(0.1 V), the reference default
    sizes = model.perf_decoder.model.token_emb.field_sizes
    return {"top_k": [math.ceil((1 - float(args["thres"])) * sizes[c]) for c in cols]}


def render_performances(model, messenger: SPMupleMessenger, collator, pieces, filter_kwargs: Optional[Dict[str, object]] = None,
                        temperature: float = 1., time_messages: bool = True, sort_messages: bool = True,
                        filter_logits_fn: Callable = top_k):
    """Whole pieces, many at once: the offline counterpart of the window loop (SURVEY §8 C5 -- the reference renders one piece at a
    time through the same loop with an infinite window).  `pieces` are `PerformanceData` as `prepare_performance_notes` leaves them
    (notes with the rendered fields MASKed, per-note score / style embeddings, messenger state); pieces must fit the decoder context
    as a whole (no truncation happens here).  All pieces advance in lock-step through `decode.render_batch` -- one persistent
    decoder-stack launch and one heads + sampling launch per note for the whole batch -- then the rendered tuples come back in ONE
    device->host copy and each piece goes through the messenger.  Sampling takes the reference's filters: `filter_logits_fn` is `top_k`
    (`filter_kwargs` `k` or `thres`; default ceil(0.1 V)), `top_p` (`thres`) or `top_a` (`min_p_pow`, `min_p_ratio`) of
    modules/sampling.py with their defaults; any other function or keyword raises ValueError.  top-a takes each piece's own
    largest probability (the reference's takes it over the batch it is given, here one piece).  Returns `[(gen_seq, messages), ...]` and completes every piece's `gen_seq` / `intermediates`."""
    from ..decode import render_batch
    tok = messenger.tokenizer
    if not pieces or any(pd.notes is None or pd.context is None or pd.embeddings is None for pd in pieces):
        raise ValueError("render_performances needs notes, score embeddings (context) and style embeddings for every piece")
    sos, eos = tok[0, SOS_TOKEN], tok[0, EOS_TOKEN]
    cols = sorted(set(range(len(tok.sizes))).difference(collator.mask_ignore_token_dims))
    sampling_kw = _batch_sampling(filter_logits_fn, filter_kwargs, model, cols)
    dev = pieces[0].context.device
    rows = []
    for pd in pieces:
        notes = pd.notes.detach().cpu().numpy().copy()
        n = notes.shape[0] - int(notes[-1, 0] == eos)     # the EOS row never enters the decoder
        rows.append((notes[:n], int(notes[0, 0] == sos)))
    S, T, F = len(rows), max(r[0].shape[0] for r in rows), rows[0][0].shape[1]
    tokens, valid = np.zeros((S, T, F), dtype=np.int64), np.zeros((S, T), dtype=bool)
    to_zero = np.zeros(S, dtype=np.int64)
    context = torch.zeros((S, T, pieces[0].context.shape[-1]), dtype=pieces[0].context.dtype, device=dev)
    style = torch.zeros((S, T, pieces[0].embeddings.shape[-1]), dtype=pieces[0].embeddings.dtype, device=dev)
    for i, ((notes, first), pd) in enumerate(zip(rows, pieces)):
        n = notes.shape[0]
        to_zero[i] = notes[first, 0] - tok.zero_token     # bars counted from the piece's first note, as in the window loop
        tokens[i, :n] = notes
        tokens[i, first:n, 0] -= to_zero[i]
        valid[i, :n] = True
        context[i, :n], style[i, :n] = pd.context[:n], pd.embeddings[:n]
    masked = tokens.copy()
    for i, (notes, first) in enumerate(rows):
        masked[i, first:notes.shape[0]][:, cols] = collator.mask_token_id
    out = render_batch(model, torch.from_numpy(tokens).to(dev), torch.from_numpy(masked).to(dev), context, style,
                       mask=torch.from_numpy(valid).to(dev), fields=cols, temperature=temperature, **sampling_kw)
    host = out.cpu().numpy()
    results = []
    for i, ((notes, first), pd) in enumerate(zip(rows, pieces)):
        n = notes.shape[0]
        seq = host[i, :n].copy()
        seq[first:, 0] += to_zero[i]
        # note 0 is the SOS row or a given note: what was rendered starts behind it, as `gen_seq` does in the window loop
        messages, pd.intermediates = messenger.tokens_to_messages(seq[1:], intermediates=pd.intermediates, return_intermediates=True,
                                                                  to_times=time_messages, sort=sort_messages)
        pd.gen_seq = torch.from_numpy(seq).to(dev)
        pd.reached_eos = True
        results.append((pd.gen_seq[1:], messages))
    return results


def _sample_meta(**fields):
    """The dataset's own sample-meta class when the reference data package is importable, else a plain namespace with the same
    fields (data/datasets/score_performance.py `ScorePerformanceSampleMeta`)."""
    try:
        from scoreperformer.data.datasets import ScorePerformanceSampleMeta
        return ScorePerformanceSampleMeta(idx=None, **fields)
    except Exception:
        return SimpleNamespace(idx=None, **fields)
