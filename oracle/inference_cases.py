"""TEST INFRASTRUCTURE ONLY -- inputs for the rendering-loop / messenger parity tests (SURVEY §8 f3).

Shared by oracle/gen_inference_golden.py (which drives the UNMODIFIED reference `ScorePerformerGenerator` / messengers with
these inputs and stores what they did) and tests/test_inference_host.py (which drives scoreperformer_b200.inference with the same
inputs and compares).  Nothing here is the reference's code: it is a synthetic vocabulary, a synthetic piece, and a stand-in for
the decoder (`FakeDecoder`) whose "samples" are a hash of what it was given, so that two drivers of the loop produce the same
renderings exactly when they hand the decoder the same windows in the same order.

Nothing under scoreperformer_b200/ may import this file.
"""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np
import torch

FIELDS = ["Bar", "Position", "Pitch", "Velocity", "Duration", "Tempo", "TimeSig", "PositionShift", "NotesInOnset",
          "PositionInOnset", "RelOnsetDev", "RelPerfDuration"]
SIZES = dict(zip(FIELDS, [260, 132, 92, 132, 133, 125, 26, 69, 16, 16, 165, 85]))        # SURVEY Appendix A.1
ZERO = 4
BEAT_RES = 8
TIME_SIGS = [(4, 4), (3, 4), (2, 4), (6, 8), (9, 8), (12, 8), (5, 4), (2, 2), (3, 8), (6, 4), (7, 8), (3, 2), (4, 8), (5, 8),
             (7, 4), (8, 8), (9, 4), (12, 4), (18, 8), (24, 8), (1, 4), (1, 8)]


def table_kwargs(**params):
    """Value tables of a synthetic SPMuple2-shaped vocabulary (sizes of Appendix A.1)."""
    p = dict(use_position_shifts=True, rel_onset_dev=True, rel_perf_duration=True, bar_tempos=False, onset_position_shifts=True,
             decode_recompute_tempos=True, onset_tempos=False, tempo_min_onset_dist=0.5, tempo_window=8., tempo_min_onsets=8,
             use_quantized_tempos=True, max_notes_in_onset=12)
    p.update(params)
    return dict(
        vocab_types_idx={k: i for i, k in enumerate(FIELDS)}, sizes=dict(SIZES), beat_res=BEAT_RES, pitch_min=21,
        velocities=np.concatenate([[0], np.linspace(2, 127, SIZES["Velocity"] - ZERO - 1).round()]).astype(np.int64),
        duration_values=np.arange(SIZES["Duration"] - ZERO) / BEAT_RES,
        tempos=30. + 2 * np.arange(SIZES["Tempo"] - ZERO),
        time_signatures=np.array(TIME_SIGS), position_shifts=np.arange(SIZES["PositionShift"] - ZERO),
        rel_onset_deviations=np.linspace(-0.9, 0.9, SIZES["RelOnsetDev"] - ZERO),
        rel_performed_durations=np.linspace(0.1, 2.5, SIZES["RelPerfDuration"] - ZERO),
        additional_params=p, use_tempos=True, zero_token=ZERO)


def make_piece(n_notes: int, seed: int, metre_change: bool = False) -> np.ndarray:
    """A performance `[n_notes, 12]` (no SOS / EOS): chords of 1-4 notes on a 4/4 grid (optionally 3/4 from the middle on), bars
    increasing, every field a real token (>= 4)."""
    rng = np.random.default_rng(seed)
    rows, bar, pos = [], 0, 0
    while len(rows) < n_notes:
        metre = 1 if metre_change and len(rows) >= n_notes // 2 else 0
        per_bar = BEAT_RES * 4 * TIME_SIGS[metre][0] // TIME_SIGS[metre][1]
        chord = int(rng.integers(1, 5))
        step = int(rng.choice([0, 2, 4, 4, 8, 8, 16])) if rows else 0
        pos += step
        while pos >= per_bar:
            pos -= per_bar
            bar += 1
        tempo = int(rng.integers(40, 70))
        for j in range(chord):
            row = [bar, pos, int(rng.integers(20, 70)), int(rng.integers(0, 120)) if rng.random() > 0.08 else 0,
                   int(rng.integers(1, 40)), tempo + int(rng.integers(0, 2)), metre, min(step, 60) if j == 0 else 0,
                   min(chord, 11), j, int(rng.integers(0, 161)), int(rng.integers(0, 81))]
            rows.append([v + ZERO for v in row])
    return np.array(rows[:n_notes], dtype=np.int64)


class Processor:
    def __init__(self, sos=2, eos=3):
        self.sos, self.eos = sos, eos

    def add_sos_token(self, seq):
        return np.concatenate((np.full_like(seq[:1], self.sos), seq), axis=0)

    def add_eos_token(self, seq):
        return np.concatenate((seq, np.full_like(seq[:1], self.eos)), axis=0)


def make_dataset(tokenizer, pieces, initial_tempo=96.):
    names = [f"piece{i}" for i in range(len(pieces))]
    return SimpleNamespace(tokenizer=tokenizer, performances=list(pieces), performance_names=names, processor=Processor(),
                           initial_tempos={n: initial_tempo for n in names})


def make_collator(ignore=(0, 1, 2, 4, 6, 7, 8, 9)):
    return SimpleNamespace(mask_token_id=1, mask_ignore_token_dims=list(ignore))


def note_embeddings(n: int, dim: int = 3) -> torch.Tensor:
    """Row i = (i, i / 2, ...): a slice is identified by its first and last rows."""
    return torch.arange(n, dtype=torch.float32)[:, None] * torch.tensor([1., .5, .25][:dim])[None]


_W = np.array([1000003, 10007, 101, 7, 31, 131, 17, 3, 53, 59, 211, 13], dtype=np.int64)


def digest(a) -> int:
    a = np.asarray(a, dtype=np.int64)
    pos = np.arange(1, a.shape[0] + 1, dtype=np.int64)[:, None]
    return int(((a * _W[None, :a.shape[1]]) * pos % 1000000007).sum() % 1000000007)


class FakeDecoder:
    """Stands in for `model.perf_decoder`: `unmask_tokens` with the reference's signature.  Every MASK of `tokens` is replaced, note
    by note, with `4 + hash(previous note, position, field) mod (V - 4)`; caches are small tensors of the right lengths whose first
    channel counts positions (so a wrong cut is visible).  Every call is logged."""

    def __init__(self, cache_classes, sizes=tuple(SIZES.values())):
        self.caches_cls, self.inter_cls, self.attn_cls = cache_classes
        self.sizes = sizes
        self.log = []

    def unmask_tokens(self, tokens, tokens_masked, temperature=1., filter_logits_fn=None, filter_kwargs=None, filter_key_ids=None,
                      caches=None, return_caches=False, disable_tqdm=False, **kwargs):
        assert tokens.dim() == 2 and tokens.shape == tokens_masked.shape
        t = tokens.cpu().numpy().copy()
        tm = tokens_masked.cpu().numpy()
        n = t.shape[0]
        ctx, sty = kwargs.get("context"), kwargs.get("style_embeddings")
        cache_len = -1
        if caches is not None:
            cache_len = int(caches.token_emb.shape[1])
            assert torch.equal(caches.token_emb[0, :, 0], torch.arange(cache_len, dtype=torch.float32)), "cache rows out of order"
            for a in caches.transformer.attention:
                assert a.keys.shape[1] == cache_len and a.values.shape[1] == cache_len
            for h in caches.transformer.hiddens:
                assert h.shape[1] == cache_len
        entry = [n, cache_len, digest(t), digest(tm)]
        for e in (ctx, sty):
            entry += [-1, -1., -1.] if e is None else [int(e.shape[1]), float(e[0, 0, 0]), float(e[0, -1, 0])]
        entry += [float(sty[0].sum()) if sty is not None else 0.]
        self.log.append(entry)
        for i in np.flatnonzero((t == 1).any(axis=1)):
            for f in np.flatnonzero(t[i] == 1):
                h = (int(t[i - 1].sum()) * 31 + int(i) * 17 + int(f) * 7919 + int(t[i, 0]) * 13) % 104729
                t[i, f] = ZERO + h % (self.sizes[f] - ZERO)
        out = torch.from_numpy(t).to(tokens.device)
        if not return_caches:
            return out
        L = n - 1
        base = torch.arange(L, dtype=torch.float32)[None, :, None]
        mk = lambda d: base.expand(1, L, d).clone()
        new = self.caches_cls(token_emb=mk(4), transformer=self.inter_cls(
            hiddens=[mk(4), mk(4)], attention=[self.attn_cls(mk(2), mk(2), None), self.attn_cls(mk(2), mk(2), None)]))
        return out, new


def make_model(decoder):
    return SimpleNamespace(perf_decoder=decoder, perf_encoder=object(), score_encoder=object())


SCENARIOS = {
    # name: (piece kwargs, table params, collator ignore, generate kwargs, window length in s, messenger kind)
    "chords_ctx48": (dict(n_notes=230, seed=1), {}, (0, 1, 2, 4, 6, 7, 8, 9),
                     dict(max_context_len=48, time_window_overflow=0.1), 0.6, "spm2"),
    "single_notes_delta": (dict(n_notes=90, seed=2), dict(decode_recompute_tempos=False), (0, 1, 2, 4, 6, 7, 8, 9),
                           dict(group_chord_notes=False, delta=True, sort_messages=True), 0.9, "spm2"),
    "tempo_is_input": (dict(n_notes=120, seed=3), {}, (0, 1, 2, 4, 5, 6, 7, 8, 9),
                       dict(max_context_len=64), 0.5, "spm2"),
    "no_caches_ctx32": (dict(n_notes=140, seed=4, metre_change=False), dict(onset_tempos=True), (0, 1, 2, 4, 6, 7, 8, 9),
                        dict(max_context_len=32, disable_caches=True, time_window_overflow=0.0), 0.4, "spm2"),
}


def run_scenario(name, generator_cls, messenger_cls, tokenizer, cache_classes, intermediates_cls):
    """Drive a generator class through a whole piece in consecutive time windows; returns the log both sides must agree on."""
    piece_kw, _, ignore, gen_kw, window, _ = SCENARIOS[name]
    gen_kw = dict(gen_kw)
    piece = make_piece(**piece_kw)
    decoder = FakeDecoder(cache_classes)
    gen = generator_cls(make_model(decoder), make_dataset(tokenizer, [piece]), make_collator(ignore), messenger_cls(tokenizer),
                        device="cpu")
    n = piece.shape[0] + 2
    gen.prepare_performance_notes(0, score_embeddings=note_embeddings(n), perf_embeddings=note_embeddings(n) + 100.)
    use_delta = gen_kw.pop("delta", False)
    delta = torch.tensor([.5, -.25, .125]) if use_delta else None
    windows, t0, ahead = [], 0., -1.
    for _ in range(400):
        before = len(decoder.log)
        seq, messages = gen.generate_performance_notes(start_time=t0, time_window=window, delta_embedding=delta, **gen_kw)
        pd = gen.perf_data
        windows.append(dict(
            calls=np.array(decoder.log[before:], dtype=np.float64).reshape(-1, 11),
            seq=np.zeros((0, 12), np.int64) if seq is None else seq.cpu().numpy(),
            messages=np.zeros((0, 4)) if len(messages) == 0 else np.asarray(messages, dtype=np.float64),
            tempos=np.zeros((0, 3)) if pd.intermediates is None or pd.intermediates.tempos is None
            else np.array(pd.intermediates.tempos, dtype=np.float64),
            pairs=np.zeros((0, 3)) if getattr(pd.intermediates, "onset_pairs", None) is None
            else np.array(pd.intermediates.onset_pairs, dtype=np.float64),
            state=np.array([-1 if pd.caches is None else pd.caches.token_emb.shape[1], int(pd.reached_eos),
                            pd.gen_seq.shape[0], float(pd.embeddings.sum())], dtype=np.float64)))
        if name == "chords_ctx48" and len(windows) == 3:
            ahead = float(gen.predict_number_of_notes(start_time=t0, time_window=4 * window))
        t0 += window
        if pd.reached_eos:
            break
    final = dict(gen_seq=gen.perf_data.gen_seq.cpu().numpy(), notes=gen.perf_data.notes.cpu().numpy(), ahead=np.float64(ahead))
    return windows, final


def random_chunks(seed: int, n_notes: int = 160, metre_change: bool = False):
    """A piece cut into consecutive chunks of 1-9 notes (chords are split across chunks on purpose)."""
    rng = np.random.default_rng(seed)
    piece = make_piece(n_notes, seed + 100, metre_change)
    cuts, i = [], 0
    while i < n_notes:
        i += int(rng.integers(1, 10))
        cuts.append(min(i, n_notes))
    return piece, cuts


# ----------------------------------------------------------------------------- seeded random cases (tests/golden/inference_live.npz)
# Each function drives one side (`arm`) through a fixed list of random cases and returns a flat {key: array} record; the tests
# compare this package's record with the stored one and, where a copy of the original project is supplied, with the original's.
def fuzz_scenarios():
    """14 random rendering scenarios (default_rng(2024)): name -> (SCENARIOS entry, SPMuple2 family?).  Every fifth one uses the
    SPMuple family (tick-based messenger, no tempo state)."""
    rng = np.random.default_rng(2024)
    out = {}
    for i in range(14):
        params = [{}, dict(decode_recompute_tempos=False), dict(onset_tempos=True), dict(use_quantized_tempos=False, tempo_window=3.)][i % 4]
        ignore = (0, 1, 2, 4, 6, 7, 8, 9) if i % 3 else (0, 1, 2, 4, 5, 6, 7, 8, 9)
        gen_kw = dict(max_context_len=int(rng.choice([24, 40, 64, 512])), group_chord_notes=bool(rng.random() < 0.7),
                      time_window_overflow=float(rng.choice([0., 0.1, 0.3])), disable_caches=bool(rng.random() < 0.2),
                      delta=bool(rng.random() < 0.4), sort_messages=bool(rng.random() < 0.5))
        entry = (dict(n_notes=int(rng.integers(40, 160)), seed=int(rng.integers(1000))), params, ignore, gen_kw,
                 float(rng.choice([0.25, 0.5, 1.0, 2.5])), "spm2")
        out[f"fuzz{i}"] = (entry, i % 5 != 4)
    return out


def run_fuzz_renderings(arm):
    """`arm(spm2, params)` -> (generator class, messenger class, tokenizer, cache classes, intermediates class).  Each field of the
    windows is stored concatenated over them, with its row count per window."""
    out = {}
    for name, (entry, spm2) in fuzz_scenarios().items():
        SCENARIOS[name] = entry
        try:
            windows, final = run_scenario(name, *arm(spm2, entry[1]))
        finally:
            SCENARIOS.pop(name)
        for k in windows[0]:
            parts = [np.atleast_2d(w[k]) if w[k].ndim < 2 else w[k] for w in windows]
            out[f"{name}/{k}"] = np.concatenate(parts)
            out[f"{name}/{k}_rows"] = np.array([len(p) for p in parts], dtype=np.int64)
        for k, v in final.items():
            out[f"{name}/final/{k}"] = v
    return out


def run_messenger_configurations(arm):
    """16 random messenger settings (default_rng(77)) with metre changes and chunkings; `arm(spm2, params)` -> messenger.  Per case:
    the messages of every chunk (SPMuple: also its tick messages) concatenated, the tempo map and the onset pairs carried at the end."""
    rng = np.random.default_rng(77)
    out = {}
    for i in range(16):
        spm2 = i % 2 == 0
        params = dict(decode_recompute_tempos=bool(rng.random() < 0.6), onset_tempos=bool(rng.random() < 0.25),
                      use_quantized_tempos=bool(rng.random() < 0.5), tempo_window=float(rng.choice([1., 4., 8., 1e6])),
                      tempo_min_onsets=int(rng.choice([2, 8, 40])), tempo_min_onset_dist=float(rng.choice([0.1, 0.5, 2.])),
                      bar_tempos=bool(rng.random() < 0.5), use_position_shifts=bool(rng.random() < 0.5),
                      onset_position_shifts=bool(rng.random() < 0.5), rel_onset_dev=True, rel_perf_duration=bool(spm2 or rng.random() < 0.7))
        if not spm2 and not params["rel_perf_duration"]:
            continue                                       # absolute PerfDuration needs its own vocabulary column
        m = arm(spm2, params)
        piece, cuts = random_chunks(int(rng.integers(10000)), n_notes=int(rng.integers(30, 400)), metre_change=bool(rng.random() < 0.4))
        state, lo, msgs = None, 0, []
        for hi in cuts:
            if not spm2:
                msgs.append(m.tokens_to_messages(piece[lo:hi].copy(), intermediates=state, to_times=False, sort=True))
            chunk_msgs, state = m.tokens_to_messages(piece[lo:hi].copy(), intermediates=state, return_intermediates=True, sort=bool(hi % 2))
            msgs.append(chunk_msgs)
            lo = hi
        out[f"case{i}/messages"] = np.concatenate(msgs)
        out[f"case{i}/tempos"] = np.asarray(state.tempos, dtype=np.float64)
        out[f"case{i}/pairs"] = np.asarray(getattr(state, "onset_pairs", None) if spm2 else [[0.]], dtype=np.float64)
    return out


def run_tokenizer_decodes(arm):
    """`decode_token_type` of every field, `compute_ticks` and both `compute_position_shifts` modes on random pieces (default_rng(5))
    with one or several (compound) metres, for the SPMuple and SPMuple2 families; `arm(spm2)` -> the object whose methods run."""
    rng = np.random.default_rng(5)
    out = {}
    for spm2 in (False, True):
        tok = arm(spm2)
        for trial in range(6):
            piece = make_piece(int(rng.integers(5, 300)), int(rng.integers(10000)), metre_change=bool(trial % 2))
            if trial >= 3:                                  # several metre changes, compound metres included
                bars = piece[:, 0] - 4
                piece[:, 6] = 4 + (bars // int(rng.integers(2, 6))) % 22
            tag = f"spm{2 if spm2 else 1}/t{trial}"
            for field in FIELDS:
                out[f"{tag}/{field}"] = np.asarray(tok.decode_token_type(piece, field))
            ticks = tok.compute_ticks(piece.copy(), 8, compute_beat_ticks=True)
            for key in ("note_on", "bar", "beat"):
                out[f"{tag}/ticks_{key}"] = np.asarray(ticks[key])
            out[f"{tag}/metres"], out[f"{tag}/metre_ticks"] = np.asarray(ticks["time_sig"][0]), np.asarray(ticks["time_sig"][1])
            on = np.sort(ticks["note_on"])
            for mode in (True, False):
                out[f"{tag}/shifts_{int(mode)}"] = np.asarray(tok.compute_position_shifts(on.copy(), onset_shift=mode))
    return out


# ----------------------------------------------------------------------------- encode_embeddings: a dataset that serves bar windows
class _Scores(list):
    _name_to_idx = {"score0": 0}


class BarWindowDataset:
    """What `ScorePerformerGenerator.encode_embeddings` touches of a ScorePerformanceDataset: whole-bar windows of one score / performance
    pair (`get(meta=...)` with `meta.start_bar` / `meta.end_bar`, SOS before bar 0, EOS behind the last bar), the bar index, the
    window limits and the segment maps."""

    def __init__(self, tokenizer, piece: np.ndarray, max_seq_len: int, max_bar: int):
        self.tokenizer, self.max_seq_len, self.max_bar = tokenizer, max_seq_len, max_bar
        self.processor = Processor()
        self.performance_names, self._performance_map = ["perf0"], {"perf0": ("score0", None)}
        self.scores, self.performances = _Scores([piece[:, :10].copy()]), [piece]
        self.initial_tempos = {"perf0": 96.}
        self._score_indices = [None]
        tick = (piece[:, 0] - ZERO) * 32 + (piece[:, 1] - ZERO)
        self._beat_maps, self._onset_maps = [ZERO + tick // 8], [ZERO + np.unique(tick, return_inverse=True)[1]]
        self.indexer = SimpleNamespace(compute_bar_indices=self._bar_indices)
        self.windows = []

    @staticmethod
    def _bar_indices(seq):
        bars = seq[:, 0] - ZERO
        first = np.searchsorted(bars, np.arange(bars[-1] + 1), side="left")       # first note of every bar (empty bars: the next note)
        return np.concatenate([first, [len(bars)]]).astype(np.int64)

    def get(self, meta):
        idx = self._score_indices[0]
        lo, hi = int(idx[meta.start_bar]), int(idx[meta.end_bar + 1])
        self.windows.append((int(meta.start_bar), int(meta.end_bar), lo, hi))
        score, perf = self.scores[0][lo:hi], self.performances[0][lo:hi]
        if meta.start_bar == 0:
            score, perf = self.processor.add_sos_token(score), self.processor.add_sos_token(perf)
        if meta.end_bar + 1 >= len(idx) - 1:
            score, perf = self.processor.add_eos_token(score), self.processor.add_eos_token(perf)
        return SimpleNamespace(score=score, perf=perf, lo=lo)


class EncoderStub:
    """`model` for encode_embeddings: the embeddings are the (bar-shifted) tokens themselves, so that what comes back shows which notes
    of which window were kept and how their bars had been moved."""

    def __init__(self, dataset):
        self.perf_decoder, self.score_encoder = object(), object()
        self.perf_encoder = SimpleNamespace(embeddings_to_latents=self._latents)
        self.dataset, self.calls = dataset, []

    def prepare_inputs(self, x):
        return x

    def allocate_inputs(self, x, device):
        return x

    def forward_encoders(self, score, score_mask, perf, perf_mask, bars, beats, onsets, deadpan_mask, compute_loss):
        assert compute_loss is False
        self.calls.append([score.shape[1], digest(score[0].numpy()), digest(perf[0].numpy())])
        return SimpleNamespace(score_embeddings=score[..., :3].float(), perf_embeddings=perf[..., [0, 1, 10]].float() + 0.5)

    @staticmethod
    def _latents(embeddings, bars, beats, onsets):
        return torch.stack([embeddings.sum(), bars.float().sum(), beats.float().sum(), onsets.float().sum(),
                            torch.tensor(float(bars.shape[1]))])


def window_collator(samples):
    (s,) = samples
    score, perf = torch.from_numpy(s.score.copy())[None], torch.from_numpy(s.perf.copy())[None]
    ones = torch.ones(score.shape[:2], dtype=torch.bool)
    seg = torch.arange(score.shape[1])[None] + ZERO
    return dict(score=score, score_mask=ones, perf=perf, perf_mask=ones.clone(), bars=seg, beats=seg.clone(), onsets=seg.clone(),
                deadpan_mask=torch.zeros(1, dtype=torch.bool))


ENCODE_CASES = {"abutting": dict(overlay_bars=0., max_seq_len=40, max_bar=6), "overlapping": dict(overlay_bars=0.5, max_seq_len=90, max_bar=64),
                "one_window": dict(overlay_bars=0.5, max_seq_len=4000, max_bar=256)}


def run_encode_case(name, generator_cls, messenger_cls, tokenizer):
    kw = ENCODE_CASES[name]
    piece = make_piece(180, 21)
    ds = BarWindowDataset(tokenizer, piece, kw["max_seq_len"], kw["max_bar"])
    model = EncoderStub(ds)
    collator = window_collator
    collator.mask_token_id, collator.mask_ignore_token_dims = 1, [0, 1, 2, 4, 6, 7, 8, 9]
    gen = generator_cls(model, ds, collator, messenger_cls(tokenizer), device="cpu")
    score_emb, perf_emb, latents = gen.encode_embeddings(0, compute_latents=True, overlay_bars=kw["overlay_bars"])
    return dict(score=score_emb.numpy(), perf=perf_emb.numpy(), latents=latents.numpy(), calls=np.array(model.calls, dtype=np.int64),
                windows=np.array(ds.windows, dtype=np.int64))
