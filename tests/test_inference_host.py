"""f3 (SURVEY §8): the rendering loop and the messengers against the unmodified reference.

tests/golden/inference_generator.npz and inference_messenger.npz were produced by oracle/gen_inference_golden.py from the
reference's `ScorePerformerGenerator`, `SPMupleMessenger`, `SPMuple2Messenger` and tokenizer methods on the synthetic vocabulary /
pieces of oracle/inference_cases.py.  Here `scoreperformer_b200.inference` gets the same inputs and the same stand-in decoder: every
decoder call (window length, cache length, token digests, embedding slices), every returned chunk, message, tempo state and cache
length must be IDENTICAL -- integers exactly, times to the last bit.  Host code only: no GPU needed.
"""
import os
import sys
from dataclasses import dataclass
from typing import List, Optional

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import inference_cases as cases  # noqa: E402
from tests import parity  # noqa: E402
from scoreperformer_b200.inference import (ScorePerformerGenerator, SPMuple2IntermediateData, SPMuple2Messenger, SPMupleMessenger,  # noqa: E402
                                           TokenTables)
from scoreperformer_b200.inference.token_tables import find_closest  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


@dataclass
class Attn:
    keys: Optional[torch.Tensor] = None
    values: Optional[torch.Tensor] = None
    qk_similarities: Optional[torch.Tensor] = None


@dataclass
class Inter:
    hiddens: Optional[List[torch.Tensor]] = None
    attention: Optional[List[Attn]] = None


@dataclass
class Caches:
    token_emb: Optional[torch.Tensor] = None
    transformer: Optional[Inter] = None


@pytest.fixture(scope="module")
def gen_golden():
    return np.load(os.path.join(GOLDEN, "inference_generator.npz"))


@pytest.fixture(scope="module")
def msg_golden():
    return np.load(os.path.join(GOLDEN, "inference_messenger.npz"))


def same(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} != {b.shape}"
    assert np.array_equal(a, b), f"{what}: max |diff| {np.abs(a.astype(np.float64) - b.astype(np.float64)).max()}"


@pytest.mark.parametrize("name", list(cases.SCENARIOS))
def test_rendering_loop_matches_reference(gen_golden, name):
    g = gen_golden
    tok = TokenTables(**cases.table_kwargs(**cases.SCENARIOS[name][1]))
    windows, final = cases.run_scenario(name, ScorePerformerGenerator, SPMuple2Messenger, tok, (Caches, Inter, Attn),
                                        SPMuple2IntermediateData)
    assert len(windows) == int(g[f"{name}/n_windows"])
    for i, w in enumerate(windows):
        for k, v in w.items():
            same(v, g[f"{name}/w{i}/{k}"], f"{name} window {i} {k}")
    for k, v in final.items():
        same(v, g[f"{name}/final/{k}"], f"{name} final {k}")


def test_scenarios_reach_the_branches_they_are_meant_for(gen_golden):
    """The goldens are only worth something if the reference actually truncated contexts, dropped and re-used caches, cut chords at
    window ends and refreshed tempo tokens while producing them."""
    g = gen_golden

    def calls(name):
        return np.concatenate([g[f"{name}/w{i}/calls"] for i in range(int(g[f"{name}/n_windows"]))])

    c = calls("chords_ctx48")
    assert c[:, 0].max() < 48 + 4 and (c[1:, 1] == -1).any() and (c[:, 1] > 0).any()      # truncated; caches dropped and re-used
    assert (c[:, 5] > 0).any()                                                           # context slices that do not start at note 0
    kept = [g[f"chords_ctx48/w{i}/seq"].shape[0] for i in range(int(g["chords_ctx48/n_windows"]))]
    made = [g[f"chords_ctx48/w{i}/calls"].shape[0] for i in range(int(g["chords_ctx48/n_windows"]))]
    assert any(m > 0 and k == 0 for m, k in zip(made, kept))                             # a window whose only chord came too late
    cache_after = [g[f"chords_ctx48/w{i}/state"][0] for i in range(len(kept))]
    assert any(b < a for a, b in zip(cache_after, cache_after[1:]))                      # cache rows cut / context truncated
    assert (calls("no_caches_ctx32")[:, 1] == -1).all()
    notes = g["tempo_is_input/final/notes"]
    assert len(np.unique(notes[1:-1, 5])) > 1 and not (notes[1:-1, 5] == 1).any()        # Tempo column rewritten, never MASKed
    assert g["single_notes_delta/w0/state"][3] != g["single_notes_delta/w5/state"][3]    # delta embedding written back


MESSENGER_CASES = {
    "spm2_refit": ("spm2", {}, 11, False),
    "spm2_refit_raw": ("spm2", dict(use_quantized_tempos=False, tempo_min_onsets=3, tempo_window=2.), 12, False),
    "spm2_token_tempo": ("spm2", dict(decode_recompute_tempos=False), 13, False),
    "spm2_onset_tempo": ("spm2", dict(onset_tempos=True), 14, True),
    "spm_beat": ("spm", {}, 15, False),
    "spm_bar_abs": ("spm", dict(bar_tempos=True, use_position_shifts=False, onset_position_shifts=True), 16, True),
    "spm_plain_shift": ("spm", dict(use_position_shifts=False, onset_position_shifts=False), 17, False),
}


@pytest.mark.parametrize("name", list(MESSENGER_CASES))
def test_messenger_matches_reference(msg_golden, name):
    """A piece fed in chunks that split chords, tempo state carried from chunk to chunk: messages (time, 144, pitch, velocity) of
    every chunk, the stateless onset times, tick messages (SPMuple), the final tempo map / onset pairs, and the one-shot decoding."""
    g = msg_golden
    family, params, seed, metre = MESSENGER_CASES[name]
    tok = TokenTables(**cases.table_kwargs(**params), spmuple2=family == "spm2")
    msgr = (SPMuple2Messenger if family == "spm2" else SPMupleMessenger)(tok)
    piece, cuts = cases.random_chunks(seed, metre_change=metre)
    state, lo = None, 0
    for i, hi in enumerate(cuts):
        chunk = piece[lo:hi]
        if f"{name}/c{i}/ticks" in g.files:
            same(msgr.tokens_to_messages(chunk.copy(), intermediates=state, to_times=False, sort=False), g[f"{name}/c{i}/ticks"],
                 f"{name} chunk {i} ticks")
        messages, state = msgr.tokens_to_messages(chunk.copy(), intermediates=state, return_intermediates=True)
        same(messages, g[f"{name}/c{i}/messages"], f"{name} chunk {i} messages")
        same(msgr.tokens_to_messages(chunk.copy(), note_attributes=False, note_off_events=False, intermediates=None, sort=False),
             g[f"{name}/c{i}/onsets"], f"{name} chunk {i} onsets")
        lo = hi
    same(state.tempos, g[f"{name}/tempos"], f"{name} tempo map")
    if family == "spm2":
        same(state.onset_pairs, g[f"{name}/pairs"], f"{name} onset pairs")
    same(msgr.tokens_to_messages(piece.copy()), g[f"{name}/whole"], f"{name} whole piece")


@pytest.mark.parametrize("metre", [0, 1])
def test_token_tables_ticks_and_shifts(msg_golden, metre):
    g = msg_golden
    tok = TokenTables(**cases.table_kwargs())
    piece = cases.make_piece(200, 31, bool(metre))
    ticks = tok.compute_ticks(piece, 8, compute_beat_ticks=True)
    tag = f"ticks{metre}"
    same(ticks["note_on"], g[f"{tag}/note_on"], "note ticks")
    same(ticks["bar"], g[f"{tag}/bar"], "bar ticks")
    same(ticks["beat"], g[f"{tag}/beat"], "beat ticks")
    same(ticks["time_sig"][0], g[f"{tag}/metres"], "metres")
    same(ticks["time_sig"][1], g[f"{tag}/metre_ticks"], "metre ticks")
    same(tok.compute_position_shifts(ticks["note_on"].copy(), onset_shift=True), g[f"{tag}/shifts_onset"], "onset shifts")
    same(tok.compute_position_shifts(ticks["note_on"].copy(), onset_shift=False), g[f"{tag}/shifts_plain"], "plain shifts")


def test_find_closest_and_table_io(msg_golden, tmp_path):
    g = msg_golden
    tok = TokenTables(**cases.table_kwargs())
    same(find_closest(tok.tempos, g["closest/probe"]), g["closest/index"], "find_closest (array)")
    same([find_closest(tok.tempos, float(v)) for v in g["closest/probe"][:40]], g["closest/scalars"], "find_closest (scalar)")
    assert tok[0, "SOS_None"] == 2 and tok[0, "EOS_None"] == 3 and tok[5, "Tempo_96"] == 4 + 33
    path = str(tmp_path / "tables.npz")
    tok.save(path)
    back = TokenTables.load(path)
    piece = cases.make_piece(50, 3)
    for field in cases.FIELDS:
        same(back.decode_token_type(piece, field), tok.decode_token_type(piece, field), field)
    assert back.additional_params == tok.additional_params and back.vocab_types_idx == tok.vocab_types_idx


def test_cut_caches_views_and_window_helpers():
    from scoreperformer_b200.inference.generators import bar_starts, chord_end, overflow_shift, resume_start
    L = 10
    mk = lambda d: torch.arange(L, dtype=torch.float32)[None, :, None].expand(1, L, d).clone()
    c = Caches(token_emb=mk(4), transformer=Inter(hiddens=[mk(4)], attention=[Attn(mk(2), mk(2), None)]))
    base = c.transformer.attention[0].keys
    c = ScorePerformerGenerator.cut_caches(c, left_idx=2, right_idx=7)
    assert c.token_emb.shape == (1, 5, 4) and c.transformer.hiddens[0].shape == (1, 5, 4)
    k = c.transformer.attention[0].keys
    assert k.shape == (1, 5, 2) and k.data_ptr() == base[:, 2:].data_ptr() and float(k[0, 0, 0]) == 2.     # a view, not a copy
    assert isinstance(c.transformer, Inter) and isinstance(c.transformer.attention[0], Attn)

    bars = np.array([4, 4, 5, 5, 5, 6, 7, 7])
    assert bar_starts(bars).tolist() == [1, 4, 5]
    notes = np.array([[4, 0], [4, 0], [4, 8], [5, 0], [5, 0], [5, 0]])
    assert [chord_end(notes, i) for i in (0, 2, 3)] == [2, 3, 6]
    assert resume_start(bars, 9, 64) == 0
    assert resume_start(bars, 9, 6) == 6                         # 9 - (4 + 1) < 6: the context restarts behind the change at 4
    assert overflow_shift(bars, 0, 6) == 5                       # 8 - 4 < 6: drop the five notes up to that bar change


def _reference_root():
    root = parity.reference_root()
    return root if root is not None and os.path.isdir(os.path.join(root, "scoreperformer", "inference")) else None


@pytest.mark.skipif(_reference_root() is None, reason="needs a copy of the original ScorePerformer project ($SPB200_REFERENCE_ROOT or baseline/_ref)")
def test_loop_around_the_reference_model_matches_the_reference_loop():
    """Live, not from goldens: the UNMODIFIED reference model (default recipe, CPU fp32, cached `unmask_tokens`) rendered once by the
    reference's generator + messenger and once by this package's -- same windows, caches handed back and forth between the reference's
    cache classes and this loop's `cut_caches` -- must give identical tuples and messages."""
    os.environ["SPB200_REFERENCE_ROOT"] = _reference_root()
    import gen_inference_golden as ref
    import ref_shim
    from scoreperformer.modules.sampling import top_k as ref_top_k
    ref_model, _ = ref_shim.build_reference_model(seed=23)
    ref_model.eval()
    piece = cases.make_piece(26, 41)
    tick = (piece[:, 0] - 4) * 32 + (piece[:, 1] - 4)
    onset = np.unique(tick, return_inverse=True)[1]
    seg = lambda a: torch.from_numpy(np.ascontiguousarray(a))[None]
    perf = torch.from_numpy(piece)[None]
    mask = torch.ones(perf.shape[:2], dtype=torch.bool)
    with torch.inference_mode():
        enc = ref_model.forward_encoders(perf=perf, perf_mask=mask, score=perf[..., :10].contiguous(), score_mask=mask, bars=seg(piece[:, 0]),
                                         beats=seg(4 + tick // 8), onsets=seg(4 + onset), deadpan_mask=torch.zeros(1, dtype=torch.bool),
                                         compute_loss=False)
    pad = lambda e: torch.cat([e[0, :1], e[0], e[0, -1:]]).clone()
    notes = np.concatenate([np.full_like(piece[:1], 2), piece, np.full_like(piece[:1], 3)])
    notes[1:-1, [3, 5, 10, 11]] = 1

    def render(generator_cls, messenger, tokenizer, interm_cls, max_context_len, **extra):
        gen = generator_cls(ref_model, cases.make_dataset(tokenizer, [piece]), cases.make_collator(), messenger, device="cpu")
        pd = gen.perf_data
        pd.perf_seq, pd.notes = piece, torch.from_numpy(notes.copy())
        pd.context, pd.embeddings = pad(enc.score_embeddings), pad(enc.perf_embeddings)
        pd.intermediates = interm_cls(initial_tempo=96.)
        t, messages = 0., []
        for _ in range(150):
            _, m = gen.generate_performance_notes(start_time=t, time_window=0.5, max_context_len=max_context_len,
                                                  filter_logits_fn=ref_top_k, filter_kwargs={"k": 1}, **extra)
            if len(m):
                messages.append(np.asarray(m))
            t += 0.5
            if pd.reached_eos:
                break
        # (a context shorter than 8 x the largest chord can stall the reference's loop for good -- generators.py:199-200 -- so the
        # end of the piece is only required of the full context)
        assert pd.reached_eos or max_context_len < 512
        return pd.gen_seq.numpy(), np.concatenate(messages)

    ref_tok = ref._ref_tokenizer(ref.SPMuple2)
    tables = TokenTables(**cases.table_kwargs())
    for ctx in (512, 20):                                  # 20: the context is truncated at bar starts and the caches are dropped
        want_tokens, want_messages = render(ref.ScorePerformerGenerator, ref.SPMuple2Messenger(ref_tok), ref_tok,
                                            ref.SPMuple2IntermediateData, ctx)
        got_tokens, got_messages = render(ScorePerformerGenerator, SPMuple2Messenger(tables), tables, SPMuple2IntermediateData, ctx)
        same(got_tokens, want_tokens, f"tokens (context {ctx})")
        same(got_messages, want_messages, f"messages (context {ctx})")
        # several chords per decoder call (the reference model's own cached unmask_tokens renders them): same rendering, greedy
        if ctx == 512:
            ahead_tokens, ahead_messages = render(ScorePerformerGenerator, SPMuple2Messenger(tables), tables, SPMuple2IntermediateData, ctx,
                                                  lookahead_notes=10)
            same(ahead_tokens, want_tokens, "tokens with lookahead")
            same(ahead_messages, want_messages, "messages with lookahead")
        assert got_tokens.shape[0] >= 16 and not (got_tokens == 1).any()


@pytest.mark.parametrize("name", list(cases.ENCODE_CASES))
def test_encode_embeddings_matches_reference(name):
    """`encode_embeddings` (generators.py:320-426): the windows asked of the dataset, the bar-shifted inputs of every encoder call, the
    embedding rows kept from every window (abutting windows, half-overlapping windows, one window) and the latents call."""
    g = np.load(os.path.join(GOLDEN, "inference_encode.npz"))
    r = cases.run_encode_case(name, ScorePerformerGenerator, SPMuple2Messenger, TokenTables(**cases.table_kwargs()))
    for k, v in r.items():
        same(v, g[f"{name}/{k}"], f"{name} {k}")
    assert r["score"].shape[0] == 182 and (len(r["windows"]) > 1) == (name != "one_window")


def test_host_library_exports_header_and_matches_numpy_on_long_pieces(monkeypatch):
    """include/spb200_host.h == the symbols of libspb200_host.so, and the C recurrence equals the numpy statement bit for bit on pieces
    long enough that the local-tempo sums run over hundreds of onsets (numpy's pairwise blocks and recursion), fed whole and in chunks
    that split chords, for every tempo mode."""
    import re
    from scoreperformer_b200.inference import native
    native.build()
    handle = native.lib()
    assert handle is not None, "libspb200_host.so missing: run __graft_entry__.build()"
    header = open(os.path.join(ROOT, "include", "spb200_host.h")).read()
    declared = set(re.findall(r"\b(spb_host_\w+)\s*\(", header))
    assert declared == {"spb_host_abi_version", "spb_host_onset_times"}
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in spb200_host.h but not exported"

    def decode(piece, cuts, params):
        msgr = SPMuple2Messenger(TokenTables(**cases.table_kwargs(**params)))
        state, lo, out = None, 0, []
        for hi in cuts:
            m, state = msgr.tokens_to_messages(piece[lo:hi].copy(), intermediates=state, return_intermediates=True)
            out.append(m)
            lo = hi
        return np.concatenate(out), state.tempos, state.onset_pairs

    rng = np.random.default_rng(9)
    for params in ({}, dict(tempo_window=1e9, tempo_min_onsets=300), dict(use_quantized_tempos=False, tempo_window=60.),
                   dict(decode_recompute_tempos=False), dict(onset_tempos=True)):
        piece = cases.make_piece(1500, int(rng.integers(1000)))
        cuts, i = [], 0
        while i < len(piece):
            i += int(rng.integers(1, 400))
            cuts.append(min(i, len(piece)))
        for c in (cuts, [len(piece)]):
            monkeypatch.setenv("SPB_HOST_NATIVE", "1")
            got = decode(piece, c, params)
            monkeypatch.setenv("SPB_HOST_NATIVE", "0")
            want = decode(piece, c, params)
            for a, b, what in zip(got, want, ("messages", "tempo map", "onset pairs")):
                same(a, b, f"{what} {params}")


PRESET = {  # the fields of the reference's data/tokenizers/spmuple_window.json that the tables depend on
    "tokenization": "SPMupleWindow", "miditok_version": "2.1.6",
    "config": {"pitch_range": [21, 109], "beat_res": {"0_2": 16, "2_4": 8, "4_8": 4, "8_16": 2, "16_64": 1}, "nb_velocities": 127,
               "special_tokens": ["PAD", "MASK", "SOS", "EOS"], "use_tempos": True, "use_time_signatures": True, "use_programs": False,
               "nb_tempos": 121, "tempo_range": [15, 480], "log_tempos": True, "programs": [0],
               "time_signature_range": {"2": [1, 2, 3, 4], "4": [1, 2, 3, 4, 5, 6], "8": [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12]},
               "additional_params": {"nb_onset_devs": 161, "nb_perf_durations": 81, "max_bar_embedding": 256, "rel_onset_dev": True,
                                     "rel_perf_duration": True, "real_max_bar_embedding": 256, "use_position_shifts": True,
                                     "onset_position_shifts": True, "use_onset_indices": True, "max_notes_in_onset": 12,
                                     "bar_tempos": False, "onset_tempos": False, "tempo_window": 8.0, "tempo_min_onset_dist": 0.5,
                                     "tempo_min_onsets": 8, "use_quantized_tempos": True, "decode_recompute_tempos": False}}}


def test_tables_from_a_tokenizer_preset():
    """`TokenTables.from_preset`: vocabulary sizes of SURVEY Appendix A.1 (sum 1251), the SPMuple / SPMuple2 bins equal to the
    reference constructors' (goldens), and a piece decodes through the messenger with the resulting tables."""
    import copy
    g = np.load(os.path.join(GOLDEN, "inference_vocab.npz"))
    t = TokenTables.from_preset(copy.deepcopy(PRESET))
    assert list(t.sizes.values()) == [260, 132, 92, 132, 133, 125, 26, 69, 16, 16, 165, 85] and list(t.vocab_types_idx) == cases.FIELDS
    assert t.spmuple2 and t.beat_res == 16 and t.additional_params["decode_recompute_tempos"] is False
    assert t.tempos[0] == 15. and t.tempos[-1] == 480. and t.velocities[0] == 0 and t.velocities[-1] == 127
    assert t.duration_values[0] == 0 and t.duration_values[1] == 1 / 16 and t.duration_values[-1] == 64
    for family, spm2 in (("spm", False), ("spm2", True)):
        for n_dev, n_dur, res, div in ((161, 81, 16, 1), (81, 41, 8, 2)):
            preset = copy.deepcopy(PRESET)
            preset["tokenization"] = "SPMupleWindow" if spm2 else "SPMupleBeat"
            preset["config"]["additional_params"].update(nb_onset_devs=n_dev, nb_perf_durations=n_dur)
            preset["config"]["beat_res"] = {k: max(1, v // div) for k, v in PRESET["config"]["beat_res"].items()}
            tt = TokenTables.from_preset(preset)
            tag = f"{family}/{n_dev}_{n_dur}_{res}"
            same(tt.position_shifts, g[f"{tag}/position_shifts"], f"{tag} position shifts")
            same(tt.rel_onset_deviations, g[f"{tag}/rel_onset_deviations"], f"{tag} onset deviations")
            same(tt.rel_performed_durations, g[f"{tag}/rel_performed_durations"], f"{tag} performed durations")
    piece = cases.make_piece(120, 8)
    piece[:, 1] = 4 + (piece[:, 1] - 4) * 2                         # the 8-per-beat grid of the synthetic piece on this 16-per-beat one
    messages = SPMuple2Messenger(t).tokens_to_messages(piece)
    assert messages.shape == (240, 4) and np.isfinite(messages).all() and np.all(np.diff(messages[:, 0]) >= 0)


def _package_arms():
    """This package's side of the seeded random cases of oracle/inference_cases.py."""
    def render(spm2, params):
        return (ScorePerformerGenerator, SPMuple2Messenger if spm2 else SPMupleMessenger,
                TokenTables(**cases.table_kwargs(**params), spmuple2=spm2), (Caches, Inter, Attn), SPMuple2IntermediateData)

    def messenger(spm2, params):
        return (SPMuple2Messenger if spm2 else SPMupleMessenger)(TokenTables(**cases.table_kwargs(**params), spmuple2=spm2))
    return render, messenger, lambda spm2: TokenTables(**cases.table_kwargs())


def _reference_arms():
    os.environ["SPB200_REFERENCE_ROOT"] = _reference_root()
    import gen_inference_golden as ref

    def render(spm2, params):
        return (ref.ScorePerformerGenerator, ref.SPMuple2Messenger if spm2 else ref.SPMupleMessenger,
                ref._ref_tokenizer(ref.SPMuple2 if spm2 else ref.SPMuple, **params), ref.REF_CACHES, ref.SPMuple2IntermediateData)

    def messenger(spm2, params):
        return (ref.SPMuple2Messenger if spm2 else ref.SPMupleMessenger)(ref._ref_tokenizer(ref.SPMuple2 if spm2 else ref.SPMuple, **params))
    return render, messenger, lambda spm2: ref._ref_tokenizer(ref.SPMuple2 if spm2 else ref.SPMuple)


def live_records(native=True):
    """This package's record of the seeded random cases, as tests/golden/inference_live.npz stores it (oracle/gen_live_golden.py)."""
    render, messenger, tokenizer = _package_arms()
    old = os.environ.get("SPB_HOST_NATIVE")
    os.environ["SPB_HOST_NATIVE"] = "1" if native else "0"
    try:
        return {"render": cases.run_fuzz_renderings(render), "messenger": cases.run_messenger_configurations(messenger),
                "tokenizer": cases.run_tokenizer_decodes(tokenizer)}
    finally:
        if old is None:
            os.environ.pop("SPB_HOST_NATIVE")
        else:
            os.environ["SPB_HOST_NATIVE"] = old


@pytest.fixture(scope="module")
def live_golden():
    """The seeded random cases as this package rendered them at the commit whose inference code the live tests last found identical
    to the original project (oracle/gen_live_golden.py); a copy of the original, where supplied, is compared live as well."""
    return np.load(os.path.join(GOLDEN, "inference_live.npz"))


@pytest.fixture(scope="module")
def live_got():
    return live_records(native=True)


def _same_record(got, g, part, what):
    want = {k[len(part) + 1:]: g[k] for k in g.files if k.startswith(part + "/")}
    assert sorted(got) == sorted(want), f"{what}: keys differ"
    for k in got:
        same(got[k], want[k], f"{what} {k}")


def test_random_renderings_match_the_reference_loop_live(live_golden, live_got):
    """Beyond the four scenario goldens: 14 random pieces, contexts, window lengths, chord grouping, style deltas, cache use, tempo
    modes and masked field sets around the stand-in decoder -- every decoder call and every window equal to the stored record, and
    to the original project's generator + messenger live where a copy is supplied."""
    _same_record(live_got["render"], live_golden, "render", "stored")
    if _reference_root() is not None:
        _same_record(live_got["render"], {f"render/{k}": v for k, v in cases.run_fuzz_renderings(_reference_arms()[0]).items()},
                     "render", "original")


def test_random_messenger_configurations_match_the_reference_live(live_golden, live_got):
    """Random tempo / shift / deviation settings, metre changes and chunkings through this package's messengers (C recurrence and
    numpy statement): messages, tick messages and carried state equal to the stored record, and to the original's messengers live
    where a copy is supplied."""
    _same_record(live_got["messenger"], live_golden, "messenger", "stored, C recurrence")
    _same_record(live_records(native=False)["messenger"], live_golden, "messenger", "stored, numpy statement")
    if _reference_root() is not None:
        _same_record(live_got["messenger"], {f"messenger/{k}": v for k, v in cases.run_messenger_configurations(_reference_arms()[1]).items()},
                     "messenger", "original")


def test_token_tables_decode_like_the_reference_tokenizer_live(live_golden, live_got):
    """Every field's `decode_token_type`, `compute_ticks` on random metre sequences and both `compute_position_shifts` modes of
    TokenTables equal to the stored record, and to the original tokenizer's own methods (SPMuple / SPMuple2) live where a copy is
    supplied."""
    _same_record(live_got["tokenizer"], live_golden, "tokenizer", "stored")
    if _reference_root() is not None:
        _same_record(live_got["tokenizer"], {f"tokenizer/{k}": v for k, v in cases.run_tokenizer_decodes(_reference_arms()[2]).items()},
                     "tokenizer", "original")


def test_host_abi_from_a_c_program(tmp_path):
    """The host C ABI without Python in the callee's process: tests/host_abi_client.c is compiled against include/spb200_host.h, linked
    to libspb200_host.so, fed the arrays of a piece, and must return what the numpy recurrence computes."""
    import shutil
    import subprocess
    from scoreperformer_b200.inference import native
    if shutil.which("gcc") is None:
        pytest.skip("no C compiler")
    lib_path = native.build()
    exe = str(tmp_path / "client")
    libdir = os.path.dirname(lib_path)
    subprocess.run(["gcc", "-O1", "-std=c11", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "host_abi_client.c"), "-o", exe,
                    "-L", libdir, "-lspb200_host", f"-Wl,-rpath,{libdir}"], check=True, capture_output=True)

    tok = TokenTables(**cases.table_kwargs())
    p = tok.additional_params
    piece = cases.make_piece(400, 12)
    ticks = tok.compute_ticks(piece, 8)["note_on"].astype(float)
    arrays = [ticks, tok.decode_token_type(piece, "Duration").astype(float), tok.decode_token_type(piece, "Tempo").astype(float),
              tok.decode_token_type(piece, "RelOnsetDev").astype(float), tok.decode_token_type(piece, "RelPerfDuration").astype(float)]
    performed = (piece[:, 3] != 4).astype(np.uint8)
    order = np.argsort(ticks, kind="stable").astype(np.int64)
    starts = np.flatnonzero(np.concatenate([[True], ticks[order][1:] != ticks[order][:-1]])).astype(np.int64)
    bounds = np.concatenate([starts, [len(order)]]).astype(np.int64)
    scale = 60 / 8
    tempos0, pairs0 = np.array([[96., 0, 0.]]), np.array([[-1., -1 / 96. * scale, 1.]])
    header = np.array([len(ticks), len(starts), 1, 1, 0, 1, p["tempo_min_onsets"], 1, len(tok.tempos), 0, 0, 0], dtype=np.int32)
    scalars = np.array([scale, 96., p["tempo_min_onset_dist"], p["tempo_window"], 0.])
    with open(tmp_path / "in.bin", "wb") as f:
        for a in [header, scalars] + arrays + [performed, order, bounds, tempos0, pairs0, tok.tempos.astype(float)]:
            f.write(np.ascontiguousarray(a).tobytes())
    subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], check=True)
    raw = open(tmp_path / "out.bin", "rb").read()
    n_t, n_p, resumed, _ = np.frombuffer(raw[:16], dtype=np.int32)
    body = np.frombuffer(raw[16:], dtype=np.float64)
    n = len(ticks)
    on, off = body[:n], body[n:2 * n]
    tempos, pairs = body[2 * n:2 * n + 3 * n_t].reshape(-1, 3), body[2 * n + 3 * n_t:].reshape(-1, 3)

    want_on, want_off = np.zeros(n), np.zeros(n)
    tok._current_midi_metadata = {"tempo_scale": scale}
    groups = np.split(order, starts[1:])
    state = SPMuple2IntermediateData(initial_tempo=96.)
    want_t, want_p = SPMuple2Messenger._recurrence(tok, p, state, tempos0.copy(), pairs0.copy(), groups, *arrays, performed.astype(bool), scale,
                                                   False, True, want_on, want_off)
    assert resumed == 0 and n_t == len(want_t) and n_p == len(want_p)
    same(on, want_on, "onset times")
    same(off, want_off, "offset times")
    same(tempos, want_t, "tempo map")
    same(pairs, want_p, "onset pairs")


@pytest.mark.parametrize("name", list(cases.SCENARIOS))
@pytest.mark.parametrize("ahead", [6, 40])
def test_lookahead_rendering_keeps_the_reference_results(gen_golden, name, ahead):
    """`lookahead_notes`: several chords per decoder call.  Everything a caller sees -- kept tuples, messages, tempo map, onset pairs,
    cache length after every window, the written-back style embeddings, the final sequence -- must equal the reference's goldens;
    only the number of decoder calls drops."""
    g = gen_golden
    piece_kw, params, ignore, gen_kw, window, kind = cases.SCENARIOS[name]
    variant = f"{name}_ahead{ahead}"
    cases.SCENARIOS[variant] = (piece_kw, params, ignore, dict(gen_kw, lookahead_notes=ahead), window, kind)
    try:
        windows, final = cases.run_scenario(variant, ScorePerformerGenerator, SPMuple2Messenger, TokenTables(**cases.table_kwargs(**params)),
                                            (Caches, Inter, Attn), SPMuple2IntermediateData)
    finally:
        cases.SCENARIOS.pop(variant)
    assert len(windows) == int(g[f"{name}/n_windows"])
    calls = ref_calls = 0
    for i, w in enumerate(windows):
        for k, v in w.items():
            if k != "calls":
                same(v, g[f"{name}/w{i}/{k}"], f"{variant} window {i} {k}")
        calls, ref_calls = calls + len(w["calls"]), ref_calls + len(g[f"{name}/w{i}/calls"])
    for k in ("gen_seq", "notes"):
        same(final[k], g[f"{name}/final/{k}"], f"{variant} final {k}")
    if name == "tempo_is_input":
        assert calls == ref_calls                           # lookahead is off when Tempo is refreshed between chords
    else:
        assert calls < ref_calls, (calls, ref_calls)
