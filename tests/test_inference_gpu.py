"""f3 on the GPU: `inference.ScorePerformerGenerator` driving the CUDA decoder (cached `unmask_tokens`) in time windows.

The loop itself is pinned to the reference on the host (tests/test_inference_host.py); what is checked here is that the loop and the
device path fit together: windows that cut chords and slice the caches must render exactly what one uninterrupted call renders
(greedy decoding), and that rendering agrees with the one-shot batched renderer up to near-ties."""
import numpy as np
import pytest
import torch

from tests import parity
import inference_cases as cases

pytestmark = pytest.mark.gpu

RENDERED = [3, 5, 10, 11]


def _piece(T, seed):
    """A synthetic performance whose notes of one onset share (Bar, Position): 12 onsets per 4/4 bar."""
    batch = parity.make_batch(1, T, seed=seed, full_length=True, deadpan_last=False)
    onset = batch["onsets"][0] - 4
    perf = batch["perf"][0].clone()
    perf[:, 0] = 4 + onset // 12
    perf[:, 1] = 4 + (onset % 12) * 2
    perf[:, 6] = 4                                                        # 4/4 throughout
    batch["perf"][0] = perf
    batch["score"][0] = perf[:, :10]
    return batch, perf


@pytest.mark.parametrize("stream", ["fused", "legacy"])
def test_windowed_rendering_on_device_equals_uninterrupted_rendering(stream, monkeypatch):
    # fused: `unmask_tokens` continues the caller-held caches on the device-resident note-step; legacy: the general cached stepper
    # (the path a request takes that the note-step cannot express) -- both must satisfy the same contract
    monkeypatch.setenv("SPB_STREAM", stream)
    from scoreperformer_b200.decode import render_batch
    from scoreperformer_b200.inference import ScorePerformerGenerator, SPMuple2IntermediateData, SPMuple2Messenger, TokenTables
    from scoreperformer_b200.modules.sampling import top_k
    T = 64
    model = parity.build_model(dropout=False, device="cuda").eval()
    batch, perf = _piece(T, seed=77)
    b = {k: v.cuda() for k, v in batch.items()}
    with torch.inference_mode():
        enc = model.forward_encoders(perf=b["perf"], perf_mask=b["perf_mask"], score=b["score"], score_mask=b["score_mask"],
                                     bars=b["bars"], beats=b["beats"], onsets=b["onsets"], deadpan_mask=b["deadpan_mask"],
                                     compute_loss=False)
    notes = perf.clone()
    notes[1:, RENDERED] = 1                                               # note 0 is given, the rest is rendered
    notes = torch.cat([notes, torch.full_like(notes[:1], 3)])             # EOS row
    pad = lambda e: torch.cat([e[0], e[0, -1:]]).clone()                  # one embedding row for the EOS position

    tok = TokenTables(**cases.table_kwargs())

    def render(time_window):
        gen = ScorePerformerGenerator(model, cases.make_dataset(tok, [perf.numpy()]), cases.make_collator(), SPMuple2Messenger(tok),
                                      device="cuda")
        pd = gen.perf_data
        pd.notes, pd.context, pd.embeddings = notes.cuda(), pad(enc.score_embeddings), pad(enc.perf_embeddings)
        pd.intermediates = SPMuple2IntermediateData(initial_tempo=96.)
        n_messages, n_windows, t0 = 0, 0, 0.
        while not pd.reached_eos and n_windows < 400:
            before = pd.gen_seq.shape[0] if pd.gen_seq is not None else 1
            seq, messages = gen.generate_performance_notes(start_time=t0, time_window=time_window, filter_logits_fn=top_k,
                                                           filter_kwargs={"k": 1})
            n_messages += len(messages)
            n_windows += 1
            if seq is not None:
                assert seq.is_cuda and pd.gen_seq.shape[0] == before + seq.shape[0]
                if pd.caches is not None:                                 # caches cover exactly the kept notes but the last
                    assert pd.caches.token_emb.shape[1] <= pd.gen_seq.shape[0] - 1
                    assert pd.caches.transformer.attention[0].keys.shape[1] == pd.caches.token_emb.shape[1]
            t0 += time_window
        assert pd.reached_eos
        return pd.gen_seq, n_messages, n_windows

    whole, m_whole, w_whole = render(1e9)
    windowed, m_win, w_win = render(0.35)
    assert w_whole <= 2 and w_win > 4, (w_whole, w_win)
    assert whole.shape == (T, 12) and torch.equal(whole, windowed)
    assert m_whole == m_win == 2 * (T - 1)                                # a note-on and a note-off per rendered note
    assert int((whole == 1).sum()) == 0
    keep = [f for f in range(12) if f not in RENDERED]
    assert torch.equal(whole[:, keep].cpu(), perf[:, keep])

    masked = perf.clone()
    masked[:, RENDERED] = 1
    want = render_batch(model, notes[None, :T].cuda(), masked[None].cuda(), enc.score_embeddings, enc.perf_embeddings)
    agree = float((whole[:, RENDERED] == want[0][:, RENDERED]).float().mean())
    assert agree > 0.85, agree


def test_render_performances_batches_whole_pieces():
    """Offline counterpart of the window loop: three pieces of different lengths (SOS / EOS rows, bars not starting at zero) rendered in
    lock-step by `render_performances`; every piece agrees with its own uninterrupted window-loop rendering up to near-ties, given
    fields come back untouched, and the messages are exactly the messenger's decoding of the returned tuples."""
    from scoreperformer_b200.inference import (PerformanceData, ScorePerformerGenerator, SPMuple2IntermediateData, SPMuple2Messenger,
                                               TokenTables, render_performances)
    from scoreperformer_b200.modules.sampling import top_k
    model = parity.build_model(dropout=False, device="cuda").eval()
    tok = TokenTables(**cases.table_kwargs())
    collator, messenger = cases.make_collator(), SPMuple2Messenger(tok)
    keep = [f for f in range(12) if f not in RENDERED]

    def piece_data(T, seed, first_bar):
        batch, perf = _piece(T, seed)
        b = {k: v.cuda() for k, v in batch.items()}
        with torch.inference_mode():
            enc = model.forward_encoders(perf=b["perf"], perf_mask=b["perf_mask"], score=b["score"], score_mask=b["score_mask"],
                                         bars=b["bars"], beats=b["beats"], onsets=b["onsets"], deadpan_mask=b["deadpan_mask"],
                                         compute_loss=False)
        perf = perf.clone()
        perf[:, 0] += first_bar                                           # a piece cut out of the middle of a score
        notes = perf.clone()
        notes[:, RENDERED] = 1
        notes = torch.cat([torch.full_like(notes[:1], 2), notes, torch.full_like(notes[:1], 3)])      # SOS ... EOS
        pad = lambda e: torch.cat([e[0, :1], e[0], e[0, -1:]]).clone()
        make = lambda: PerformanceData(perf_seq=perf.numpy(), notes=notes.cuda(), context=pad(enc.score_embeddings),
                                       embeddings=pad(enc.perf_embeddings), intermediates=SPMuple2IntermediateData(initial_tempo=96.))
        return perf, make

    specs = [piece_data(40, 5, 0), piece_data(64, 6, 7), piece_data(51, 7, 3)]
    pieces = [make() for _, make in specs]
    results = render_performances(model, messenger, collator, pieces, filter_kwargs={"k": 1})
    assert len(results) == 3
    for (perf, make), pd, (seq, messages) in zip(specs, pieces, results):
        n = perf.shape[0]
        assert seq.is_cuda and seq.shape == (n, 12) and pd.gen_seq.shape == (n + 1, 12) and pd.reached_eos
        got = seq.cpu()
        assert int((got == 1).sum()) == 0 and torch.equal(got[:, keep], perf[:, keep])
        assert messages.shape == (2 * n, 4)
        want_messages = messenger.tokens_to_messages(got.numpy(), intermediates=SPMuple2IntermediateData(initial_tempo=96.))
        assert np.array_equal(messages, want_messages)
        assert np.all(np.diff(messages[:, 0]) >= 0)                       # sorted by time

        gen = ScorePerformerGenerator(model, cases.make_dataset(tok, [perf.numpy()]), collator, messenger, device="cuda")
        gen.perf_data = make()
        loop_seq, loop_messages = gen.generate_performance_notes(time_window=1e9, filter_logits_fn=top_k, filter_kwargs={"k": 1})
        assert gen.perf_data.reached_eos and loop_seq.shape == (n, 12)
        agree = float((loop_seq[:, RENDERED] == seq[:, RENDERED]).float().mean())
        assert agree > 0.85, agree


def test_lookahead_rendering_on_device_equals_chord_by_chord_rendering():
    """`lookahead_notes`: several chords per decoder call on the CUDA decoder must render what chord-by-chord calls render (greedy),
    with fewer calls."""
    from scoreperformer_b200.inference import ScorePerformerGenerator, SPMuple2IntermediateData, SPMuple2Messenger, TokenTables
    from scoreperformer_b200.modules.sampling import top_k
    T = 64
    model = parity.build_model(dropout=False, device="cuda").eval()
    batch, perf = _piece(T, seed=78)
    b = {k: v.cuda() for k, v in batch.items()}
    with torch.inference_mode():
        enc = model.forward_encoders(perf=b["perf"], perf_mask=b["perf_mask"], score=b["score"], score_mask=b["score_mask"],
                                     bars=b["bars"], beats=b["beats"], onsets=b["onsets"], deadpan_mask=b["deadpan_mask"],
                                     compute_loss=False)
    notes = perf.clone()
    notes[1:, RENDERED] = 1
    notes = torch.cat([notes, torch.full_like(notes[:1], 3)])
    pad = lambda e: torch.cat([e[0], e[0, -1:]]).clone()
    tok = TokenTables(**cases.table_kwargs())

    def render(ahead):
        gen = ScorePerformerGenerator(model, cases.make_dataset(tok, [perf.numpy()]), cases.make_collator(), SPMuple2Messenger(tok),
                                      device="cuda")
        pd = gen.perf_data
        pd.notes, pd.context, pd.embeddings = notes.cuda(), pad(enc.score_embeddings), pad(enc.perf_embeddings)
        pd.intermediates = SPMuple2IntermediateData(initial_tempo=96.)
        calls, original = [0], model.perf_decoder.unmask_tokens

        def counted(*a, **k):
            calls[0] += 1
            return original(*a, **k)

        model.perf_decoder.unmask_tokens = counted
        try:
            t0, messages = 0., []
            for _ in range(400):
                _, m = gen.generate_performance_notes(start_time=t0, time_window=0.7, filter_logits_fn=top_k, filter_kwargs={"k": 1},
                                                      lookahead_notes=ahead)
                messages.extend(np.asarray(m).tolist())
                t0 += 0.7
                if pd.reached_eos:
                    break
        finally:
            del model.perf_decoder.unmask_tokens
        assert pd.reached_eos
        return pd.gen_seq, np.array(messages), calls[0]

    plain, plain_messages, plain_calls = render(0)
    ahead, ahead_messages, ahead_calls = render(12)
    assert torch.equal(plain, ahead) and np.array_equal(plain_messages, ahead_messages)
    assert ahead_calls < plain_calls, (ahead_calls, plain_calls)
