"""The render session of the streaming decoder calls (decode._RenderSession): staged weights, stack plan and buffers kept on the
device between the chord calls of real-time rendering.

Reference: the same calls with the session switched off, i.e. `render_decoder(start, kv_init)` per call -- staging, plan and
prepared terms rebuilt every time.  Tokens must be identical at every call and the returned keys / values bitwise equal."""
import contextlib

import numpy as np
import pytest
import torch

from tests import parity
from tests.test_render_session_host import fingerprint
import inference_cases as cases

pytestmark = pytest.mark.gpu

RENDERED = [3, 5, 10, 11]
CHORDS = [1, 3, 2, 1, 4, 2, 1, 1, 3, 2, 5, 1, 2, 3, 1, 2]


@contextlib.contextmanager
def _without_session():
    from scoreperformer_b200 import decode
    saved = decode._session_for
    decode._session_for = lambda *a, **k: None
    try:
        yield
    finally:
        decode._session_for = saved


def _sessions(model):
    from scoreperformer_b200 import decode
    return decode._SESSIONS.get(model.perf_decoder.model, {})


def _restages(model):
    return sum(s.restages for s in _sessions(model).values())


def _encoded(model, B, T, seed):
    batch = {k: v.cuda() for k, v in parity.make_batch(B, T, seed=seed, full_length=True, deadpan_last=False).items()}
    with torch.inference_mode():
        enc = model.forward_encoders(perf=batch["perf"], perf_mask=batch["perf_mask"], score=batch["score"], score_mask=batch["score_mask"],
                                     bars=batch["bars"], beats=batch["beats"], onsets=batch["onsets"], deadpan_mask=batch["deadpan_mask"],
                                     compute_loss=False)
    return batch["perf"], enc.score_embeddings.float(), enc.perf_embeddings.float()


def _kv(caches):
    return [torch.cat([a.keys, a.values], -1).clone() for a in caches.transformer.attention]


class _Piece:
    """A piece rendered chord by chord through `unmask_tokens` the way inference/generators.py calls it: a window [w0, n) of known
    notes plus the new chord, the caches of the window's prefix; a window longer than `max_len` restarts `keep` notes back without
    caches (so that call runs the general stepper and the next one continues the stepper's caches)."""

    def __init__(self, model, perf, ctx, sty, k=1, max_len=24, keep=12):
        self.model, self.ctx, self.sty, self.k, self.max_len, self.keep = model, ctx, sty, k, max_len, keep
        self.cur = perf.clone()
        self.cur[:, 1:, RENDERED] = 1
        self.n, self.w0, self.caches, self.i = 1, 0, None, 0

    def done(self):
        return self.n >= self.cur.shape[1]

    def step(self):
        from scoreperformer_b200.modules.sampling import top_k
        k = min(CHORDS[self.i % len(CHORDS)], self.cur.shape[1] - self.n)
        self.i += 1
        n = self.n + k
        if n - self.w0 > self.max_len:
            self.w0, self.caches = n - k - self.keep, None
        tokens = self.cur[:, self.w0:n].clone()
        masked = tokens.clone()
        masked[:, :, RENDERED] = 1
        with torch.inference_mode():
            out, self.caches = self.model.perf_decoder.unmask_tokens(
                tokens, masked, context=self.ctx[:, self.w0:n], style_embeddings=self.sty[:, self.w0:n], caches=self.caches,
                return_caches=True, filter_logits_fn=top_k, filter_kwargs={"k": self.k})
        self.cur[:, self.n:n] = out[:, -k:]
        self.n = n
        return out.clone(), _kv(self.caches)


def _render_alone(model, piece_args, k, seed=0):
    torch.manual_seed(seed)
    p = _Piece(model, *piece_args, k=k)
    calls = []
    while not p.done():
        calls.append(p.step())
    return calls, p.cur


def _assert_same_calls(got, want):
    assert len(got) == len(want)
    for i, ((o1, kv1), (o2, kv2)) in enumerate(zip(got, want)):
        assert torch.equal(o1, o2), f"call {i}: tokens differ"
        assert len(kv1) == len(kv2) and all(torch.equal(a.view(torch.int16), b.view(torch.int16)) for a, b in zip(kv1, kv2)), \
            f"call {i}: keys / values differ"


@pytest.mark.parametrize("k", [1, 8])
def test_batched_chord_calls_equal_call_by_call_rendering(k):
    model = parity.build_model(dropout=False, device="cuda").eval()
    args = _encoded(model, 3, 72, seed=11)
    with _without_session():
        want, want_seq = _render_alone(model, args, k)
    got, got_seq = _render_alone(model, args, k)
    _assert_same_calls(got, want)
    assert torch.equal(got_seq, want_seq)
    assert _sessions(model), "the streaming calls did not use the render session"


def _generator_run(model, lookahead, k, max_context_len):
    """The rendering loop in 0.35 s windows; every decoder call's tokens and returned keys / values."""
    from scoreperformer_b200.inference import ScorePerformerGenerator, SPMuple2IntermediateData, SPMuple2Messenger, TokenTables
    from scoreperformer_b200.modules.sampling import top_k
    from tests.test_inference_gpu import _piece
    T = 64
    batch, perf = _piece(T, seed=77)
    b = {kk: v.cuda() for kk, v in batch.items()}
    with torch.inference_mode():
        enc = model.forward_encoders(perf=b["perf"], perf_mask=b["perf_mask"], score=b["score"], score_mask=b["score_mask"],
                                     bars=b["bars"], beats=b["beats"], onsets=b["onsets"], deadpan_mask=b["deadpan_mask"],
                                     compute_loss=False)
    notes = perf.clone()
    notes[1:, RENDERED] = 1
    notes = torch.cat([notes, torch.full_like(notes[:1], 3)])
    pad = lambda e: torch.cat([e[0], e[0, -1:]]).clone()
    tok = TokenTables(**cases.table_kwargs())
    gen = ScorePerformerGenerator(model, cases.make_dataset(tok, [perf.numpy()]), cases.make_collator(), SPMuple2Messenger(tok), device="cuda")
    pd = gen.perf_data
    pd.notes, pd.context, pd.embeddings = notes.cuda(), pad(enc.score_embeddings), pad(enc.perf_embeddings)
    pd.intermediates = SPMuple2IntermediateData(initial_tempo=96.)
    calls, original = [], model.perf_decoder.unmask_tokens

    def recorded(*a, **kw):
        res, caches = original(*a, **kw)
        calls.append((res.clone(), _kv(caches), kw.get("caches") is None))
        return res, caches

    model.perf_decoder.unmask_tokens = recorded
    torch.manual_seed(5)
    try:
        t0, messages = 0., []
        for _ in range(400):
            _, m = gen.generate_performance_notes(start_time=t0, time_window=0.35, filter_logits_fn=top_k, filter_kwargs={"k": k},
                                                  lookahead_notes=lookahead, max_context_len=max_context_len)
            messages.extend(np.asarray(m).tolist())
            t0 += 0.35
            if pd.reached_eos:
                break
    finally:
        del model.perf_decoder.unmask_tokens
    assert pd.reached_eos
    return calls, pd.gen_seq, messages


@pytest.mark.parametrize("lookahead", [0, 12])
@pytest.mark.parametrize("k", [1, 8])
def test_generator_rendering_equals_call_by_call_rendering(lookahead, k):
    model = parity.build_model(dropout=False, device="cuda").eval()
    with _without_session():
        want, want_seq, want_msg = _generator_run(model, lookahead, k, max_context_len=24)
    got, got_seq, got_msg = _generator_run(model, lookahead, k, max_context_len=24)
    assert sum(fresh for _, _, fresh in got) > 2, "the windows were never truncated"
    _assert_same_calls([c[:2] for c in got], [c[:2] for c in want])
    assert torch.equal(got_seq, want_seq) and got_msg == want_msg


def test_prepared_rows_equal_whole_window_preparation():
    """Rows s..T-1 of P2 / C2 / AdaLN terms prepared on the new rows alone equal those rows of the whole-window preparation of
    render_decoder (M = B * T = 1200 rows: a whole-window GEMM takes its wide-tile configuration, the slice does not)."""
    from scoreperformer_b200 import decode, kernels as K
    from scoreperformer_b200.models.scoreperformer.transformer import TupleTransformerCaches
    from scoreperformer_b200.modules.transformer.attend import AttentionIntermediates
    from scoreperformer_b200.modules.transformer.transformer import TransformerIntermediates
    model = parity.build_model(dropout=False, device="cuda").eval()
    dec = model.perf_decoder.model
    B, T, s = 3, 400, 390
    perf, ctx, sty = _encoded(model, B, T, seed=12)
    masked = perf.clone()
    masked[:, :, RENDERED] = 1
    tokens = perf.clone()
    tokens[:, s + 1:, RENDERED] = 1
    g = torch.Generator(device="cuda").manual_seed(0)
    att = [AttentionIntermediates(torch.randn(B, s, 64, device="cuda", generator=g).to(torch.bfloat16),
                                  torch.randn(B, s, 64, device="cuda", generator=g).to(torch.bfloat16)) for _ in range(dec.transformer.depth)]
    z = torch.zeros(B, s, 256, device="cuda")
    caches = TupleTransformerCaches(token_emb=z, transformer=TransformerIntermediates(hiddens=[z] * 5, attention=att))
    with torch.inference_mode():
        session = decode._session_for(dec, tokens, RENDERED, 1, sty)
        session.render(dec, tokens.clone(), masked, ctx, sty, None, RENDERED, 1.0, 1, s, caches)
        # the whole-window preparation as render_decoder does it
        w = decode._DecoderWeights(dec)
        _, b_comp = w.compose_front()
        sizes, F, Dm = dec.token_emb.field_sizes, perf.shape[-1], dec.dim
        x2, _, _ = K.embed_ln_fwd(masked.reshape(-1, F).contiguous(), w.table, sizes, w.ln_w, w.ln_b)
        x2p = K.gemm(x2, w.wp16, bias=w.bp, out_dtype=torch.bfloat16)
        P2 = K.gemm(x2p, w.wm_r, bias=w.bm + b_comp, out_dtype=torch.float32).view(B, T, Dm)
        ctx16 = K.cast_bf16(ctx.contiguous().view(B * T, -1))
        C2 = K.gemm(ctx16, w.wc_r, bias=w.bc, out_dtype=torch.float32).view(B, T, Dm)
        gb = session.plan.prepare_adaln(sty.contiguous())
    torch.cuda.synchronize()
    assert torch.equal(session.P2[:, s:T].view(torch.int32), P2[:, s:].view(torch.int32))
    assert torch.equal(session.C2[:, s:T].view(torch.int32), C2[:, s:].view(torch.int32))
    assert torch.equal(session.gb_all[:, s:T].view(torch.int16), gb[:, s:].view(torch.int16))


def _modify_train_step(model, ts, batch):
    model.train()
    ts.step(batch)
    model.eval()


@pytest.mark.parametrize("change", ["train_step", "load_state_dict", "data_add", "value_mlp_element"])
def test_weight_changes_restage_the_session(change):
    from scoreperformer_b200.train_step import TrainStep
    model = parity.build_model(dropout=False, device="cuda")
    dec = model.perf_decoder.model
    ts = None
    if change == "train_step":                      # the flat buffers exist before the session: only the fingerprint can tell
        model.perf_encoder.exact_latent_shapes = False
        ts = TrainStep(model, lr=1e-3, use_graph=False)
        train_batch = {k: v.cuda() for k, v in parity.make_batch(2, 48, seed=5).items()}
        _modify_train_step(model, ts, train_batch)  # the encoder's lazily made state is then made outside inference mode
    model.eval()
    args = _encoded(model, 1, 40, seed=13)
    torch.manual_seed(0)
    piece = _Piece(model, *args, max_len=1000)
    for _ in range(3):
        piece.step()
    assert _restages(model) == 1
    session = next(iter(_sessions(model).values()))
    fp = int(session.state[0])
    piece.step()
    assert _restages(model) == 1 and int(session.state[0]) == fp         # unchanged weights: stable fingerprint, nothing restaged

    if change == "train_step":
        _modify_train_step(model, ts, train_batch)
    elif change == "load_state_dict":
        model.load_state_dict(parity.build_model(dropout=False, seed_weights=1, device="cuda").state_dict())
    elif change == "data_add":
        dec.transformer.layers[2][1].to_out.weight.data.add_(1e-2)
    else:
        with torch.no_grad():
            dec.token_emb.embs["Velocity"].value_layer[1][0].weight[3, 7] += 0.25
    # the next streaming call restages and renders what a fresh rendering with the new weights renders from the same state
    saved = (piece.cur.clone(), piece.n, piece.w0, piece.caches, piece.i)
    with _without_session():
        want = piece.step()
    piece.cur, piece.n, piece.w0, piece.caches, piece.i = saved
    got = piece.step()
    _assert_same_calls([got], [want])
    assert _restages(model) == 2 and int(session.state[0]) != fp
    piece.step()
    assert _restages(model) == 2


def test_interleaved_pieces_and_kept_caches():
    model = parity.build_model(dropout=False, device="cuda").eval()
    a_args, b_args = _encoded(model, 1, 48, seed=21), _encoded(model, 1, 48, seed=22)
    want_a, _ = _render_alone(model, a_args, 1)
    want_b, _ = _render_alone(model, b_args, 1)
    pa, pb = _Piece(model, *a_args), _Piece(model, *b_args)
    got_a, got_b = [], []
    kept, kept_rows = None, None
    while not (pa.done() and pb.done()):
        if not pa.done():
            got_a.append(pa.step())
            if len(got_a) == 3:                     # a cache object handed out earlier keeps its rows after later calls
                kept, kept_rows = pa.caches, _kv(pa.caches)
        if not pb.done():
            got_b.append(pb.step())
    _assert_same_calls(got_a, want_a)
    _assert_same_calls(got_b, want_b)
    assert all(torch.equal(x, y) for x, y in zip(_kv(kept), kept_rows))


def test_stepper_caches_continue_on_the_session(monkeypatch):
    """Caches the general stepper produced (SPB_STREAM=legacy) are copied into the session and continued."""
    model = parity.build_model(dropout=False, device="cuda").eval()
    args = _encoded(model, 1, 40, seed=23)
    piece = _Piece(model, *args, max_len=1000)
    monkeypatch.setenv("SPB_STREAM", "legacy")
    for _ in range(3):
        piece.step()
    assert not _sessions(model)
    monkeypatch.delenv("SPB_STREAM")
    saved = (piece.cur.clone(), piece.n, piece.w0, piece.caches, piece.i)
    with _without_session():
        want = [piece.step() for _ in range(3)]
    piece.cur, piece.n, piece.w0, piece.caches, piece.i = saved
    got = [piece.step() for _ in range(3)]
    _assert_same_calls(got, want)
    assert _sessions(model)


def test_session_begin_in_isolation():
    """The begin kernel alone (no stack kernel): fingerprint equal to the numpy statement, stale flag, advance words cleared,
    start position written; tensors of odd lengths and unaligned starts take the kernel's scalar paths."""
    from scoreperformer_b200 import kernels as K
    g = torch.Generator(device="cuda").manual_seed(1)
    base = torch.randn(1 << 20, device="cuda", generator=g)
    tensors = [base[:333], base[1001:1001 + 4097], base[8192:8192 + 64], torch.randn(5, 7, device="cuda", generator=g),
               torch.randint(-2 ** 31, 2 ** 31 - 1, (1023,), dtype=torch.int32, device="cuda", generator=g), base[1 << 19:]]
    model = parity.build_model(dropout=False, device="cuda")
    tensors += list(model.perf_decoder.model.parameters()) + list(model.perf_decoder.model.buffers())
    tensors = [t.detach() for t in tensors]
    table = K.fingerprint_table(tensors)
    state = torch.zeros(4, dtype=torch.int64, device="cuda")
    advance = torch.tensor([5, 7], dtype=torch.int32, device="cuda")
    pos = torch.tensor([99], dtype=torch.int64, device="cuda")
    want = fingerprint([t.cpu().numpy() for t in tensors])
    u64 = lambda v: int(v) & ((1 << 64) - 1)
    K.session_begin(table, state, advance, pos, 17)
    torch.cuda.synchronize()
    assert advance.tolist() == [0, 0] and int(pos) == 17
    assert u64(state[0]) == want and int(state[1]) == 0 and int(state[2]) == 0 and int(state[3]) == 1
    advance.fill_(3)
    K.session_begin(table, state, advance, pos, 0)
    torch.cuda.synchronize()
    assert advance.tolist() == [0, 0] and int(pos) == 0 and u64(state[0]) == want and int(state[3]) == 0
    tensors[1][100] = -tensors[1][100]
    K.session_begin(table, state, advance, pos, 3)
    torch.cuda.synchronize()
    assert int(state[3]) == 1 and u64(state[0]) == fingerprint([t.cpu().numpy() for t in tensors]) != want


def test_launches_per_streaming_call():
    """A continuing call launches session_begin + the terms of its new rows (at most 8 package launches) + 6 per note."""
    from scoreperformer_b200 import kernels as K
    model = parity.build_model(dropout=False, device="cuda").eval()
    args = _encoded(model, 1, 40, seed=24)
    counts = {}
    for mode in ("parent", "session"):
        piece = _Piece(model, *args, max_len=1000)
        ctx = _without_session() if mode == "parent" else contextlib.nullcontext()
        with ctx:
            for _ in range(4):
                piece.step()
            rows = []
            for _ in range(6):
                n0 = piece.n
                before = K.LAUNCHES
                piece.step()
                rows.append((piece.n - n0, K.LAUNCHES - before))
        counts[mode] = rows
    print("package launches per continuing call (notes, launches):", counts)
    for notes, launches in counts["session"]:
        assert launches <= 8 + 6 * notes, counts
    assert all(s[1] < p[1] for s, p in zip(counts["session"], counts["parent"]))
