"""CPU: the top-p / top-a / per-token-ban request of batched rendering -- argument checks of the C entry point and of
`decode.render_decoder`, and how `inference.render_performances` maps the reference's filter functions onto `render_batch`."""
import ctypes
import math
import types

import numpy as np
import pytest
import torch

import inference_cases as cases
from scoreperformer_b200 import lib as spb_lib

SIZES = [260, 132, 92, 132, 133, 125, 26, 69, 16, 16, 165, 85]
RENDERED = [3, 5, 10, 11]


# ------------------------------------------------------------------ C entry point: rejected before any launch
def _filtered(top_p=None, a_pow=None, a_ratio=None, bans=None, n_banned=2, vocab=(132, 125, 165, 85)):
    """Calls spb_sample_fields_filtered with placeholder device pointers: only requests the argument checks reject may go here."""
    spb_lib.build()
    n = len(vocab)
    ints = lambda xs: (ctypes.c_int * n)(*xs)
    floats = lambda xs: None if xs is None else (ctypes.c_float * n)(*xs)
    bits = None if bans is None else (ctypes.c_uint32 * (8 * n))(*bans)
    fake = ctypes.c_void_p(16)
    rc = spb_lib.lib().spb_sample_fields_filtered(fake, 12 * 128, fake, ints(RENDERED), ints([0] * n), ints(vocab), ints([1] * n), n,
                                                 n_banned, 1.0, 0, fake, fake, 4, 8, 12, None, floats(top_p), floats(a_pow),
                                                 floats(a_ratio), bits, None)
    return rc, spb_lib.lib().spb_last_error().decode()


def test_filtered_entry_rejects_bad_filters():
    rc, msg = _filtered(top_p=[0.5, -1, -1, -1], a_pow=[2, 2, 2, 2], a_ratio=[0.02, 0, 0, 0])
    assert rc == -1 and "at most one of top-p and top-a" in msg
    for bad in (float("nan"), float("inf")):
        rc, msg = _filtered(top_p=[0.5, bad, -1, -1])
        assert rc == -1 and "top_p must be finite" in msg
        rc, msg = _filtered(a_pow=[2, bad, 2, 2], a_ratio=[0.02] * 4)
        assert rc == -1 and "top-a parameters must be finite" in msg
    rc, msg = _filtered(a_pow=[2, 2, 2, 2])
    assert rc == -1 and "go together" in msg
    # a field whose every token is banned: field 11 (V 85) with PAD / MASK by n_banned and the rest by the mask
    words = [0] * 24 + [0xFFFFFFFF, 0xFFFFFFFF, 0x1FFFFF, 0, 0, 0, 0, 0]
    rc, msg = _filtered(bans=words)
    assert rc == -1 and "field 11: every token is banned" in msg
    rc, msg = _filtered(top_p=[0.5] * 4, vocab=(132, 300, 165, 85))
    assert rc == -1 and "V <= 256" in msg


# ------------------------------------------------------------------ render_decoder: request checks (before any device work)
def _fake_decoder():
    return types.SimpleNamespace(token_emb=types.SimpleNamespace(field_sizes=SIZES), lm_head=None)


@pytest.mark.parametrize("kw, match", [
    (dict(top_p=0.9, top_k=5), "cannot be combined"),
    (dict(top_a=(2.0, 0.02), top_k=None, top_p=0.5), "at most one"),
    (dict(top_a=(2.0, 0.02), top_k=[1, 1, 1, 1]), "cannot be combined"),
    (dict(top_p=-0.1), "finite threshold >= 0"),
    (dict(top_p=float("nan")), "finite threshold >= 0"),
    (dict(top_p=float("inf")), "finite threshold >= 0"),
    (dict(top_a=(2.0, 0.0)), "min_p_ratio > 0"),
    (dict(top_a=(float("inf"), 0.02)), "finite"),
    (dict(banned_tokens={11: [4, 85]}), r"ids \[85\] are outside its vocabulary of 85"),
    (dict(banned_tokens={5: [-1]}), "outside its vocabulary"),
    (dict(banned_tokens={0: [4]}), "not rendered"),
    (dict(banned_tokens={8: list(range(2, 16))}, fields=(8,)), "leave no token"),
])
def test_render_decoder_rejects_bad_requests(kw, match):
    from scoreperformer_b200.decode import render_decoder
    fields = kw.pop("fields", RENDERED)
    x = torch.zeros(1, 4, 12, dtype=torch.int64)
    with pytest.raises(ValueError, match=match):
        render_decoder(_fake_decoder(), x, x, torch.zeros(1, 4, 256), torch.zeros(1, 4, 64), fields=fields, **kw)


def test_filter_request_accepts_and_lists_bans():
    from scoreperformer_b200.decode import _check_filters
    assert _check_filters(1, 0.0, None, None, RENDERED, SIZES) == [[], [], [], []]
    assert _check_filters(None, None, (2.0, 0.02), None, RENDERED, SIZES) == [[], [], [], []]
    bans = _check_filters(1, 0.5, None, {10: [7, 5, 7], 3: (131,)}, RENDERED, SIZES)
    assert bans == [[131], [], [5, 7], []]
    assert _check_filters(None, None, None, {8: list(range(2, 15))}, (8,), SIZES) == [list(range(2, 15))]     # token 15 is left


# ------------------------------------------------------------------ render_performances -> render_batch
@pytest.fixture
def recorder(monkeypatch):
    from scoreperformer_b200 import decode
    calls = []

    def fake_render_batch(model, tokens, masked, context, style, **kw):
        calls.append(kw)
        out = tokens.clone()
        out[out == 1] = 4                                        # the lowest real token of every field
        return out

    monkeypatch.setattr(decode, "render_batch", fake_render_batch)
    return calls


def _pieces():
    from scoreperformer_b200.inference import PerformanceData, SPMuple2IntermediateData
    pieces = []
    for n, seed in ((9, 1), (14, 2)):
        perf = torch.from_numpy(cases.make_piece(n, seed))
        notes = perf.clone()
        notes[:, RENDERED] = 1
        notes = torch.cat([torch.full_like(notes[:1], 2), notes, torch.full_like(notes[:1], 3)])
        pieces.append(PerformanceData(perf_seq=perf.numpy(), notes=notes, context=torch.zeros(n + 2, 256),
                                      embeddings=torch.zeros(n + 2, 64), intermediates=SPMuple2IntermediateData(initial_tempo=96.)))
    return pieces


def _render(calls, fn=None, kw=None, **extra):
    from scoreperformer_b200.inference import SPMuple2Messenger, TokenTables, render_performances
    model = types.SimpleNamespace(perf_decoder=types.SimpleNamespace(model=_fake_decoder()))
    messenger = SPMuple2Messenger(TokenTables(**cases.table_kwargs()))
    calls.clear()
    args = {} if fn is None else {"filter_logits_fn": fn}
    results = render_performances(model, messenger, cases.make_collator(), _pieces(), filter_kwargs=kw, **args, **extra)
    assert len(calls) == 1 and len(results) == 2
    return calls[0]


def test_render_performances_default_call_is_unchanged(recorder):
    """The arguments `render_batch` received before top-p / top-a existed: top_k from `k`, else None (ceil(0.1 V))."""
    for kw, k in ((None, None), ({}, None), ({"k": 1}, 1), ({"k": 7}, 7), ({"k": None}, None)):
        got = _render(recorder, kw=kw, temperature=0.8)
        assert set(got) == {"mask", "fields", "temperature", "top_k"}, got.keys()
        assert got["top_k"] == k and got["fields"] == RENDERED and got["temperature"] == 0.8
        assert got["mask"].tolist() == [[True] * 10 + [False] * 5, [True] * 15]


def test_render_performances_maps_reference_filters(recorder):
    from scoreperformer_b200.modules.sampling import top_a, top_k, top_p
    strip = lambda d: {k: v for k, v in d.items() if k not in ("mask", "fields", "temperature")}
    assert strip(_render(recorder, top_k, {"k": 3})) == {"top_k": 3}
    assert strip(_render(recorder, top_k, {"thres": 0.9, "k": 5})) == {"top_k": 5}
    # thres alone: the reference's k = ceil((1 - thres) V) of each rendered field's head
    assert strip(_render(recorder, top_k, {"thres": 0.5})) == {"top_k": [math.ceil(0.5 * SIZES[f]) for f in RENDERED]}
    assert strip(_render(recorder, top_k, {"thres": 0.9})) == {"top_k": [math.ceil((1 - 0.9) * SIZES[f]) for f in RENDERED]}
    assert strip(_render(recorder, top_p)) == {"top_p": 0.9}
    assert strip(_render(recorder, top_p, {"thres": 0.5})) == {"top_p": 0.5}
    assert strip(_render(recorder, top_p, {"thres": 0})) == {"top_p": 0.0}
    assert strip(_render(recorder, top_a)) == {"top_a": (2.0, 0.02)}
    assert strip(_render(recorder, top_a, {"min_p_ratio": 0.1})) == {"top_a": (2.0, 0.1)}
    assert strip(_render(recorder, top_a, {"min_p_pow": 1.5, "min_p_ratio": 0.2})) == {"top_a": (1.5, 0.2)}

    # the same functions of the original package (module scoreperformer.modules.sampling) are recognised by name
    def original(fn):
        clone = types.FunctionType(fn.__code__, fn.__globals__, fn.__name__, fn.__defaults__)
        clone.__module__ = "scoreperformer.modules.sampling"
        return clone
    assert strip(_render(recorder, original(top_p), {"thres": 0.3})) == {"top_p": 0.3}
    assert strip(_render(recorder, original(top_k), {"k": 2})) == {"top_k": 2}


@pytest.mark.parametrize("fn, kw, match", [
    ("other", None, "top_k, top_p or top_a"),
    ("top_p", {"k": 3}, r"top_p takes \['thres'\], not \['k'\]"),
    ("top_k", {"k": 1, "temperature": 2.0}, "not \\['temperature'\\]"),
    ("top_a", {"thres": 0.5}, "top_a takes"),
])
def test_render_performances_rejects_what_it_cannot_render(recorder, fn, kw, match):
    from scoreperformer_b200.modules import sampling
    f = (lambda logits, **_: logits) if fn == "other" else getattr(sampling, fn)
    with pytest.raises(ValueError, match=match):
        _render(recorder, f, kw)
    assert recorder == []
