"""Top-p, top-a and per-field token bans in the heads + sampling kernel (csrc/decode_stack.cu `sample_fields_kernel`) and in batched
rendering, against an fp32 torch statement of the reference's filters (modules/sampling.py) on the same bf16 inputs."""
import numpy as np
import pytest
import torch

from tests import parity
import inference_cases as cases

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
SIZES = [260, 132, 92, 132, 133, 125, 26, 69, 16, 16, 165, 85]
OFFS = [int(x) for x in np.concatenate([[0], np.cumsum(SIZES[:-1])])]
FIELDS = [3, 5, 10, 11]
T, F = 6, 12
N_DRAW = 4096
EDGE = 1e-4          # tokens whose filter membership is this close to the threshold are exempt (bf16 products, other sum order)


@pytest.fixture(scope="module")
def heads():
    """bf16 head projections e [64, F * 128] and the tied table, the fp32 logits of the rendered fields (PAD / MASK banned)."""
    torch.manual_seed(12)
    table = (torch.randn(sum(SIZES), 128, device="cuda") * 0.3).to(BF16)
    e = torch.randn(64, F * 128, device="cuda")
    e[1] *= 0.25                                                 # a flatter row: many tokens inside the nucleus
    e = e.to(BF16)
    logits = {f: e[:, f * 128:(f + 1) * 128].float() @ table[OFFS[f]:OFFS[f] + SIZES[f]].float().t() for f in FIELDS}
    for f in FIELDS:
        logits[f][:, :2] = -float("inf")
    return e, table, logits


def _draw(k, e, table, row, seeds, temperature=1.0, topk=1, **filters):
    """Tokens [len(seeds) * N_DRAW, len(FIELDS)] drawn from row `row` of e repeated N_DRAW times, one launch per seed."""
    e1 = e[row:row + 1].repeat(N_DRAW, 1).contiguous()
    pos = torch.tensor([2], device="cuda")
    out = []
    for seed in seeds:
        tok = torch.zeros(N_DRAW, T, F, dtype=torch.int64, device="cuda")
        k.sample_fields(e1, table, FIELDS, [OFFS[f] for f in FIELDS], [SIZES[f] for f in FIELDS], [topk] * len(FIELDS), tok, pos,
                        temperature=temperature, seed=seed, **filters)
        out.append(tok[:, 3, FIELDS])
    return torch.cat(out)


def _statement(lg, top_p=None, top_a=None):
    """(kept bool [V], exempt bool [V]) of the reference filter on one fp32 row of logits (banned = -inf)."""
    from scoreperformer_b200.modules.sampling import top_a as ref_top_a, top_p as ref_top_p
    lg = lg[None].double()
    probs = torch.softmax(lg, -1)[0]
    if top_p is not None:
        kept = torch.isfinite(ref_top_p(lg.clone(), top_p))[0]
        val, ind = torch.sort(lg[0], descending=True, stable=True)
        before = torch.cumsum(torch.softmax(val, -1), 0) - torch.softmax(val, -1)              # mass ranked ahead of each token
        exempt = torch.zeros_like(kept)
        exempt[ind] = ((before - top_p).abs() < EDGE) & (torch.arange(len(ind), device=lg.device) > 0)
    else:
        kept = torch.isfinite(ref_top_a(lg.clone(), *top_a))[0]
        limit = probs.max() ** top_a[0] * top_a[1]
        exempt = (probs - limit).abs() < 1e-3 * limit                                 # relative: limits can be tiny
    return kept & torch.isfinite(lg[0]), exempt & torch.isfinite(lg[0])


def _check(drawn, lg, kept, exempt, temperature, tag, bound=0.04):
    """Every draw in the kept set (or exempt); frequencies within `bound` of the renormalised softmax at the temperature."""
    V = lg.numel()
    ok = kept | exempt
    assert bool(ok[drawn].all()), (tag, sorted(set(drawn[~ok[drawn]].tolist())))
    assert not bool(torch.isinf(lg[drawn]).any()), tag                               # PAD / MASK / banned never drawn
    if bool(exempt.any()):
        return                                                                        # the kept set itself is uncertain
    want = torch.softmax(torch.where(kept, lg.double(), -float("inf")) / temperature, -1)
    got = torch.bincount(drawn, minlength=V).double() / drawn.numel()
    err = float((got - want).abs().max())
    assert err < bound, (tag, err)


@pytest.mark.parametrize("temperature", [0.7, 1.0, 1.5])
@pytest.mark.parametrize("thres", [0.05, 0.5, 0.9, 0.999])
def test_top_p_matches_statement(heads, thres, temperature):
    from scoreperformer_b200 import kernels as k
    e, table, logits = heads
    for row in (0, 1):
        drawn = _draw(k, e, table, row, seeds=(11, 12, 13), temperature=temperature, top_p=[thres] * 4)
        for j, f in enumerate(FIELDS):
            lg = logits[f][row]
            kept, exempt = _statement(lg, top_p=thres)
            _check(drawn[:, j], lg, kept, exempt, temperature, (row, f, thres, temperature))


@pytest.mark.parametrize("params", [(2.0, 0.02), (1.0, 0.5)])
@pytest.mark.parametrize("temperature", [0.7, 1.5])
def test_top_a_matches_statement(heads, params, temperature):
    from scoreperformer_b200 import kernels as k
    e, table, logits = heads
    for row in (0, 1):
        drawn = _draw(k, e, table, row, seeds=(21, 22, 23), temperature=temperature, top_a=[params] * 4)
        for j, f in enumerate(FIELDS):
            lg = logits[f][row]
            kept, exempt = _statement(lg, top_a=params)
            _check(drawn[:, j], lg, kept, exempt, temperature, (row, f, params, temperature))


def test_bans_come_before_every_filter(heads):
    """Per-field bans, the arg-max among them: never drawn, and the filters see the logits without them (top-k 5 included)."""
    from scoreperformer_b200 import kernels as k
    e, table, logits = heads
    gen = torch.Generator().manual_seed(3)
    for row in (0, 1):
        bans = []
        for f in FIELDS:
            extra = torch.randint(2, SIZES[f], (6,), generator=gen).tolist()
            bans.append(sorted(set(extra) | {int(logits[f][row].argmax())}))
        lgs = []
        for f, ids in zip(FIELDS, bans):
            lg = logits[f][row].clone()
            lg[ids] = -float("inf")
            lgs.append(lg)
        for name, kw in (("top_p", dict(top_p=[0.8] * 4)), ("top_a", dict(top_a=[(2.0, 0.02)] * 4)), ("top_k", dict(topk=5))):
            drawn = _draw(k, e, table, row, seeds=(31, 32), temperature=1.2, banned=bans, **kw)
            for j, (f, lg, ids) in enumerate(zip(FIELDS, lgs, bans)):
                assert not bool(torch.isin(drawn[:, j], torch.tensor(ids, device="cuda")).any()), (name, f)
                if name == "top_k":
                    val, ind = lg.topk(5)
                    kept = torch.zeros_like(lg, dtype=torch.bool)
                    kept[ind[torch.isfinite(val)]] = True
                    exempt = torch.zeros_like(kept)
                else:
                    kept, exempt = _statement(lg, **({"top_p": 0.8} if name == "top_p" else {"top_a": (2.0, 0.02)}))
                _check(drawn[:, j], lg, kept, exempt, 1.2, (name, row, f))


def test_top_p_limits(heads):
    """thres = 0 is the arg-max, token for token (near-ties exempt); thres >= 1 reaches the full softmax."""
    from scoreperformer_b200 import kernels as k
    e, table, logits = heads
    tokens = torch.zeros(e.shape[0], T, F, dtype=torch.int64, device="cuda")
    pos = torch.tensor([2], device="cuda")
    k.sample_fields(e, table, FIELDS, [OFFS[f] for f in FIELDS], [SIZES[f] for f in FIELDS], [1] * 4, tokens, pos, temperature=1.3,
                    seed=5, top_p=[0.0] * 4)
    for f in FIELDS:
        top2 = logits[f].topk(2, dim=-1).values
        clear = (top2[:, 0] - top2[:, 1]) > 1e-3
        assert torch.equal(tokens[clear, 3, f], logits[f].argmax(-1)[clear]), f
    for thres in (1.0, 3.0):
        for row in (0, 1):
            drawn = _draw(k, e, table, row, seeds=(41, 42, 43), temperature=1.5, top_p=[thres] * 4)
            for j, f in enumerate(FIELDS):
                lg = logits[f][row]
                _check(drawn[:, j], lg, torch.isfinite(lg), torch.zeros_like(lg, dtype=torch.bool), 1.5, (thres, row, f))


@pytest.mark.parametrize("topk", [1, 5, 32])
def test_filters_off_draw_what_the_plain_entry_draws(heads, topk):
    """spb_sample_fields_filtered with every filter off (and an empty ban set) returns exactly spb_sample_fields' tokens."""
    from scoreperformer_b200 import kernels as k
    e, table, _ = heads
    e_many = e.repeat(64, 1).contiguous()                           # 4096 scores, 64 distinct rows
    pos = torch.tensor([2], device="cuda")
    outs = []
    for kw in ({}, dict(top_p=[-1.0] * 4, top_a=[None] * 4, banned=[[]] * 4), dict(banned=[[]] * 4)):
        tok = torch.zeros(e_many.shape[0], T, F, dtype=torch.int64, device="cuda")
        k.sample_fields(e_many, table, FIELDS, [OFFS[f] for f in FIELDS], [SIZES[f] for f in FIELDS], [topk] * 4, tok, pos,
                        temperature=0.9, seed=77, **kw)
        outs.append(tok)
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


# ------------------------------------------------------------------ batched rendering
@pytest.fixture(scope="module")
def render_setup():
    g = parity.golden("render_t24.npz")
    model = parity.build_model(dropout=False, device="cuda").eval()
    batch = parity.make_batch(1, int(g["T"]), seed=int(g["seed"]), full_length=True, deadpan_last=False)
    b = {kk: v.cuda() for kk, v in batch.items()}
    with torch.inference_mode():
        enc = model.forward_encoders(perf=b["perf"], perf_mask=b["perf_mask"], score=b["score"], score_mask=b["score_mask"], bars=b["bars"],
                                     beats=b["beats"], onsets=b["onsets"], deadpan_mask=b["deadpan_mask"], compute_loss=False)
    rep = lambda t: t.repeat(3, *([1] * (t.dim() - 1)))
    tokens_in = rep(torch.from_numpy(g["tokens_in"]).cuda())
    args = (tokens_in, rep(b["masked_perf"]), rep(enc.score_embeddings), rep(enc.perf_embeddings))
    return model, args, rep(b["perf_mask"])


def test_render_batch_top_p_on_the_fused_step(render_setup):
    from scoreperformer_b200 import kernels as K
    from scoreperformer_b200.decode import render_batch
    model, args, mask = render_setup
    launches = {}
    outs = {}
    for name, kw in (("greedy", dict(top_k=1)), ("p0", dict(top_p=0.0)), ("p9", dict(top_p=0.9, top_k=None))):
        torch.manual_seed(9)
        K.LAUNCHES = 0
        outs[name] = render_batch(model, *args, mask=mask, **kw)
        launches[name] = K.LAUNCHES
    assert torch.equal(outs["p0"], outs["greedy"])
    assert launches["p9"] == launches["greedy"] == launches["p0"], launches
    torch.manual_seed(9)
    again = render_batch(model, *args, mask=mask, top_p=0.9, top_k=None)
    assert torch.equal(again, outs["p9"])
    assert int((outs["p9"] == 1).sum()) == int((args[0][:, 0] == 1).sum())   # every MASK after note 0 was filled
    keep = [f for f in range(12) if f not in FIELDS]
    assert torch.equal(outs["p9"][..., keep], args[0][..., keep])


@pytest.mark.parametrize("decode", ["fused", "legacy"])
def test_render_batch_bans_and_top_a(render_setup, decode, monkeypatch):
    """Bans hold on the fused step and on the launch-per-operator step with host-side sampling (top-p / top-a of modules.sampling)."""
    monkeypatch.setenv("SPB_DECODE", decode)
    from scoreperformer_b200.decode import render_batch
    model, args, mask = render_setup
    greedy = render_batch(model, *args, mask=mask)
    bans = {f: sorted(set(greedy[:, 1:, f].flatten().tolist())) for f in (3, 10)}  # every token greedy decoding chose
    for kw in (dict(top_p=0.9), dict(top_a=(2.0, 0.02)), dict(top_p=0.0)):
        torch.manual_seed(4)
        out = render_batch(model, *args, mask=mask, banned_tokens=bans, **kw)
        assert int((out == 1).sum()) == int((args[0][:, 0] == 1).sum()), kw
        for f, ids in bans.items():
            assert not bool(torch.isin(out[:, 1:, f], torch.tensor(ids, device="cuda")).any()), (kw, f)


def test_render_performances_top_p():
    """Pieces of different lengths through `render_performances` with the reference's top_p: every MASK filled, given fields kept,
    messages exactly the messenger's decoding of the returned tuples; the same torch seed renders the same pieces."""
    from scoreperformer_b200.inference import PerformanceData, SPMuple2IntermediateData, SPMuple2Messenger, TokenTables, render_performances
    from scoreperformer_b200.modules.sampling import top_p
    model = parity.build_model(dropout=False, device="cuda").eval()
    tok = TokenTables(**cases.table_kwargs())
    collator, messenger = cases.make_collator(), SPMuple2Messenger(tok)
    keep = [f for f in range(12) if f not in FIELDS]

    def piece(T_, seed):
        batch = parity.make_batch(1, T_, seed=seed, full_length=True, deadpan_last=False)
        onset = batch["onsets"][0] - 4
        perf = batch["perf"][0].clone()
        perf[:, 0] = 4 + onset // 12
        perf[:, 1] = 4 + (onset % 12) * 2
        perf[:, 6] = 4
        batch["perf"][0] = perf
        batch["score"][0] = perf[:, :10]
        b = {kk: v.cuda() for kk, v in batch.items()}
        with torch.inference_mode():
            enc = model.forward_encoders(perf=b["perf"], perf_mask=b["perf_mask"], score=b["score"], score_mask=b["score_mask"],
                                         bars=b["bars"], beats=b["beats"], onsets=b["onsets"], deadpan_mask=b["deadpan_mask"],
                                         compute_loss=False)
        notes = perf.clone()
        notes[:, FIELDS] = 1
        notes = torch.cat([torch.full_like(notes[:1], 2), notes, torch.full_like(notes[:1], 3)])
        pad = lambda x: torch.cat([x[0, :1], x[0], x[0, -1:]]).clone()
        return perf, lambda: PerformanceData(perf_seq=perf.numpy(), notes=notes.cuda(), context=pad(enc.score_embeddings),
                                             embeddings=pad(enc.perf_embeddings), intermediates=SPMuple2IntermediateData(initial_tempo=96.))

    specs = [piece(40, 5), piece(64, 6), piece(51, 7)]
    runs = []
    for _ in range(2):
        torch.manual_seed(17)
        runs.append(render_performances(model, messenger, collator, [make() for _, make in specs], filter_kwargs={"thres": 0.8},
                                        filter_logits_fn=top_p))
    for (perf, _), (seq, messages), (seq2, _) in zip(specs, runs[0], runs[1]):
        n = perf.shape[0]
        got = seq.cpu()
        assert got.shape == (n, 12) and int((got == 1).sum()) == 0 and torch.equal(got[:, keep], perf[:, keep])
        want = messenger.tokens_to_messages(got.numpy(), intermediates=SPMuple2IntermediateData(initial_tempo=96.))
        assert np.array_equal(messages, want)
        assert torch.equal(seq, seq2)
