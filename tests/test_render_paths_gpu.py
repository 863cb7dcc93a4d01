"""The note-step configurations of `decode.render_decoder`: one input front, the stack chosen by the plan, the sampler chosen by
`fused_sampling`.  Launches per note-step, agreement of every configuration with the default one on teacher-forced inputs, and
graph replay against eager steps where the sampling kernel ends the step without the stack kernel's in-kernel front."""
import pytest
import torch

from tests import parity

pytestmark = pytest.mark.gpu

FIELDS = [3, 5, 10, 11]


@pytest.fixture(scope="module")
def model():
    return parity.build_model(dropout=False, device="cuda").eval()


def _inputs(model, B, T, seed):
    """(tokens with note 0 complete and the rest MASKed, masked_perf, score embeddings, style embeddings, mask, teacher)."""
    b = {k: v.cuda() for k, v in parity.make_batch(B, T, seed=seed, deadpan_last=False).items()}
    with torch.inference_mode():
        enc = model.forward_encoders(perf=b["perf"], perf_mask=b["perf_mask"], score=b["score"], score_mask=b["score_mask"], bars=b["bars"],
                                     beats=b["beats"], onsets=b["onsets"], deadpan_mask=b["deadpan_mask"], compute_loss=False)
    tokens = b["masked_perf"].clone()
    tokens[:, 0] = b["perf"][:, 0]
    return tokens, b["masked_perf"], enc.score_embeddings, enc.perf_embeddings, b["perf_mask"], b["perf"]


def _configure(name, monkeypatch):
    """render_batch keywords of one note-step configuration (and the environment / module state it needs)."""
    from scoreperformer_b200 import decode
    if name == "adaln_per_step":            # no prepared AdaLN terms: the front runs as launches before the stack kernel
        monkeypatch.setattr(decode, "ADALN_TERMS_MAX_BYTES", 0)
    if name == "legacy":                    # launch-per-operator stack + host-side sampling
        monkeypatch.setenv("SPB_DECODE", "legacy")
    if name == "host_sampling":             # stack kernel + host-side sampling
        return dict(generator=torch.Generator("cuda"), top_k=1)
    return {}


@pytest.mark.parametrize("name,per_step", [("default", 6), ("adaln_per_step", 9)])
@pytest.mark.parametrize("use_graph", [True, False])
def test_launches_per_note_step(model, monkeypatch, name, per_step, use_graph):
    """The default note-step is six launches, eager or replayed from a graph; with the AdaLN terms evaluated per step it is nine
    (gather, tuple embedding, front GEMM, emb_norm, project_emb GEMM, stack, head projection, its LayerNorm, heads + sampling)."""
    from scoreperformer_b200 import kernels as K
    from scoreperformer_b200.decode import render_batch
    kw = _configure(name, monkeypatch)
    tokens, masked, score, style, mask, _ = _inputs(model, 2, 40, seed=3)
    launches = {}
    for T in (24, 40):
        K.LAUNCHES = 0
        render_batch(model, tokens[:, :T], masked[:, :T], score[:, :T], style[:, :T], mask=mask[:, :T], use_graph=use_graph, **kw)
        torch.cuda.synchronize()
        launches[T] = K.LAUNCHES
    assert (launches[40] - launches[24]) / (40 - 24) == per_step, launches


def test_step_configurations_agree_with_the_default(model, monkeypatch):
    """Teacher-forced on the same inputs, every configuration fills every MASK and makes the default configuration's greedy
    decisions, up to near-ties of bf16 logits (the bar of test_persistent_decode_stack_matches_operator_path)."""
    from scoreperformer_b200.decode import render_batch
    tokens, masked, score, style, mask, teacher = _inputs(model, 16, 96, seed=31)
    valid = mask[:, 1:, None].expand(-1, -1, len(FIELDS))
    outs = {}
    for name in ("default", "adaln_per_step", "host_sampling", "legacy"):
        with monkeypatch.context() as mp:
            kw = _configure(name, mp)
            outs[name] = render_batch(model, tokens, masked, score, style, mask=mask, teacher=teacher, **kw)
        assert int((outs[name] == 1).sum()) == int((tokens[:, 0] == 1).sum()), name        # every MASK after note 0 was filled
        keep = [f for f in range(tokens.shape[-1]) if f not in FIELDS]
        assert torch.equal(outs[name][..., keep], tokens[..., keep]), name
    for name in ("adaln_per_step", "host_sampling", "legacy"):
        same = (outs[name][:, 1:, FIELDS] == outs["default"][:, 1:, FIELDS])[valid]
        agree = float(same.float().mean())
        print(f"{name}: {agree:.4f} of {same.numel()} greedy decisions agree with the default note-step")
        assert agree >= 0.97, (name, agree)


@pytest.mark.parametrize("top_k", [1, 8])
def test_graph_replay_equals_eager_steps(model, monkeypatch, top_k):
    """Stack kernel without the in-kernel front, fused sampling: the sampling kernel advances the position and clears the stack
    kernel's grid barrier, so a replayed rendering must equal one of eager steps token for token (free-running, same seed)."""
    from scoreperformer_b200.decode import render_batch
    _configure("adaln_per_step", monkeypatch)
    tokens, masked, score, style, mask, _ = _inputs(model, 8, 64, seed=11)
    outs = []
    for use_graph in (True, False):
        torch.manual_seed(5)
        outs.append(render_batch(model, tokens, masked, score, style, mask=mask, top_k=top_k, use_graph=use_graph))
    assert int((outs[0] == 1).sum()) == int((tokens[:, 0] == 1).sum())
    assert torch.equal(outs[0], outs[1])
