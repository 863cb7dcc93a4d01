"""CPU: host-side logic -- drop-in API surface, config plumbing, C-ABI symbol table, gradient buckets over gloo."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

from tests import parity
from scoreperformer_b200 import lib as spb_lib
from scoreperformer_b200.config import load_recipe, wrap
from scoreperformer_b200.models import EVALUATORS, MODELS
from scoreperformer_b200.recipes import default_model_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = parity.reference_root()
NO_REF = "needs a copy of the original ScorePerformer project for its recipes ($SPB200_REFERENCE_ROOT or baseline/_ref)"


def test_registries_and_state_dict_layout():
    assert set(MODELS) == {"Performer", "ScorePerformer"} and set(EVALUATORS) == {"ScorePerformerEvaluator"}
    model = parity.build_model()
    sd = model.state_dict()
    assert len(sd) == 463
    assert sum(p.numel() for p in model.parameters()) == 11_603_049
    # tied tables: one storage under every alias (SURVEY Appendix A.3)
    a = sd["perf_decoder.model.token_emb.embs.Velocity.index_weight"]
    for alias in ("score_encoder", "perf_encoder", "perf_decoder.model.lm_head"):
        key = f"{alias}.token_emb.embs.Velocity.index_weight" if "lm_head" not in alias else f"{alias}.embs.Velocity.index_weight"
        assert sd[key].data_ptr() == a.data_ptr(), key
    assert sd["perf_decoder.model.lm_head.project_emb.weight"].data_ptr() == sd["perf_decoder.model.token_emb.project_emb.weight"].data_ptr()
    g = parity.golden("train_b2_t48.npz")
    for k in g["grad_norm_keys"]:
        assert str(k) in sd, k
    assert sd["perf_encoder.vae_head.onset_mean.linear.weight"].shape == (4, 316)
    assert sd["perf_decoder.model.transformer.final_norm.linear.weight"].shape == (512, 64)


def test_outputs_and_forward_signature_match_reference_names():
    import dataclasses
    import inspect
    from scoreperformer_b200.models.scoreperformer.model import ScorePerformer, ScorePerformerOutputs, ScorePerformerEncoderOutputs
    from scoreperformer_b200.models.scoreperformer.mmd_transformer import MMDTupleTransformerOutput
    assert [f.name for f in dataclasses.fields(ScorePerformerOutputs)] == \
        ["perf_decoder", "score_encoder", "perf_encoder", "classifiers", "loss", "losses"]
    assert [f.name for f in dataclasses.fields(ScorePerformerEncoderOutputs)] == \
        ["score_embeddings", "score_mask", "perf_embeddings", "score_encoder", "perf_encoder"]
    assert [f.name for f in dataclasses.fields(MMDTupleTransformerOutput)][-6:] == \
        ["latents", "embeddings", "full_embeddings", "dropout_mask", "loss", "losses"]
    assert list(inspect.signature(ScorePerformer.forward).parameters)[1:] == \
        ["perf", "perf_mask", "score", "score_mask", "noisy_perf", "noisy_perf_mask", "masked_perf", "labels", "bars", "beats",
         "onsets", "directions", "deadpan_mask"]


def test_cpu_forward_fails_loudly():
    model = parity.build_model()
    batch = parity.make_batch(1, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback|CUDA"):
        model(**batch)


@pytest.mark.skipif(REF is None, reason=NO_REF)
def test_unmodified_recipes_load_and_match_builtin_default():
    cfg = load_recipe("scoreperformer/base.yaml", os.path.join(REF, "recipes"))["model"]
    builtin = default_model_config()
    for stack in ("score_encoder", "perf_encoder", "perf_decoder"):
        got = {k: v for k, v in cfg[stack].items()}
        want = {k: v for k, v in builtin[stack].items()}
        want["token_embeddings"] = {k: v for k, v in want["token_embeddings"].items() if k != "token_values"}
        assert got == want, stack
    assert cfg["classifiers"]["classifier"] == builtin["classifiers"]["classifier"]
    assert cfg["dim"] == 256 and cfg["mode"] == "mixlm" and cfg["tie_token_emb"] is True
    for name in ("no_classifiers.yaml", "custom_hierarchy.yaml", "minimal.yaml", "ablation/no_saln.yaml", "ablation/no_score_enc.yaml",
                 "ablation/no_masked_seq.yaml", "ablation/no_cont_tokens.yaml", "ablation/no_io_tie.yaml"):
        assert "model" in load_recipe("scoreperformer/" + name, os.path.join(REF, "recipes")), name


@pytest.mark.skipif(REF is None, reason=NO_REF)
@pytest.mark.parametrize("name", ["no_classifiers.yaml", "custom_hierarchy.yaml", "ablation/no_saln.yaml", "ablation/no_score_enc.yaml",
                                  "ablation/no_masked_seq.yaml", "ablation/no_cont_tokens.yaml", "ablation/no_io_tie.yaml"])
def test_variant_recipes_construct(name):
    """Every shipped recipe must construct (API surface); only the default family has a CUDA forward in round 1."""
    import copy
    cfg = load_recipe("scoreperformer/" + name, os.path.join(REF, "recipes"))["model"]
    base = default_model_config()
    cfg["num_tokens"], cfg["num_score_tokens"] = base["num_tokens"], base["num_score_tokens"]
    for stack in ("score_encoder", "perf_encoder", "perf_decoder"):
        if cfg.get(stack) is not None:
            keys = base["num_score_tokens"] if stack == "score_encoder" else base["num_tokens"]
            cfg[stack]["token_embeddings"]["token_values"] = {k: base["perf_decoder"]["token_embeddings"]["token_values"][k] for k in keys}
    if cfg.get("classifiers") is not None:
        cfg["classifiers"]["num_classes"] = base["classifiers"]["num_classes"]
        cfg["classifiers"]["class_samples"] = base["classifiers"]["class_samples"]
    model = MODELS["ScorePerformer"].init(wrap(copy.deepcopy(cfg)))
    assert sum(p.numel() for p in model.parameters()) > 1_000_000


def test_constructor_error_behaviour():
    from scoreperformer_b200.modules.transformer import FeedForward
    ff = FeedForward.init({"mult": 2, "glu": True, "bogus_key": 1, "_private": 2}, dim=64)      # unknown keys dropped with a warning
    assert ff.inner_dim == 128
    with pytest.raises(RuntimeError, match="mandatory"):
        FeedForward.init({"dim": "???"})


def test_c_abi_exports_every_declared_symbol():
    """The shared library must export exactly what include/spb200.h declares (no compute calls here)."""
    path = spb_lib.build()
    handle = ctypes.CDLL(path)
    header = open(os.path.join(ROOT, "include", "spb200.h")).read()
    declared = set(re.findall(r"^(?:int|const char\*)\s+(spb_\w+)\(", header, flags=re.M))
    assert len(declared) >= 18
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in spb200.h but not exported"
    assert declared - {"spb_last_error", "spb_abi_version"} == set(spb_lib.SIGNATURES), "lib.py binding table out of sync with the header"
    assert spb_lib.lib().spb_abi_version() == 1
    # error path works without a GPU: bad arguments are rejected before any launch
    rc = spb_lib.lib().spb_gemm_bf16(None, None, None, 0, 0, 0, 0, 0, 8, 8, 8, None, None, 0, None, 0, 1, 0, None, None)
    assert rc == -1 and b"null operand" in spb_lib.lib().spb_last_error()


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "scoreperformer_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "model_oracle" not in src and "import oracle" not in src and "ref_shim" not in src, os.path.join(dirpath, f)


def test_gradient_buckets_gloo_world2():
    """N>1 path on CPU: two gloo ranks with different gradients end up with the mean in every p.grad."""
    script = os.path.join(ROOT, "tests", "ddp_gloo_worker.py")
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                          "--master-port", "29613", script], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert res.stdout.count("DDP-OK") == 2, res.stdout[-2000:]


def test_constructor_initialises_bit_identically_to_the_reference():
    """DESIGN.md section 1: parameters are registered in the reference's order, so under the same seed the constructor draws the
    same numbers.  tests/golden/init_seed23.npz holds key order, shapes and checksums of the UNMODIFIED reference's state_dict
    under torch.manual_seed(23) (oracle/gen_golden.py:gen_init); both directions of a strict load follow from equal key sets.
    The checksums are float64 sums whose last bits depend on the order torch reduced in on the generating host (its SIMD width):
    they are compared with the correctly rounded sum within 4 eps * sum|x| (every golden lies within 0.82 eps * sum|x| of it), a few
    ulps of the sum and far below one float32 ulp of a weight."""
    import copy
    import math
    import numpy as np
    from tests import parity
    from scoreperformer_b200.models import ScorePerformer
    from scoreperformer_b200.recipes import default_model_config
    g = parity.golden("init_seed23.npz")
    torch.manual_seed(int(g["seed"]))
    model = ScorePerformer.init(copy.deepcopy(default_model_config(dropout=True)))
    sd = model.state_dict()
    keys = list(sd.keys())
    assert keys == [str(k) for k in g["keys"]], "state_dict keys / order differ from the reference"
    eps = float(np.finfo(np.float64).eps)
    for k, shape, s_ref, a_ref, f_ref in zip(keys, g["shapes"], g["sums"], g["abs_sums"], g["first"]):
        t = sd[k]
        assert "x".join(map(str, t.shape)) == str(shape), k
        values = t.double().reshape(-1).tolist()
        abs_sum = math.fsum(map(abs, values))
        tol = 4 * eps * abs_sum
        assert abs(math.fsum(values) - float(s_ref)) <= tol and abs(abs_sum - float(a_ref)) <= tol, f"{k}: initial values differ"
        if t.numel():
            assert float(t.reshape(-1)[0]) == float(f_ref), k
    # a state_dict with exactly these keys and shapes loads strictly (and the reference, having the same, accepts ours)
    clone = ScorePerformer.init(copy.deepcopy(default_model_config(dropout=True)))
    missing, unexpected = clone.load_state_dict(sd, strict=True)
    assert not missing and not unexpected


def test_mixlm_masking_statement_matches_reference_collator():
    """data/packed.mixlm_mask_sequence == MixedLMPerformanceCollator.mask_sequence of the unmodified reference (golden vectors for
    three settings, oracle/gen_golden.py:gen_collator); pack_batch keeps exactly the information the collator output carries."""
    from tests import parity
    from scoreperformer_b200.data import PackedBatchSpec, mixlm_mask_sequence, pack_batch
    from scoreperformer_b200.data.packed import packed_bytes
    from scoreperformer_b200.synthetic import make_batch
    g = parity.golden("collator_mixlm.npz")
    seq = torch.from_numpy(g["seq"])
    specs = {"recipe": PackedBatchSpec(),
             "all_dims": PackedBatchSpec(mask_ignore_token_ids=(0, 3), mask_ignore_token_dims=(), label_pad_ignored_dims=False),
             "keep_labels": PackedBatchSpec(mask_ignore_token_dims=(0, 5), label_pad_ignored_dims=False)}
    for tag, spec in specs.items():
        masked, labels = mixlm_mask_sequence(seq, spec)
        assert torch.equal(masked, torch.from_numpy(g[f"{tag}/masked"])) and torch.equal(labels, torch.from_numpy(g[f"{tag}/labels"])), tag
    batch = make_batch(4, 64, seed=3)
    packed = pack_batch(batch, check=True, pin=False)
    assert packed_bytes(packed) < 0.15 * sum(v.numel() * v.element_size() for v in batch.values())
    bad = dict(batch)
    bad["perf_mask"] = batch["perf_mask"].clone()
    bad["perf_mask"][0, 3] = False                       # a hole: not a prefix mask
    with pytest.raises(ValueError):
        pack_batch(bad, pin=False)


def test_trainer_sampler_shards_an_epoch():
    """f4 host logic: with N ranks every rank draws a disjoint shard of the epoch's permutation (experiments/trainer.py:166-174 gets
    a DistributedSampler), reshuffled by set_epoch, and the step count per epoch follows drop_last on both levels."""
    from scoreperformer_b200.synthetic import SyntheticDataset, collate_rows
    from scoreperformer_b200.trainer import make_sampler, steps_per_epoch
    data = SyntheticDataset(37, 16, seed=1)
    assert make_sampler(data, 1, 0, True, 0) is None
    shards = []
    for rank in range(4):
        s = make_sampler(data, 4, rank, True, 5)
        s.set_epoch(0)
        e0 = list(iter(s))
        s.set_epoch(1)
        assert list(iter(s)) != e0 and len(e0) == 37 // 4
        shards.append(e0)
    flat = [i for sh in shards for i in sh]
    assert len(set(flat)) == len(flat) == 36
    assert steps_per_epoch(37, 4, 4) == 2 and steps_per_epoch(24, 4) == 6
    batch = collate_rows([data[i] for i in shards[0][:3]])
    assert batch["perf"].shape[0] == 3 and set(batch) == set(data[0])



def test_streaming_unmask_dispatch(monkeypatch):
    """decode.unmask_mixlm decides on the host which path a request takes; the decisions (and the caches handed in and out) are checked
    here with the device paths replaced by recorders: a fresh window and a window continuing caller-held caches go to the
    device-resident note-step with the right start / keys|values, everything it cannot express goes to the general stepper."""
    import types
    import torch
    from scoreperformer_b200 import decode
    from scoreperformer_b200.modules.sampling import top_k, top_p
    from scoreperformer_b200.models.scoreperformer.transformer import TupleTransformerCaches
    from scoreperformer_b200.modules.transformer.attend import AttentionIntermediates
    from scoreperformer_b200.modules.transformer.transformer import TransformerIntermediates

    sizes = [260, 132, 92, 132, 133, 125, 26, 69, 16, 16, 165, 85]
    dec = types.SimpleNamespace(training=False, dim=256, token_emb=types.SimpleNamespace(field_sizes=sizes),
                                transformer=types.SimpleNamespace(depth=4), eval=lambda: None, train=lambda mode=True: None)
    wrapper = types.SimpleNamespace(model=dec, mask_token_id=1, pad_token_id=0)
    calls = []

    def fake_render(d, out, masked, context, style, **kw):
        calls.append(("device", kw))
        res = out.clone()
        res[res == 1] = 7
        if kw.get("return_kv"):
            T = out.shape[1]
            return res, [torch.arange(T, dtype=torch.float32)[None, :, None].expand(out.shape[0], T, 128).to(torch.bfloat16).clone()
                         for _ in range(4)]
        return res

    def fake_stepper(w, out, masked, mask, notes, hit, *rest):
        calls.append(("stepper", rest[-2]))
        res = out.clone()
        res[res == 1] = 9
        return res, "stepper-caches"

    monkeypatch.setattr(decode, "render_decoder", fake_render)
    monkeypatch.setattr(decode, "_unmask_stepwise", fake_stepper)

    def window(n, k):
        t = torch.randint(4, 16, (1, n, 12))
        t[:, n - k:, [3, 5, 10, 11]] = 1
        m = t.clone()
        m[:, :, [3, 5, 10, 11]] = 1
        return t, m, torch.zeros(1, n, 256), torch.zeros(1, n, 64)

    def run(n, k, caches=None, return_caches=True, fn=top_k, kw={"k": 1}, **extra):
        t, m, ctx, sty = window(n, k)
        calls.clear()
        return decode.unmask_mixlm(wrapper, t, m, 1.0, fn, kw, None, caches, return_caches, context=ctx, style_embeddings=sty, **extra)

    # fresh window, caches requested: device path from position 0, caches in the reference's layout come back
    out, caches = run(4, 3)
    assert calls[0][0] == "device" and calls[0][1]["start"] == 0 and calls[0][1]["kv_init"] == [] and calls[0][1]["use_graph"] is False
    assert int((out == 1).sum()) == 0 and isinstance(caches, TupleTransformerCaches)
    assert caches.token_emb.shape == (1, 3, 256) and len(caches.transformer.hiddens) == 5 and len(caches.transformer.attention) == 4
    assert caches.transformer.attention[0].keys.shape == (1, 3, 64) and caches.transformer.attention[0].values.shape == (1, 3, 64)
    # continuing those caches with two new notes: starts at the cache length, keys | values are handed over as [B, start, 128] bf16
    out, caches2 = run(6, 2, caches=caches)
    kind, kw = calls[0]
    assert kind == "device" and kw["start"] == 3 and len(kw["kv_init"]) == 4
    assert kw["kv_init"][0].shape == (1, 3, 128) and kw["kv_init"][0].dtype == torch.bfloat16
    assert torch.equal(kw["kv_init"][0][0, :, 0].float(), torch.arange(3.)) and caches2.token_emb.shape[1] == 5
    # caches in the stepper's own format (real hiddens) are accepted as well: only keys and values are read
    full = TupleTransformerCaches(token_emb=torch.ones(1, 3, 256), transformer=TransformerIntermediates(
        hiddens=[torch.ones(1, 3, 256)] * 5, attention=[AttentionIntermediates(torch.ones(1, 3, 64), torch.zeros(1, 3, 64)) for _ in range(4)]))
    run(6, 2, caches=full)
    assert calls[0][0] == "device" and calls[0][1]["start"] == 3 and float(calls[0][1]["kv_init"][2][0, 1, 0]) == 1.0
    # what the note-step cannot express goes to the general stepper: cache length != known prefix, unknown filter, no caches behind
    # a known prefix, the legacy switch; the one-shot request without caches keeps the captured-graph path
    run(7, 2, caches=caches)
    assert calls[0][0] == "stepper"
    run(6, 2, caches=caches, fn=top_p, kw={"thres": 0.5})
    assert calls[0][0] == "stepper"
    run(6, 2, caches=None)
    assert calls[0][0] == "stepper"
    monkeypatch.setenv("SPB_STREAM", "legacy")
    run(6, 2, caches=caches)
    assert calls[0][0] == "stepper"
    monkeypatch.delenv("SPB_STREAM")
    out = run(4, 3, return_caches=False)
    assert calls[0][0] == "device" and "start" not in calls[0][1] and int((out == 1).sum()) == 0
