"""End-to-end parity of the sm_100a training step against the CPU oracle and the reference-generated goldens."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import parity

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def model():
    return parity.build_model(dropout=False, device="cuda")


@pytest.mark.parametrize("name", ["train_b2_t48.npz", "train_b3_t33.npz"])
def test_step_matches_reference_golden(model, name):
    """Losses / hidden states / selected gradients against vectors produced by the UNMODIFIED reference."""
    g = parity.golden(name)
    batch = parity.make_batch(int(g["B"]), int(g["T"]), seed=int(g["seed"]))
    out = parity.run_product_step(model, batch, parity.z_from_golden(g))
    for key, want in zip(g["loss_keys"], g["loss_vals"]):
        got = float(out.losses[str(key)])
        assert abs(got - want) <= 2e-2 * max(abs(want), 1e-2), f"{key}: {got} vs reference {want}"
    assert abs(float(out.loss) - float(g["loss"])) <= 2e-2 * abs(float(g["loss"]))
    for name_, t in (("score_hidden", out.score_encoder.hidden_state), ("perf_hidden", out.perf_encoder.hidden_state),
                     ("embeddings", out.perf_encoder.embeddings), ("dec_hidden", out.perf_decoder.hidden_state)):
        want = torch.from_numpy(g[name_])
        err = float((t.detach().float().cpu() - want).abs().max() / want.abs().max())
        assert err < parity.ACT_RTOL, f"{name_}: {err}"
    sd = dict(model.state_dict(keep_vars=True))
    for k in g.files:
        if k.startswith("grad/"):
            cd = parity.cosine_distance(sd[k[5:]].grad.float().cpu(), torch.from_numpy(g[k]))
            assert cd <= 5e-3, f"{k}: cosine distance {cd}"
    for key in ("Velocity", "Tempo", "RelOnsetDev", "RelPerfDuration", "Bar", "NotesInOnset"):
        want = torch.from_numpy(g[f"logits/{key}"])
        err, rms = parity.logits_deviation(out.perf_decoder.logits[key].float().cpu(), want)
        assert err < parity.LOGIT_MAX_RTOL and rms < parity.LOGIT_RMS_RTOL, f"logits/{key}: worst element {err}, rms {rms}"


@pytest.mark.parametrize("B,T,seed", [(2, 48, 1), (4, 256, 1234), (3, 130, 7)])
def test_step_matches_oracle(model, B, T, seed):
    """Full gradient check (every parameter) against the oracle on the same seeded batch; C1 is (4, 256)."""
    torch.manual_seed(seed)
    batch = parity.make_batch(B, T, seed=seed)
    z = [torch.randn(256, d) for d in (32, 20, 8, 4)]
    parity.compare_step(model, batch, z)


@pytest.mark.parametrize("B,T", [(64, 512), (16, 2048)])
def test_full_size_step_matches_oracle(model, B, T):
    """C2 (64 x 512) and C4 (16 x 2048) at full size: the oracle runs in strict fp32 on the same B200 (seconds instead of the
    minutes the host CPU would need).  At these sizes the beat / onset levels have more than 4096 valid latents, so the MMD
    subsample branch (mmd_transformer.py:515-517) is on the path: the oracle draws the permutation and the CUDA path gets
    the same rows."""
    torch.manual_seed(B + T)
    batch = parity.make_batch(B, T, seed=1234)
    z = [torch.randn(256, d) for d in (32, 20, 8, 4)]
    rep = parity.compare_step(model, batch, z, oracle_device="cuda")
    assert rep["mmd_subsampled_levels"], "expected at least one latent level above the 4096-row MMD cap at this size"
    torch.cuda.empty_cache()


def test_dropout_training_step_runs():
    """Recipe dropouts on: finite loss and gradients, different seeds give different losses."""
    m = parity.build_model(dropout=True, device="cuda")
    batch = {k: v.cuda() for k, v in parity.make_batch(4, 128, seed=3).items()}
    m.train()
    torch.manual_seed(1)
    l1 = m(**batch).loss
    l1.backward()
    torch.manual_seed(2)
    l2 = m(**batch).loss
    assert torch.isfinite(l1) and torch.isfinite(l2) and float(l1) != float(l2)
    for n, p in m.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), n


def test_train_step_graph_matches_eager_and_redraws_dropout():
    """CUDA-graph replay == eager math (dropouts off), and with dropouts on every replay draws fresh masks (device RNG offset)."""
    from scoreperformer_b200.train_step import TrainStep
    batch = {k: v.cuda() for k, v in parity.make_batch(2, 64, seed=5).items()}
    losses = {}
    for use_graph in (False, True):
        torch.manual_seed(0)
        m = parity.build_model(dropout=False, device="cuda")
        m.train()
        m.perf_encoder.exact_latent_shapes = False
        ts = TrainStep(m, lr=1e-4, use_graph=use_graph)
        torch.manual_seed(1)
        seq = []
        for _ in range(7):                       # 3 eager warm-ups, capture, replays
            seq.append(float(ts.step(batch)))
        losses[use_graph] = seq
    # the MMD prior sample comes from torch's CUDA generator in both modes: compare the deterministic LM part of the loss
    assert losses[True][6] < losses[True][0], f"loss should go down over 7 steps on one batch: {losses}"
    for a, b in zip(losses[False][:3], losses[True][:3]):
        assert abs(a - b) < 5e-3 * abs(a), (losses[False], losses[True])      # fp32 atomics make runs differ in the last bits
    assert abs(losses[False][6] - losses[True][6]) < 0.1 * abs(losses[False][6]), (losses[False], losses[True])

    m = parity.build_model(dropout=True, device="cuda")
    m.train()
    ts = TrainStep(m, lr=0.0, use_graph=True)     # lr 0: only the dropout masks / prior samples change between replays
    vals = [float(ts.losses["Velocity"]) for _ in range(6) if ts.step(batch) is not None]
    assert len(set(round(v, 6) for v in vals[3:])) == 3, f"graph replays must redraw dropout masks, got {vals}"


def test_prefetched_host_batches_feed_the_same_steps():
    """`prefetch()` + `step_prefetched()` (pinned host batch copied on a side stream, overlapping the running step) trains on
    exactly the batches it was given: with dropouts off and lr 0 the per-batch losses equal those of plain `step()`."""
    from scoreperformer_b200.train_step import TrainStep
    torch.manual_seed(0)
    m = parity.build_model(dropout=False, device="cuda")
    m.train()
    m.perf_encoder.exact_latent_shapes = False
    ts = TrainStep(m, lr=0.0, use_graph=True)
    host = [{k: v.pin_memory() for k, v in parity.make_batch(2, 64, seed=s).items()} for s in (5, 6, 7)]
    dev = [{k: v.cuda() for k, v in b.items()} for b in host]
    want = []
    for i in range(9):                                   # warm-ups, capture, replays; round-robin over three batches
        want.append(float(ts.losses["Velocity"]) if ts.step(dev[i % 3]) is not None else None)
    got = []
    ts.prefetch(host[0])
    for i in range(9):
        loss = ts.step_prefetched()
        ts.prefetch(host[(i + 1) % 3])                   # next batch's copy overlaps this step
        assert loss is not None
        got.append(float(ts.losses["Velocity"]))
    for i in range(9):
        assert abs(got[i] - want[i % 3 + 6]) < 1e-4 * abs(got[i]), (i, got, want)


RECIPE_IGNORE = ["Bar", "Position", "Pitch", "Duration", "TimeSig", "PositionShift", "NotesInOnset", "PositionInOnset"]


@pytest.mark.parametrize("name", ["train_b2_t48.npz", "train_b3_t33.npz"])
@pytest.mark.parametrize("tag,kw", [("recipe", dict(weighted_distance=True, ignore_keys=RECIPE_IGNORE)), ("plain", dict(weighted_distance=False))])
def test_evaluator_matches_reference(model, name, tag, kw):
    """ScorePerformerEvaluator fed by the head kernel's statistics (hits / |value - target| sums accumulated while the logits are in
    tensor memory) against the metrics the UNMODIFIED reference evaluator produced on the same batch (evaluator.py:48-106), and
    against its own logits-based statement.  Accuracies are ratios of small counts: one near-tie may flip."""
    from scoreperformer_b200.models.scoreperformer.evaluator import ScorePerformerEvaluator
    from scoreperformer_b200.synthetic import SyntheticTokenizer
    g = parity.golden(name)
    batch = parity.make_batch(int(g["B"]), int(g["T"]), seed=int(g["seed"]))
    ev = ScorePerformerEvaluator(model, tokenizer=SyntheticTokenizer(), **kw)
    try:
        out = parity.run_product_step(model, batch, parity.z_from_golden(g))
        assert out.perf_decoder.eval_stats is not None, "the LM wrapper did not hand back the head kernel's statistics"
        labels = {"labels": batch["labels"].cuda()}
        fused = ev(labels, out)
        out.perf_decoder.eval_stats = None                      # same outputs through the materialised logits
        plain = ev(labels, out)
    finally:
        model.perf_decoder.eval_token_values = None
    want = dict(zip([str(k) for k in g[f"eval/{tag}/keys"]], g[f"eval/{tag}/vals"]))
    assert list(fused.keys()) == list(want.keys()) == list(plain.keys())
    rows = float((batch["labels"][:, 1:] != -100).sum()) / 4          # labelled rows per field
    for k, w in want.items():
        tol = 2.5 / rows + 1e-3 if k.startswith("accuracy") else 3e-2 * abs(w) + 1e-3
        assert abs(float(fused[k]) - w) <= tol, f"{k}: head kernel {float(fused[k])} vs reference {w}"
        assert abs(float(plain[k]) - w) <= tol, f"{k}: logits path {float(plain[k])} vs reference {w}"
        assert abs(float(plain[k]) - float(fused[k])) <= tol, k


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one host")
def test_train_step_nccl_world2():
    """Data-parallel TrainStep over NCCL: parameters stay identical across ranks, equal the single-process result on the same data,
    and the bucketed all-reduce captured inside the step graph equals one all-reduce after backward (tests/ddp_nccl_worker.py)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29517", os.path.join(root, "tests", "ddp_nccl_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert res.returncode == 0 and res.stdout.count("DDP-NCCL-OK") == 2, res.stdout[-3000:] + res.stderr[-3000:]


def test_static_segment_tables_report_overflow():
    """ADVICE r1: in sync-free mode ids beyond the static table are skipped by the pooling kernel -- that must be visible.  A batch
    whose beat ids run past T + 4 raises the device counter; the default synthetic batch does not."""
    from scoreperformer_b200.train_step import TrainStep
    m = parity.build_model(dropout=False, device="cuda").train()
    ts = TrainStep(m, lr=0.0, use_graph=False)
    m.perf_encoder.exact_latent_shapes = False
    batch = {k: v.cuda() for k, v in parity.make_batch(2, 48, seed=2).items()}
    ts.step(batch)
    assert ts.segment_overflow_count() == 0
    sparse = dict(batch)
    sparse["beats"] = batch["beats"] * 8                 # far fewer than one note per beat: ids run ahead of the note count
    ts.step(sparse)
    want = int(((sparse["beats"] >= 48 + 4) & batch["perf_mask"]).sum())
    assert want > 0 and ts.segment_overflow_count() == want
    m.perf_encoder.slot_capacity = int(sparse["beats"].max()) + 1
    m.perf_encoder.segment_overflow.zero_()
    ts.step(sparse)
    assert ts.segment_overflow_count() == 0


@pytest.mark.gpu
def test_frozen_label_fields_count_unexpected_labels():
    """ADVICE r1: the label fields are probed on the first batch and frozen (the reference re-checks them every batch,
    wrappers.py:49-59).  Labels that later appear in an excluded field must be visible: a device counter, read through TrainStep."""
    from scoreperformer_b200.train_step import TrainStep
    m = parity.build_model(dropout=False, device="cuda").train()
    ts = TrainStep(m, lr=0.0, use_graph=False)
    batch = {k: v.cuda() for k, v in parity.make_batch(2, 48, seed=2).items()}
    ts.step(batch)
    fields = m.perf_decoder.label_fields
    assert ts.unexpected_label_count() == 0 and 0 < len(fields) < batch["labels"].shape[-1]
    excluded = [i for i in range(batch["labels"].shape[-1]) if i not in fields][0]
    odd = dict(batch)
    odd["labels"] = batch["labels"].clone()
    odd["labels"][:, 1:9, excluded] = 5              # the wrapper shifts the labels by one position: 8 labelled rows per sequence
    ts.step(odd)
    assert ts.unexpected_label_count() == 2 * 8


@pytest.mark.gpu
def test_trainer_checkpoint_resume(tmp_path):
    """f4: the epoch loop around TrainStep -- DataLoader, ExponentialLR per epoch through the device-side learning rate, a
    checkpoint in the reference's layout (experiments/trainer.py:296-347) and a resumed run that continues like the uninterrupted one."""
    from scoreperformer_b200.synthetic import SyntheticDataset, collate_rows
    from scoreperformer_b200.trainer import DataParallelTrainer, steps_per_epoch

    def build(seed=0):
        torch.manual_seed(seed)
        m = parity.build_model(dropout=False, device="cuda").train()
        m.perf_decoder.label_fields = (3, 5, 10, 11)
        return m

    data = SyntheticDataset(24, 48, seed=7)
    assert steps_per_epoch(24, 4) == 6
    full = DataParallelTrainer(build(), data, collate_rows, batch_size=4, lr=1e-3, lr_gamma=0.5, output_dir=str(tmp_path), seed=5)
    torch.manual_seed(21)
    logs = full.fit(epochs=2)
    assert [e["step"] for e in logs] == list(range(1, 13)) and abs(full.step.lr - 5e-4) < 1e-12
    assert logs[-1]["loss"] < logs[0]["loss"]

    half = DataParallelTrainer(build(), data, collate_rows, batch_size=4, lr=1e-3, lr_gamma=0.5, output_dir=str(tmp_path), seed=5)
    torch.manual_seed(21)
    half.fit(epochs=1)
    path = half.save_checkpoint()
    ckpt = torch.load(path, weights_only=False)
    assert set(ckpt) == {"experiment", "model", "optimizer"} and set(ckpt["model"]) == {"config", "state_dict"}
    assert set(ckpt["optimizer"]) == {"state", "param_groups"} and "exp_avg_sq" in ckpt["optimizer"]["state"][0]

    resumed = DataParallelTrainer(build(seed=123), data, collate_rows, batch_size=4, lr=1e-3, lr_gamma=0.5, output_dir=str(tmp_path), seed=5)
    resumed.load_checkpoint(path)
    assert resumed.epoch == 1 and resumed.global_step == 6
    logs2 = resumed.fit(epochs=2)
    assert [e["step"] for e in logs2] == list(range(7, 13))
    # same data order (the loader's generator is reseeded per epoch); the MMD prior samples differ (their RNG state is not part of
    # the reference's checkpoint either), so the comparison is loose
    for a, b in zip(logs2, logs[6:]):
        assert abs(a["loss"] - b["loss"]) < 0.05 * abs(b["loss"]), (a, b)


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_trainer_nccl_world2(tmp_path):
    """f4 on two GPUs: DistributedSampler shards, identical parameters on both ranks, rank-0 checkpoint, resume (tests/trainer_nccl_worker.py)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29519", os.path.join(root, "tests", "trainer_nccl_worker.py")]
    env = dict(os.environ, SPB_TEST_OUT=str(tmp_path))
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root, env=env)
    assert res.returncode == 0 and res.stdout.count("TRAINER-NCCL-OK") == 2, res.stdout[-3000:] + res.stderr[-3000:]


@pytest.mark.gpu
def test_untied_lm_head_trains():
    """recipes/scoreperformer/ablation/no_io_tie.yaml: the untied `lm` head (embeddings.py:287-313, one nn.Linear per field) with the
    masked per-field cross-entropy of wrappers.py:45-59.  Loss and gradients against fp32 torch on the same hidden states, then one
    optimisation step of a model built with that head."""
    from scoreperformer_b200 import fused
    torch.manual_seed(3)
    n, D = 777, 256
    sizes = (260, 85, 16)
    hidden = torch.randn(n, D, device="cuda", requires_grad=True)
    Ws = [torch.nn.Parameter(torch.randn(v, D, device="cuda") * D ** -0.5) for v in sizes]
    bs = [torch.nn.Parameter(torch.randn(v, device="cuda") * 0.1) for v in sizes]
    labels = torch.stack([torch.randint(0, v, (n,), device="cuda") for v in (sizes[0], 7, sizes[1], sizes[2])], dim=-1)
    labels[::3] = -100
    labels[:, 1] = -100                                   # column 1 carries no labels and is not listed
    fields = (0, 2, 3)
    params = [p for w, b in zip(Ws, bs) for p in (w, b)]
    loss, per_field, count = fused.UntiedHeadCEFn.apply(hidden, labels, -100, fields, *params)
    loss.backward()
    got = [hidden.grad.clone()] + [p.grad.clone() for p in params]
    hidden.grad = None
    for p in params:
        p.grad = None
    ref_losses = [F.cross_entropy(hidden @ w.t() + b, labels[:, f], ignore_index=-100) for w, b, f in zip(Ws, bs, fields)]
    ref = sum(ref_losses) / len(ref_losses)
    ref.backward()
    want = [hidden.grad] + [p.grad for p in params]
    assert abs(float(loss) - float(ref)) < 5e-3 * abs(float(ref))
    assert all(abs(float(a) - float(b)) < 5e-3 * abs(float(b)) for a, b in zip(per_field, ref_losses))
    assert [int(c) for c in count] == [int((labels[:, f] != -100).sum()) for f in fields]
    for a, b in zip(got, want):
        assert rel_cos(a, b) < 5e-3, rel_cos(a, b)

    # the whole model with that head: one step runs and moves the head
    import copy
    from scoreperformer_b200.models import ScorePerformer
    from scoreperformer_b200.recipes import default_model_config
    from scoreperformer_b200.train_step import TrainStep
    cfg = copy.deepcopy(default_model_config(dropout=False))
    cfg["perf_decoder"]["lm_head"] = {"_target_": "lm"}
    model = ScorePerformer.init(cfg)
    parity.fill_model_(model, 0)
    model = model.cuda().train()
    heads = model.perf_decoder.model.lm_head.heads
    before = {k: h.weight.detach().clone() for k, h in heads.items()}
    ts = TrainStep(model, lr=3e-4, use_graph=False)
    batch = {k: v.cuda() for k, v in parity.make_batch(2, 48, seed=2).items()}
    losses = [float(ts.step(batch)) for _ in range(10)]
    assert all(l == l for l in losses) and losses[-1] < losses[0], losses
    moved = [k for k, h in heads.items() if not torch.equal(h.weight.detach(), before[k])]
    assert len(moved) == len(model.perf_decoder.label_fields) > 0


def rel_cos(a, b):
    a, b = a.float().flatten(), b.float().flatten()
    return float(1 - torch.dot(a, b) / (a.norm() * b.norm()).clamp(min=1e-20))

