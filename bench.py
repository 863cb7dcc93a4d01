#!/usr/bin/env python
"""Benchmark of the ScorePerformer training step (BASELINE.json: train note-tuples/s at 1/2/4/8 B200).

    python bench.py --gpus N --steps K --warmup W            # our sm_100a arm
    python bench.py --impl reference ...                      # the reference algorithm on the host CPU (oracle port)

A "step" is one full training step of the default recipe (forward, backward, gradient all-reduce when N > 1, clip,
AdamW) on one synthetic SPMuple batch of `configs[1]`: B=64 sequences x T=512 notes per GPU, bf16 tensor-core math,
fp32 master weights, recipe dropouts ON.  `value` times K steps with the batch resident in HBM; `e2e` times the same
steps fed from pinned host memory (H2D of the int64 batch every step, D2H of the loss every step).
One JSON line is printed by rank 0.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "train note-tuples/sec"
UNIT = "note-tuples/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c4", "c5"],
                    help="c2 = configs[1] (64 x 512 per GPU, the headline); c4 = configs[3], the long-context variant (16 x 2048 per GPU); "
                         "c5 = configs[4], batched KV-cached rendering of 256 scores x 1024 notes (prints bench_render.py's line)")
    ap.add_argument("--batch", type=int, default=None, help="sequences per GPU (default: 64 for c2, 16 for c4)")
    ap.add_argument("--seq", type=int, default=None, help="notes per sequence (default: 512 for c2, 2048 for c4)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="run the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--profile-kernels", action="store_true", help="print the per-kernel launch table of one step")
    ap.add_argument("--timeline", default=None,
                    help="warm up, then record the kernels of 3 steps with torch.profiler (CUPTI) into this CSV "
                         "(name, stream, start_us, dur_us) and exit -- a diagnostic, never a bench value")
    ap.add_argument("--ncu-step", action="store_true",
                    help="warm up, then run ONE step between cudaProfilerStart/Stop and exit (use with ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the measurements, run one more step of the timed path from the seeded initial weights and "
                         "optimizer state and write what it computed (loss, loss terms, evaluator metrics, updated parameters, a "
                         "fixed sample of the gradients; c5: the tokens of the last timed call) as DIR/<name>.npy, so two builds "
                         "can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs covers the timed path of --impl b200")
    if args.batch is None:
        args.batch = 64 if args.config == "c2" else 16
    if args.seq is None:
        args.seq = 512 if args.config == "c2" else 2048
    return args


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], tflops=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured (MEASURED_PEAKS.json, sustained)")
    return dict(hbm_gbs=6650.0, tflops=1400.0, source="fallback (B200_PROFILING.md)")


# ----------------------------------------------------------------------------- clocks sampling
class ClockSampler:
    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.thread = [], None, None
        self.gpu_index = gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- algorithmic work (SURVEY.md section 8(d))
def algorithmic_flops_per_tuple(T: int) -> float:
    """fwd+bwd FLOPs per note-tuple of a training step: 3 * (24.28 MF + 8192 * T)."""
    return 3.0 * (24.28e6 + 8192.0 * T)


# ----------------------------------------------------------------------------- reference arm / CPU baseline
# The UNMODIFIED reference is a copy of the original project found by tests/parity.reference_root() ($SPB200_REFERENCE_ROOT, else
# baseline/_ref), driven through oracle/ref_shim.py, which only supplies stand-ins for the absent omegaconf / miditok imports.
# Without one the oracle port is timed instead, kind "port".
def _reference_root():
    from tests.parity import reference_root
    return reference_root()


def build_reference(device: str = "cpu"):
    """(model, kind): the reference ScorePerformer of the default recipe (seed 23, recipe dropouts ON, train mode)."""
    root = _reference_root()
    if root is None:
        return None, "port"
    os.environ["SPB200_REFERENCE_ROOT"] = root
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import warnings
    warnings.filterwarnings("ignore")
    import ref_shim
    model, _ = ref_shim.build_reference_model(seed=23)
    model.train()
    return model.to(device), "reference"


def time_reference_cpu(batch: int, seq: int, steps: int, warmup: int):
    """fwd+bwd of the reference on the host cores (fp32, all threads, dropouts on as the recipe has them; no optimiser, as
    BASELINE.md section 5 specifies).  Returns dict(value, best_ms, mean_ms, cores, kind)."""
    from scoreperformer_b200.synthetic import make_batch
    torch.set_num_threads(os.cpu_count() or 1)
    model, kind = build_reference("cpu")
    data = make_batch(batch, seq, seed=1234)
    if model is None:                      # oracle port (dropouts off: the port has none)
        from tests import parity
        import model_oracle as mo
        pm = parity.build_model(dropout=False, device="cpu")
        sd, spec = parity.oracle_state(pm), parity.oracle_spec(pm)
        z = [torch.randn(256, d) for d in (32, 20, 8, 4)]

        def one():
            for v in sd.values():
                v.grad = None
            mo.scoreperformer_forward(sd, data, spec, z)["loss"].backward()
    else:
        def one():
            model.zero_grad(set_to_none=True)
            model(**data).loss.backward()
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        one()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    best, mean = min(times) * 1e3, 1e3 * sum(times) / len(times)
    return dict(value=batch * seq / (best / 1e3), best_ms=best, mean_ms=mean, cores=torch.get_num_threads(), kind=kind)


def time_reference_gpu(batch: int, seq: int, steps: int = 3, warmup: int = 2):
    """Informational (SURVEY 2.2): the same reference modules in eager mode under bf16 autocast on this B200 -- what a user gets
    today by moving the unmodified reference to the GPU.  fwd+bwd only, CUDA-event timed."""
    from scoreperformer_b200.synthetic import make_batch
    try:
        model, kind = build_reference("cuda")
        if model is None:
            return {"unavailable": "baseline/_ref missing"}
        data = {k: v.cuda() for k, v in make_batch(batch, seq, seed=1234).items()}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for i in range(warmup + steps):
            if i == warmup:
                torch.cuda.synchronize()
                ev[0].record()
            model.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                out = model(**data)
            out.loss.backward()
        ev[1].record()
        torch.cuda.synchronize()
        ms = ev[0].elapsed_time(ev[1]) / steps
        res = {"value": batch * seq / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "kind": kind,
               "what": f"unmodified reference modules, eager PyTorch, bf16 autocast, fwd+bwd of B={batch} x T={seq} on this GPU "
                       f"(no optimiser step), mean of {steps} steps"}
        del model, data, out
        torch.cuda.empty_cache()
        return res
    except Exception as e:        # informational leg: never take the bench line down
        torch.cuda.empty_cache()
        return {"unavailable": f"{type(e).__name__}: {e}"[:300]}


def workload_config(B, T, world, graph=True):
    which = "configs[1]" if (B, T) == (64, 512) else ("configs[3], long context" if (B, T) == (16, 2048) else "custom shape")
    return {"workload": "ScorePerformer default recipe (recipes/scoreperformer/base.yaml) training step: fwd+bwd+clip+AdamW + the "
                        "recipe's evaluator metrics (trainer.py:462-464), "
                        f"bf16 tensor-core math / fp32 master weights, recipe dropouts on ({which})",
            "global_batch": B * world, "per_gpu_batch": B, "seq_len": T, "parallelism": f"dp{world}", "cuda_graph": graph,
            "l2": "per-step activations (>3 GB) far exceed the 126 MB L2; no explicit flush needed"}


DUMP_GRAD_SAMPLES = 1 << 20
DUMP_MAX_BYTES = 64_000_000


def step_outputs(model, ts, loss):
    """Host copies of what a caller has after a training step: the loss, its terms and the evaluator's metrics, every parameter
    as updated by the step, and the gradients at 2^20 fixed positions (drawn with seed 0 from the parameters' gradients
    concatenated in registration order, so the sample does not depend on how the step lays out its buffers)."""
    def host(t):
        t = torch.as_tensor(t).detach().cpu()
        return (t.double() if t.dtype == torch.float64 else t.float()).numpy()
    out = {"loss": host(loss)}
    out.update({f"losses.{k}": host(v) for k, v in ts.losses.items()})
    out.update({f"metrics.{k}": host(v) for k, v in (ts.metrics or {}).items()})
    params = [(k, p) for k, p in model.named_parameters() if p.grad is not None]
    out.update({f"param.{k}": host(p) for k, p in params})
    grads = torch.cat([p.grad.detach().reshape(-1) for _, p in params])
    idx = torch.randint(grads.numel(), (DUMP_GRAD_SAMPLES,), generator=torch.Generator().manual_seed(0)).sort().values
    out["grad_sample"] = host(grads[idx.to(grads.device)])
    return out


def step_from(model, ts, initial, batch):
    """One step of the timed path (captured afresh for the restored state, then replayed) from `initial` = (model state_dict,
    optimizer state) on `batch`, and its outputs (step_outputs)."""
    sd, opt = initial
    model.load_state_dict(sd)
    ts.load_optimizer_state_dict(opt)                    # also drops the captured graphs
    ts.mark_weights_changed()
    return step_outputs(model, ts, ts.step(batch))


def write_outputs(directory, outputs):
    """One DIR/<name>.npy per array ('/' in loss and metric names becomes '.')."""
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_MAX_BYTES}-byte budget")
    os.makedirs(directory, exist_ok=True)
    import numpy as np
    for name, a in outputs.items():
        np.save(os.path.join(directory, name.replace("/", ".") + ".npy"), a)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    b, t = 4, args.seq                     # bounded sample of the arm's workload: 4 of its 64 sequences per step, same T
    r = time_reference_cpu(b, t, max(1, args.steps), max(1, min(args.warmup, 2)))
    cfg = workload_config(args.batch, t, max(1, args.gpus))
    cfg["reference_sample"] = f"each step = fwd+bwd of {b} of the {args.batch} sequences (T={t}) on the host CPU; value from the best step"
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["best_ms"], "ms_per_step_mean": r["mean_ms"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                         "sample": f"fwd+bwd of B={b} x T={t} per step, fp32, recipe dropouts on, best of {args.steps} steps "
                                   f"({r['kind']}: " + ("unmodified reference from baseline/_ref" if r["kind"] == "reference"
                                                        else "oracle port, dropouts off") + ")"},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- our arm
def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.config == "c5":
        import bench_render
        bench_render.main([] if args.dump_outputs is None else ["--dump-outputs", args.dump_outputs])
        return

    import torch.distributed as dist
    from scoreperformer_b200 import kernels as K
    from scoreperformer_b200.models import ScorePerformer
    from scoreperformer_b200.train_step import TrainStep
    from scoreperformer_b200.recipes import default_model_config
    from scoreperformer_b200.synthetic import make_batch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl b200 needs a CUDA device: scoreperformer_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    torch.manual_seed(23)
    model = ScorePerformer.init(default_model_config(dropout=True)).to(dev)
    model.train()
    model.perf_encoder.exact_latent_shapes = False          # static segment tables: no host sync inside the step
    model.perf_decoder.label_fields = (3, 5, 10, 11)        # MixedLM collator labels (base.yaml:64-65): no probe sync
    ts = TrainStep(model, lr=2e-4, weight_decay=1e-6, grad_clip=2.0, use_graph=not args.no_graph)
    # the seeded starting point of the step --dump-outputs replays: the weights every later step starts from carry the rounding of
    # the earlier steps' atomic reductions (their order varies from run to run), so only this state is the same in every run
    initial = (copy.deepcopy(model.state_dict()), ts.optimizer_state_dict()) if args.dump_outputs else None
    # the reference trainer evaluates its metrics after every training step (experiments/trainer.py:462-464, recipe settings
    # base.yaml:195-198): the timed step does too -- the head kernel accumulates the statistics, the evaluator divides
    from scoreperformer_b200.models.scoreperformer.evaluator import ScorePerformerEvaluator
    from scoreperformer_b200.synthetic import SyntheticTokenizer
    ts.set_evaluator(ScorePerformerEvaluator(
        model, tokenizer=SyntheticTokenizer(), weighted_distance=True,
        ignore_keys=["Bar", "Position", "Pitch", "Duration", "TimeSig", "PositionShift", "NotesInOnset", "PositionInOnset"]))

    B, T = args.batch, args.seq
    host_batch = {k: v.pin_memory() for k, v in make_batch(B, T, seed=1234 + rank).items()}
    dev_batch = {k: v.to(dev) for k, v in host_batch.items()}
    # what crosses the host-device link per step: the collated batch in its natural width (uint16 tokens, int32 segment ids,
    # uint8 directions, lengths); masked tokens, labels and masks are rebuilt on the device (data/packed.py, csrc/collate.cu)
    from scoreperformer_b200.data.packed import pack_batch, packed_bytes
    packed_host = pack_batch(host_batch, check=True)
    h2d_bytes = packed_bytes(packed_host)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n_steps, feed):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_steps):
            feed()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms

    for _ in range(max(4, args.warmup)):                     # >= 3 eager steps, then capture + first replay
        ts.step(dev_batch)

    if args.ncu_step:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        ts.step(dev_batch)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return

    if args.timeline:
        from torch.profiler import profile, ProfilerActivity
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                ts.step(dev_batch)
            torch.cuda.synchronize()
        with open(args.timeline, "w") as f:
            f.write("name,stream,start_us,dur_us\n")
            for ev in prof.events():
                if ev.device_type == torch.autograd.DeviceType.CUDA:
                    name = ev.name.replace(",", ";")[:100]
                    f.write(f"{name},{getattr(ev, 'device_index', 0)}:{getattr(ev, 'stream', getattr(ev, 'device_resource_id', 0))},"
                            f"{ev.time_range.start:.3f},{ev.time_range.end - ev.time_range.start:.3f}\n")
        return

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total = timed(args.steps, lambda: ts.step(dev_batch))
    launches = ts.launches_per_step * args.steps
    clocks = sampler.stop() if rank == 0 else None

    # end to end: every step's int64 batch comes from pinned host memory and every step's loss is read back to the host.  The
    # copy of step i+1 is issued (side stream) before the host waits for step i's loss, the way a prefetching input pipeline
    # feeds a trainer, so the H2D transfer overlaps compute instead of serialising with it.
    def e2e_step():
        loss = ts.step_prefetched()                          # waits for this step's H2D copy, expands it on the device, runs the step
        ts.prefetch_packed(packed_host)                      # next step's pinned host -> device copy, overlapped
        return float(loss)                                   # D2H read of the step's result (sync)

    ts.prefetch_packed(packed_host)
    e2e_step()
    ms_e2e = timed(args.steps, e2e_step)

    ms_step = ms_total / args.steps
    tuples = B * T * world
    value = tuples / (ms_step / 1e3)
    e2e_value = tuples / (ms_e2e / args.steps / 1e3)

    # ---- roofline of the dominant kernel family (the tcgen05 GEMM): time every GEMM launch of one step with CUDA events
    peaks = load_peaks()
    roofline = None
    if True:                                  # every rank runs the instrumented step (it contains the gradient all-reduce)
        records = []
        orig = K.gemm

        def timed_gemm(a, b, **kw):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            out = orig(a, b, **kw)
            e.record()
            m, k_ = (a.shape[1], a.shape[0]) if kw.get("trans_a") else a.shape
            n = b.shape[1] if kw.get("trans_b") else b.shape[0]
            records.append((s, e, 2.0 * m * n * k_, (m, n, k_)))
            return out
        K.gemm = timed_gemm
        import scoreperformer_b200.fused as fused_mod
        fused_mod.K.gemm = timed_gemm
        # the other tensor-core kernels of the step, timed the same way: fused feed-forward forward, attention forward / backward
        other = {"ffn_fwd": [], "ffn_bwd": [], "attention_fwd": [], "attention_bwd": []}
        orig_other = {name: getattr(K, name) for name in other}

        def wrap(name):
            fn = orig_other[name]

            def timed_fn(*a, **kw):
                s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s_.record()
                out_ = fn(*a, **kw)
                e_.record()
                other[name].append((s_, e_))
                return out_
            return timed_fn
        for name in other:
            setattr(K, name, wrap(name))
        ts.use_graph = False
        # the timed step overlaps independent branches on side streams; for the per-kernel roofline every GEMM must own the GPU
        # while it is timed, so the instrumented eager steps run single-stream
        branch_env = {k: os.environ.get(k) for k in ("SPB_SIDE_STREAM", "SPB_ENC_BRANCH", "SPB_WGRAD_BRANCH")}
        for k in branch_env:
            os.environ[k] = "0"
        for _ in range(3):                    # first eager passes only warm the allocator (the graph owns a private pool)
            records.clear()
            for v_ in other.values():
                v_.clear()
            torch.cuda._sleep(int(60e6))      # ~30 ms spin kernel: lets the CPU run ahead so event pairs see GPU time only
            ts.step(dev_batch)
            torch.cuda.synchronize()
        K.gemm = orig
        fused_mod.K.gemm = orig
        for name, fn in orig_other.items():
            setattr(K, name, fn)
        for k, v in branch_env.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        tot_ms = sum(s.elapsed_time(e) for s, e, _, _ in records)
        tot_fl = sum(f for _, _, f, _ in records)
        # dominant launch shape = the one with the largest share of GEMM time (FFN1 forward at C2)
        by_shape = {}
        for s_, e_, f_, shp in records:
            a = by_shape.setdefault(shp, [0, 0.0, f_])
            a[0] += 1
            a[1] += s_.elapsed_time(e_)
        top_shape, (top_n, top_ms, top_fl) = max(by_shape.items(), key=lambda kv: kv[1][1])
        achieved = top_fl / (top_ms / top_n / 1e3) / 1e12
        # DRAM bytes of the dominant launch shape from the committed `ncu --set full` capture (profiles/r02_gemm_traffic.json); null
        # if the dominant shape of this run is not the captured one
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            if tuple(tj.get("shape_MNK", ())) == tuple(top_shape):
                traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
        roofline = {"bound": "tensor",
                    "kernel": f"gemm_bf16_kernel (tcgen05/TMEM/TMA), dominant launch M,N,K={top_shape} x{top_n} per step",
                    "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops"],
                    "traffic": traffic, "algorithmic_flops_per_launch": top_fl, "avg_launch_us": top_ms / top_n * 1e3,
                    "all_gemm_launches_per_step": len(records), "all_gemm_ms_per_step": tot_ms,
                    "all_gemm_achieved_tflops": tot_fl / (tot_ms / 1e3) / 1e12, "gemm_share_of_step": tot_ms / ms_step,
                    "peak_source": peaks["source"],
                    "step_algorithmic_tflops": algorithmic_flops_per_tuple(T) * B * T / (ms_step / 1e3) / 1e12,
                    "step_frac_of_peak": algorithmic_flops_per_tuple(T) * B * T / (ms_step / 1e3) / 1e12 / peaks["tflops"]}
        # algorithmic FLOPs per launch: fused feed-forward 2*n*D*(2H + H); attention 4*B*heads*T^2*64 forward (x2.5 backward),
        # halved under the causal mask (the decoder's 4 of the 10 layers) -- the launches are timed together, so an average
        n_rows, Dm, Hh = B * T, 256, 1024
        attn_full = 4.0 * B * 4 * T * T * 64
        attn_avg = attn_full * (6 + 4 * 0.5) / 10
        alg = {"ffn_fwd": 2.0 * n_rows * Dm * 3 * Hh, "ffn_bwd": 2.0 * n_rows * Dm * 3 * Hh, "attention_fwd": attn_avg,
               "attention_bwd": 2.5 * attn_avg}
        names = {"ffn_fwd": "ffn_fwd_pair_kernel (GEMM1 -> GLU -> GEMM2 -> +residual, u / h on chip)",
                 "ffn_bwd": "ffn_bwd_pair_kernel (dh = dy W2 on chip -> GLU' -> du in place -> dxn = du W1, bias gradient)",
                 "attention_fwd": "attn_fwd_tc_kernel (S, P, O in TMEM)", "attention_bwd": "attn_bwd_tc_kernel (+ dQ convert)"}
        # algorithmic HBM bytes per launch of the fused feed-forward kernels (DESIGN.md section 3) and the DRAM bytes ncu measured
        # for one launch (profiles/r02_ncu_full_ffn_fused.txt, r02_ncu_full_ffn_bwd.txt)
        hbm = {"ffn_fwd": {"algorithmic_bytes": n_rows * (512 + 1024 + 1024 + 4096 + 2048.0), "traffic": 53547264 + 182329344},
               "ffn_bwd": {"algorithmic_bytes": n_rows * (512 + 4096 + 4096 + 512.0), "traffic": 153690368 + 95829760}}
        extra = []
        for name, evs in other.items():
            if not evs:
                continue
            ms_ = sum(s_.elapsed_time(e_) for s_, e_ in evs)
            tf = alg[name] * len(evs) / (ms_ / 1e3) / 1e12
            ent = {"kernel": names[name], "launches_per_step": len(evs), "avg_launch_us": ms_ / len(evs) * 1e3,
                   "algorithmic_flops_per_launch": alg[name], "achieved": tf, "unit": "TFLOP/s", "frac": tf / peaks["tflops"],
                   "share_of_step": ms_ / ms_step}
            if name in hbm and (B * T == 32768):
                gbs = hbm[name]["algorithmic_bytes"] * len(evs) / (ms_ / 1e3) / 1e9
                ent.update({"hbm_algorithmic_bytes_per_launch": hbm[name]["algorithmic_bytes"], "hbm_achieved_gbs": gbs,
                            "hbm_frac": gbs / peaks["hbm_gbs"], "traffic": hbm[name]["traffic"]})
            extra.append(ent)
        roofline["other_tensor_kernels"] = extra
        if args.profile_kernels:
            agg = {}
            for s, e, f, shp in records:
                a = agg.setdefault(shp, [0, 0.0, 0.0])
                a[0] += 1
                a[1] += s.elapsed_time(e)
                a[2] += f
            for shp, (c, ms_, f) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
                print(f"# gemm M,N,K={shp}: {c} launches, {ms_:.3f} ms, {f / ms_ / 1e9:.1f} TFLOP/s", file=sys.stderr)

    cpu_baseline = reference_gpu = None
    if rank == 0 and not args.no_cpu_baseline:
        r = time_reference_cpu(4, 256, steps=5, warmup=2)
        cpu_baseline = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                        "sample": "configs[0]: fwd+bwd of B=4 x T=256 (1024 note-tuples) per step, fp32, recipe dropouts on, "
                                  "2 warm-up + best of 5 steps (BASELINE.md section 5)", "ms_per_step": r["best_ms"],
                        "ms_per_step_mean": r["mean_ms"]}
        reference_gpu = time_reference_gpu(B, T)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": workload_config(B, T, world, not args.no_graph),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches,
            "gpu_launches_per_step": launches / args.steps,
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "reference_gpu": reference_gpu,
        }
        print(json.dumps(line), flush=True)
    if initial is not None:
        ts.use_graph = not args.no_graph                 # the roofline pass above switched to eager steps
        outputs = step_from(model, ts, initial, dev_batch)
        if rank == 0:
            write_outputs(args.dump_outputs, outputs)
    if world > 1:
        ts.close()                       # the captured graphs hold NCCL kernels: release them before the communicator goes
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
