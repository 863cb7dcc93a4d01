"""Cost of the logit filters of the heads + sampling kernel, timed with CUDA events: the kernel alone at B = 256 scores and four
fields (top-k 5, top-p 0.9, top-a (2, 0.02)), and a 256 x 1024-note `render_batch` greedy and with top-p 0.9.  The card's name and
power limit are read in the same run and printed with the numbers (one JSON line; `--out FILE` also writes it)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import torch  # noqa: E402

SIZES = [260, 132, 92, 132, 133, 125, 26, 69, 16, 16, 165, 85]
FIELDS = [3, 5, 10, 11]


def card():
    res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return res.stdout.strip().splitlines()[0] if res.returncode == 0 and res.stdout.strip() else torch.cuda.get_device_name()


def time_events(fn, iters):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / iters * 1e3          # microseconds per call


def kernel_times(iters):
    from scoreperformer_b200 import kernels as K
    torch.manual_seed(0)
    offs = [0]
    for v in SIZES[:-1]:
        offs.append(offs[-1] + v)
    B, T, F = 256, 8, len(SIZES)
    table = (torch.randn(sum(SIZES), 128, device="cuda") * 0.3).to(torch.bfloat16)
    e = torch.randn(B, F * 128, device="cuda").to(torch.bfloat16)
    tokens = torch.zeros(B, T, F, dtype=torch.int64, device="cuda")
    pos = torch.tensor([2], device="cuda")
    cases = {"top_k_5": dict(topk=5), "top_p_0.9": dict(top_p=[0.9] * 4), "top_a_2_0.02": dict(top_a=[(2.0, 0.02)] * 4),
             "greedy": dict(topk=1)}
    out = {}
    for name, kw in cases.items():
        kw = dict(kw)
        k = kw.pop("topk", 1)
        call = lambda: K.sample_fields(e, table, FIELDS, [offs[f] for f in FIELDS], [SIZES[f] for f in FIELDS], [k] * 4, tokens, pos,
                                       temperature=1.0, seed=1, **kw)
        time_events(call, 50)                               # warm-up
        out[name] = round(min(time_events(call, iters) for _ in range(3)), 3)
    return out


def render_times(B, T, reps):
    from tests import parity
    from scoreperformer_b200.decode import render_batch
    model = parity.build_model(dropout=False, device="cuda").eval()
    batch = {k: v.cuda() for k, v in parity.make_batch(B, T, seed=5, full_length=True, deadpan_last=False).items()}
    with torch.inference_mode():
        enc = model.forward_encoders(perf=batch["perf"], perf_mask=batch["perf_mask"], score=batch["score"], score_mask=batch["score_mask"],
                                     bars=batch["bars"], beats=batch["beats"], onsets=batch["onsets"], deadpan_mask=batch["deadpan_mask"],
                                     compute_loss=False)
        tokens = batch["masked_perf"].clone()
        tokens[:, 0] = batch["perf"][:, 0]
        args = (tokens, batch["masked_perf"], enc.score_embeddings, enc.perf_embeddings)
        out = {}
        modes = {"greedy": dict(top_k=1), "top_p_0.9": dict(top_p=0.9, top_k=None)}
        for kw in modes.values():                           # warm every path (allocations, graph pools)
            render_batch(model, *args, mask=batch["perf_mask"], **kw)
        times = {name: [] for name in modes}
        for _ in range(reps):                               # alternate the two modes
            for name, kw in modes.items():
                start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                start.record()
                render_batch(model, *args, mask=batch["perf_mask"], **kw)
                end.record()
                end.synchronize()
                times[name].append(start.elapsed_time(end) / 1e3)
        for name, ts in times.items():
            out[name] = {"seconds_best": min(ts), "seconds_all": ts, "notes_per_s": B * (T - 1) / min(ts)}
    return out


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=2000)
    ap.add_argument("--scores", type=int, default=256)
    ap.add_argument("--notes", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise RuntimeError("sampling_timing.py needs a CUDA device")
    res = {"card": card(), "kernel_us_per_call_B256_4fields": kernel_times(args.iters),
           "render_batch": {"scores": args.scores, "notes": args.notes, **render_times(args.scores, args.notes, args.reps)}}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
