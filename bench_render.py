#!/usr/bin/env python
"""configs[4]: batched KV-cached rendering, 256 scores x 1024 notes on one GPU (notes/s), beside the reference algorithm's
batch-1 cached loop on the host CPU (oracle port).  Secondary benchmark; bench.py carries the headline metric."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import torch  # noqa: E402


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--scores", type=int, default=256)
    ap.add_argument("--notes", type=int, default=1024)
    ap.add_argument("--cpu-notes", type=int, default=48)
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the tokens the last timed call rendered as DIR/tokens.npy (float32: the ids are exact)")
    args = ap.parse_args(argv)
    from tests import parity
    from scoreperformer_b200 import kernels as K
    from scoreperformer_b200.decode import render_batch
    model = parity.build_model(dropout=False, device="cuda").eval()
    B, T = args.scores, args.notes
    batch = {k: v.cuda() for k, v in parity.make_batch(B, T, seed=5, full_length=True, deadpan_last=False).items()}
    with torch.inference_mode():
        t0 = time.perf_counter()
        enc = model.forward_encoders(perf=batch["perf"], perf_mask=batch["perf_mask"], score=batch["score"], score_mask=batch["score_mask"],
                                     bars=batch["bars"], beats=batch["beats"], onsets=batch["onsets"], deadpan_mask=batch["deadpan_mask"],
                                     compute_loss=False)
        torch.cuda.synchronize()
        t_enc = time.perf_counter() - t0
        tokens = batch["masked_perf"].clone()
        tokens[:, 0] = batch["perf"][:, 0]
        render_batch(model, tokens[:, :8], batch["masked_perf"][:, :8], enc.score_embeddings[:, :8], enc.perf_embeddings[:, :8])   # warm-up
        torch.cuda.synchronize()
        # every call prepares its per-position terms, captures one note-step in a CUDA graph and replays it; the FIRST full-size call
        # also pays for the allocator's cudaMallocs (KV caches, prepared terms, the graph's private pool) -- reported separately as
        # `cold_seconds`, the value is the best of three warm calls (a rendering service renders score after score)
        times = []
        for rep in range(4):
            K.LAUNCHES = 0
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = render_batch(model, tokens, batch["masked_perf"], enc.score_embeddings, enc.perf_embeddings, mask=batch["perf_mask"])
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        dt_cold, dt = times[0], min(times[1:])
    if args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "tokens.npy"), out.cpu().numpy().astype(np.float32))
    notes = B * (T - 1)
    # CPU reference: batch-1 cached greedy loop of the oracle port on a short score
    import model_oracle as mo
    cpu_model = parity.build_model(dropout=False, device="cpu")
    sd = parity.oracle_state(cpu_model, requires_grad=False)
    spec = parity.oracle_spec(cpu_model)
    n = args.cpu_notes
    cb = parity.make_batch(1, n, seed=5, full_length=True, deadpan_last=False)
    with torch.no_grad():
        sh = mo.encoder_forward(sd, "score_encoder", cb["score"], cb["score_mask"], list(spec.num_score_tokens), spec.depth_score, spec)
        pe = mo.perf_encoder_forward(sd, cb, spec, None, training=False, compute_loss=False)["embeddings"]
        tk = cb["masked_perf"].clone()
        tk[:, 0] = cb["perf"][:, 0]
        t0 = time.perf_counter()
        mo.render_greedy(sd, spec, tk, cb["masked_perf"], sh, pe, use_cache=True)
        dt_cpu = time.perf_counter() - t0
    kv_bytes = sum(1024 * t for t in range(1, T)) * B          # SURVEY 8(d): 4 layers x (k|v) x 64 x bf16 = 1024 B per cached position
    print(json.dumps({
        "metric": "rendered notes/sec (greedy, KV-cached, batched)", "value": notes / dt, "unit": "notes/s", "n_gpus": 1,
        "config": {"workload": f"configs[4]: {B} scores x {T} notes, fields (3,5,10,11) rendered note by note", "scores": B, "notes": T},
        "seconds": dt, "cold_seconds": dt_cold, "warm_seconds_all": times[1:], "encoder_seconds": t_enc, "gpu_launches": K.LAUNCHES, "filled_mask_tokens": int((out != tokens).sum()),
        "roofline": {"bound": "hbm", "achieved": kv_bytes / dt / 1e9, "peak": 6450.6, "unit": "GB/s", "frac": kv_bytes / dt / 1e9 / 6450.6,
                     "note": "algorithmic KV-cache reads only (SURVEY 8(d)); a note-step is 6 launches captured in a CUDA graph: one gather at the device-side position, the tuple embedding of the previous note, ONE persistent kernel for the rest of the input front and the 4-layer decoder stack (grid-barrier phases, tensor-core attention over the KV cache, csrc/decode_stack.cu; everything that does not depend on sampled tokens -- masked-tuple and context terms, AdaLN terms -- is prepared for all positions before the loop), head projection + LayerNorm (2), ONE head + sampling kernel whose last CTA advances the position"},
        "cpu_baseline": {"value": (n - 1) / dt_cpu, "unit": "notes/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"oracle port of unmask_tokens, batch 1, cached, {n} notes"}}))


if __name__ == "__main__":
    main()
