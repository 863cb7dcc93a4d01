import sys, time, torch
sys.path.insert(0, ".")
from tests import parity
from scoreperformer_b200 import decode
model = parity.build_model(dropout=False, device="cuda").eval()
B, T = 256, 1024
batch = {k: v.cuda() for k, v in parity.make_batch(B, T, seed=5, full_length=True, deadpan_last=False).items()}
with torch.inference_mode():
    enc = model.forward_encoders(perf=batch["perf"], perf_mask=batch["perf_mask"], score=batch["score"], score_mask=batch["score_mask"],
                                 bars=batch["bars"], beats=batch["beats"], onsets=batch["onsets"], deadpan_mask=batch["deadpan_mask"], compute_loss=False)
    tokens = batch["masked_perf"].clone(); tokens[:, 0] = batch["perf"][:, 0]
    decode.render_batch(model, tokens[:, :8], batch["masked_perf"][:, :8], enc.score_embeddings[:, :8], enc.perf_embeddings[:, :8])
    torch.cuda.synchronize()
    # instrument: wrap graph replay and capture
    orig_replay = torch.cuda.CUDAGraph.replay
    marks = {}
    def replay(self):
        if "first_replay" not in marks:
            torch.cuda.synchronize(); marks["first_replay"] = time.perf_counter()
        return orig_replay(self)
    torch.cuda.CUDAGraph.replay = replay
    for rep in range(3):
        marks.clear()
        torch.cuda.synchronize(); t0 = time.perf_counter()
        out = decode.render_batch(model, tokens, batch["masked_perf"], enc.score_embeddings, enc.perf_embeddings, mask=batch["perf_mask"])
        torch.cuda.synchronize(); t1 = time.perf_counter()
        print(f"rep {rep}: total {t1 - t0:.3f} s; before first replay {marks['first_replay'] - t0:.3f} s; replays {t1 - marks['first_replay']:.3f} s")
