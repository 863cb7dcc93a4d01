"""KV-cached incremental decoding (SURVEY.md section 8 row a13).

Two entry points over the same kernels:

* `cached_stack_step` -- the cache path of `Transformer.forward` (modules/transformer/transformer.py:161-186,219-221) with
  the reference's cache contract (`TransformerIntermediates`: per attention layer the input hiddens `[B,t,D]` and
  `AttentionIntermediates(keys[B,t,64], values[B,t,64])`), used by `unmask_tokens` / `generate` and therefore by an
  unchanged `inference/generators.py`.
* `render_batch` -- the batched, device-resident form of `ScorePerformerMixedLMWrapper.unmask_tokens`
  (models/scoreperformer/wrappers.py:324-407): all scores advance in lockstep, KV caches are preallocated
  `[depth, B, T, 128]` buffers written in place (no per-step `torch.cat`), no host sync inside the loop.
"""
from __future__ import annotations

import math
import weakref
from typing import Callable, Dict, List, Optional, Sequence, Tuple, Union

import torch
from torch import Tensor

from . import fused, kernels as K

BF16, F32 = torch.bfloat16, torch.float32
# largest bf16 [B, T, (2 depth + 1) 512] table of AdaLN terms render_decoder prepares ahead of its loop; a larger rendering has the
# stack kernel evaluate them step by step
ADALN_TERMS_MAX_BYTES = 8 << 30


class _StackWeights:
    """bf16 copies of one stack's weights, prepared once per decode session."""

    def __init__(self, tr):
        tr._check_fused()
        self.depth, self.H, self.D = tr.depth, tr.heads, tr.dim
        self.ada = tr.ada_norm
        self.layers = []
        norms_w, norms_b = [], []
        for l in range(tr.depth):
            na, attn, _ = tr.layers[2 * l]
            nf, ff, _ = tr.layers[2 * l + 1]
            for n in (na[0], nf[0]):
                w, b = tr._norm_params(n)
                norms_w.append(w.detach())
                norms_b.append(b.detach())
            self.layers.append(dict(
                wqkv=K.cast_bf16(torch.cat([attn.to_q.weight, attn.to_k.weight, attn.to_v.weight], 0).detach().contiguous()),
                wo=K.cast_bf16(attn.to_out.weight.detach().contiguous()),
                ls=attn.logslopes().detach().reshape(-1).float().contiguous(),
                w1=K.cast_bf16(ff.ff[0].proj.weight.detach().contiguous()), b1=ff.ff[0].proj.bias.detach().float().contiguous(),
                w2=K.cast_bf16(ff.ff[3].weight.detach().contiguous())))
        w, b = tr._norm_params(tr.final_norm)
        norms_w.append(w.detach())
        norms_b.append(b.detach())
        if self.ada:
            self.w_ada = K.cast_bf16(torch.cat(norms_w, 0).contiguous())
            self.b_ada = fused.ada_bias_minus_one(norms_b, self.D).contiguous()      # gb = (gamma - 1 | beta), see rowops.cu
        else:
            self.norm_w, self.norm_b = [w.float().contiguous() for w in norms_w], [b.float().contiguous() for b in norms_b]

    def norm(self, i: int, x: Tensor, gb_all: Optional[Tensor], out_dtype=BF16) -> Tensor:
        if self.ada:
            gb = gb_all[:, i * 2 * self.D:(i + 1) * 2 * self.D]
            return K.layer_norm_fwd(x, None, None, gb, out_dtype=out_dtype, need_stats=False)[0]
        return K.layer_norm_fwd(x, self.norm_w[i], self.norm_b[i], out_dtype=out_dtype, need_stats=False)[0]


class _DecoderWeights:
    """What a rendering stages from the performance decoder's parameters before its note loop: the stack's bf16 weights, the
    computed token table (value MLPs) and its bf16 copy, bf16 copies of the front / head projections.  Biases and norm weights are
    views of the parameters."""

    def __init__(self, dec):
        te_mod, head = dec.token_emb, dec.lm_head
        self.sw = _StackWeights(dec.transformer)
        self.table = te_mod.table().detach().contiguous()
        self.table16 = K.cast_bf16(self.table)
        self.ln_w, self.ln_b = te_mod.norm.weight.detach(), te_mod.norm.bias.detach()
        self.wp16 = K.cast_bf16(te_mod.project_emb.weight.detach().contiguous())
        self.bp = te_mod.project_emb.bias.detach()
        self.wm16 = K.cast_bf16(te_mod.project_multiemb.weight.detach().contiguous())
        self.bm = te_mod.project_multiemb.bias.detach()
        self.en_w, self.en_b = dec.emb_norm.weight.detach(), dec.emb_norm.bias.detach()
        self.wc16 = K.cast_bf16(dec.project_emb.weight.detach().contiguous())
        self.bc = dec.project_emb.bias.detach()
        self.whead16 = K.cast_bf16(head.proj_weight_kn().detach().contiguous())
        self.hn_w, self.hn_b = head.norm.weight.detach(), head.norm.bias.detach()
        self.emb = head.split_dims[0]
        self.offs = [0]
        for v in te_mod.field_sizes[:-1]:
            self.offs.append(self.offs[-1] + v)
        Dm = dec.dim
        self.wm_r, self.wc_l, self.wc_r = self.wm16[:, Dm:], self.wc16[:, :Dm], self.wc16[:, Dm:]
        self._te_mod, self._Dm = te_mod, Dm

    def compose_front(self) -> Tuple[Tensor, Tensor]:
        """project_emb of the tuple embedding and the left half of project_multiemb are two linear maps in a row: composed in fp32
        (W = Wm_left Wp, its bias joins the prepared term), so a note-step needs one GEMM for both.  Returns (W bf16 [D, F * 128],
        bias fp32 [D])."""
        te_mod, Dm = self._te_mod, self._Dm
        wm_full = te_mod.project_multiemb.weight.detach().float()
        w_comp16 = K.cast_bf16((wm_full[:, :Dm] @ te_mod.project_emb.weight.detach().float()).contiguous())        # [D, F * 128]
        b_comp = (wm_full[:, :Dm] @ self.bp.float()).contiguous()                                                     # [D]
        return w_comp16, b_comp


def _stack_step(sw: _StackWeights, x_last: Tensor, style_last: Optional[Tensor], kv_caches: Sequence[Tensor], key_mask: Optional[Tensor],
                pos: int, hid_out: Optional[List[Tensor]] = None, pos_dev: Optional[Tensor] = None) -> Tensor:
    """One new position through the stack.  x_last fp32 [B, D]; kv_caches[l] bf16 [B, cap, 128] already holding rows < pos;
    row `pos` is written here (by the attention kernel itself).  With `pos_dev` (device int64 [1]) the position is only known on
    the device -- `pos` is ignored and every launch is CUDA-graph replayable.  Returns the final-norm output fp32 [B, D]."""
    gb_all = None
    if sw.ada:
        gb_all = K.gemm(K.cast_bf16(style_last.float().contiguous()), sw.w_ada, bias=sw.b_ada, out_dtype=BF16)
    if key_mask is None:
        rowmask = None
    elif pos_dev is None:
        rowmask = key_mask[:, pos].contiguous()
    else:
        rowmask = key_mask.index_select(1, pos_dev).reshape(-1).contiguous()
    cur = x_last
    for l, w in enumerate(sw.layers):
        if hid_out is not None:
            hid_out.append(cur)
        xn = sw.norm(2 * l, cur, gb_all)
        qkv = K.gemm(xn, w["wqkv"], out_dtype=BF16)
        cap = kv_caches[l].shape[1]
        o = K.attention_decode(qkv, kv_caches[l], key_mask, w["ls"], sw.H, cap if pos_dev is not None else pos + 1, pos,
                               pos_dev=pos_dev, append_kv=True)
        cur = K.gemm(o, w["wo"], residual=cur, rowmask=rowmask, out_dtype=F32)
        xn = sw.norm(2 * l + 1, cur, gb_all)
        u = K.gemm(xn, w["w1"], bias=w["b1"], out_dtype=BF16)
        h = K.glu_fwd(u, 0.0, 0)
        cur = K.gemm(h, w["w2"], residual=cur, out_dtype=F32)
    return sw.norm(2 * sw.depth, cur, gb_all, out_dtype=F32)


@torch.no_grad()
def cached_stack_step(tr, x: Tensor, mask: Optional[Tensor], style: Optional[Tensor], cache, return_hiddens: bool):
    """Reference cache contract: only the last position of `x` is new; returns the full-length output (and caches)."""
    from .modules.transformer.attend import AttentionIntermediates
    from .modules.transformer.transformer import TransformerIntermediates
    b, t, d = x.shape
    sw = _StackWeights(tr)
    assert len(cache.attention) == tr.depth and len(cache.hiddens) == tr.depth + 1
    kvs = []
    for inter in cache.attention:                         # [B, t-1, 64] each -> working buffer [B, t, 128]
        kv = torch.empty((b, t, 128), dtype=BF16, device=x.device)
        kv[:, :t - 1, :64] = inter.keys
        kv[:, :t - 1, 64:] = inter.values
        kvs.append(kv)
    hid_new: List[Tensor] = []
    km = None if mask is None else mask.contiguous()
    out_last = _stack_step(sw, x[:, -1].float().contiguous(), None if style is None else style[:, -1], kvs, km, t - 1, hid_new)
    out = torch.cat([cache.hiddens[-1].float(), out_last[:, None]], dim=1)
    if not return_hiddens:
        return out
    hiddens = [torch.cat([c.float(), h[:, None]], dim=1) for c, h in zip(cache.hiddens[:-1], hid_new)] + [out]
    att = [AttentionIntermediates(keys=kv[..., :64], values=kv[..., 64:]) for kv in kvs]
    return out, TransformerIntermediates(hiddens=hiddens, attention=att)


@torch.no_grad()
def render_batch(model, perf: Tensor, masked_perf: Tensor, score_hidden: Tensor, style: Tensor, mask: Optional[Tensor] = None,
                 fields: Sequence[int] = (3, 5, 10, 11), temperature: float = 1.0, top_k: Union[int, Sequence[int], None] = 1,
                 generator: Optional[torch.Generator] = None, teacher: Optional[Tensor] = None, use_graph: bool = True,
                 top_p: Optional[float] = None, top_a: Optional[Tuple[float, float]] = None,
                 banned_tokens: Optional[Dict[int, Sequence[int]]] = None) -> Tensor:
    """`render_decoder` on the performance decoder of a ScorePerformer model."""
    return render_decoder(model.perf_decoder.model, perf, masked_perf, score_hidden, style, mask=mask, fields=fields,
                          temperature=temperature, top_k=top_k, generator=generator, teacher=teacher, use_graph=use_graph,
                          top_p=top_p, top_a=top_a, banned_tokens=banned_tokens)


def _check_filters(top_k, top_p, top_a, banned_tokens, fields: Sequence[int], sizes: Sequence[int], n_special: int = 2):
    """Validate the sampling request of `render_decoder`; returns the per-field lists of banned ids (empty lists: none)."""
    if top_p is not None and top_a is not None:
        raise ValueError("top_p and top_a are two logit filters: pass at most one")
    if (top_p is not None or top_a is not None) and top_k not in (None, 1):
        raise ValueError(f"top_k={top_k!r} cannot be combined with top_p / top_a: pass top_k=None (or 1)")
    if top_p is not None and not (math.isfinite(float(top_p)) and float(top_p) >= 0.0):
        raise ValueError(f"top_p must be a finite threshold >= 0, got {top_p!r}")
    if top_a is not None:
        if len(top_a) != 2 or not all(math.isfinite(float(x)) for x in top_a) or float(top_a[1]) <= 0.0:
            raise ValueError(f"top_a must be a finite (min_p_pow, min_p_ratio) pair with min_p_ratio > 0, got {top_a!r}")
    bans = [[] for _ in fields]
    for f, ids in (banned_tokens or {}).items():
        if f not in fields:
            raise ValueError(f"banned_tokens names field {f}, which is not rendered (fields {list(fields)})")
        ids = sorted({int(v) for v in ids})
        bad = [v for v in ids if not 0 <= v < sizes[f]]
        if bad:
            raise ValueError(f"banned_tokens of field {f}: ids {bad} are outside its vocabulary of {sizes[f]}")
        if len(set(ids) | set(range(n_special))) >= sizes[f]:
            raise ValueError(f"banned_tokens of field {f} leave no token to emit")
        bans[list(fields).index(f)] = ids
    return bans


@torch.no_grad()
def render_decoder(dec, perf: Tensor, masked_perf: Tensor, score_hidden: Tensor, style: Tensor, mask: Optional[Tensor] = None,
                   fields: Sequence[int] = (3, 5, 10, 11), temperature: float = 1.0, top_k: Union[int, Sequence[int], None] = 1,
                   generator: Optional[torch.Generator] = None, teacher: Optional[Tensor] = None, use_graph: bool = True,
                   start: int = 0, kv_init: Optional[Sequence[Tensor]] = None, return_kv: bool = False, top_p: Optional[float] = None,
                   top_a: Optional[Tuple[float, float]] = None, banned_tokens: Optional[Dict[int, Sequence[int]]] = None):
    """Fill `fields` of every note >= 1 of `perf` [B, T, F], note by note, for all B scores in lockstep.

    perf / masked_perf: int64 [B, T, F]; score_hidden fp32 [B, T, D]; style fp32 [B, T, S]; mask bool [B, T].
    `top_k=1` is greedy (the parity mode, `filter_kwargs={'k': 1}` in the reference); larger k samples from the top-k
    softmax at `temperature`; `top_k=None` uses the reference default ceil(0.1 * V); a sequence gives one k per field.
    `top_p` (nucleus threshold, modules/sampling.py `top_p`; 0 keeps the arg-max only) or `top_a` ((min_p_pow, min_p_ratio),
    `top_a`) replaces top-k -- then `top_k` must be None or 1.  Both filters see the softmax at temperature 1 of each score's own
    logits (the reference's `top_a` takes its maximum probability over the whole batch it is handed; here it is per score, which
    is the same for one score); the kept tokens are drawn from at `temperature`.  `banned_tokens` maps a field index to token ids
    that field never emits (the reference's `filter_key_ids`), applied with the PAD / MASK ban before the filter.
    `teacher` [B, T, F] (optional) is fed as the already-rendered prefix instead of the model's own samples (teacher forcing,
    used by the parity tests to compare every step independently); the returned tensor still holds the model's predictions.
    `use_graph`: capture one note-step in a CUDA graph and replay it (positions are device-side); sampling with a custom
    `generator` runs eagerly.
    Continuation (the streaming `unmask_tokens` call): with `start = s > 0` the notes 0..s are complete in `perf`, `kv_init[l]` bf16
    [B, s, 128] holds the keys | values of decoder positions < s for every layer, and only the positions s..T-2 run (notes s+1..T-1
    are rendered).  `return_kv` also returns the per-layer caches [B, T, 128] (rows < T-1 valid).
    """
    from .modules import sampling
    sizes = dec.token_emb.field_sizes
    bans = _check_filters(top_k, top_p, top_a, banned_tokens, fields, sizes)
    B, T, F = perf.shape
    dev = perf.device
    st = _DecoderWeights(dec)
    sw, table, table16, ln_w, ln_b, wp16, bp, bm = st.sw, st.table, st.table16, st.ln_w, st.ln_b, st.wp16, st.bp, st.bm
    en_w, en_b, wc16, bc, whead16, hn_w, hn_b = st.en_w, st.en_b, st.wc16, st.bc, st.whead16, st.hn_w, st.hn_b
    emb, offs = st.emb, st.offs
    ctx16 = K.cast_bf16(score_hidden.float().contiguous().view(B * T, -1)).view(B, T, -1)
    km = None if mask is None else mask.contiguous()
    kv_caches = [torch.zeros((B, T, 128), dtype=BF16, device=dev) for _ in range(sw.depth)]
    assert 0 <= start <= T - 1 and (start == 0 or (kv_init is not None and len(kv_init) == sw.depth))
    for kv, init in zip(kv_caches, kv_init or ()):
        assert init.shape == (B, start, 128)
        kv[:, :start] = init
    out = perf.clone()
    feed = (out if teacher is None else teacher).contiguous()

    # The position lives on the device: every index below is a device gather / scatter, so ONE captured step replays for
    # all T-1 notes (`use_graph`), instead of ~50 host launches per note.
    pos_t = torch.full((1,), start, dtype=torch.int64, device=dev)           # i
    field_idx = torch.tensor(list(fields), dtype=torch.int64, device=dev)
    neg_inf = -float("inf")
    style_f = style.float().contiguous()

    # SPB_DECODE=legacy runs the launch-per-operator stack and samples on the host side: the reference of the parity tests
    legacy = K._os.environ.get("SPB_DECODE", "fused") != "fused"
    # the whole decoder stack of a note-step is ONE persistent kernel when the stack has the recipe's shape (csrc/decode_stack.cu)
    plan = None
    if not legacy and K.decode_stack_ok(sw.depth, sw.D, sw.H, sw.layers[0]["w2"].shape[1], sw.ada, style_f.shape[-1], T):
        plan = K.DecodeStackPlan(sw.layers, sw.w_ada, sw.b_ada, kv_caches, B, style_f.shape[-1])

    filtered = top_p is not None or top_a is not None
    if filtered:
        ks = [1] * len(fields)                                                  # ignored by the filtered fields
    elif not isinstance(top_k, (list, tuple)):
        ks = [top_k if top_k is not None else -(-sizes[f] // 10) for f in fields]
    else:
        ks = [int(k) for k in top_k]
        assert len(ks) == len(fields), "top_k: one k per rendered field"
    fused_sampling = (not legacy and generator is None and emb == 128 and len(fields) <= 8 and all(sizes[f] <= 256 for f in fields)
                      and all(1 <= k <= 32 for k in ks))
    seed = K.seed_from_torch() if filtered or any(k > 1 for k in ks) else 0
    # the filters and bans of the sampling launch (all None: the plain top-k call)
    filt_kw = dict(top_p=None if top_p is None else [float(top_p)] * len(fields),
                   top_a=None if top_a is None else [(float(top_a[0]), float(top_a[1]))] * len(fields),
                   banned=bans if any(bans) else None)
    ban_idx = {f: torch.tensor(ids, dtype=torch.int64, device=dev) for f, ids in zip(fields, bans) if ids}
    # with the stack kernel and the sampling kernel both in the step, the sampling kernel's last CTA ends the step: position += 1,
    # grid-barrier word of the stack kernel back to zero
    sampler_ends_step = plan is not None and fused_sampling

    # Everything of a note-step that does not depend on the tokens sampled so far is evaluated for ALL positions before the loop,
    # in large launches: the masked tuple of note i+1 through the embedding and its half of project_multiemb (+ bias), and the
    # context half of project_emb (+ bias).  A step then adds its own half (the previous, complete tuple) as a GEMM with a residual.
    Dm = dec.dim
    wm_r, wc_l, wc_r = st.wm_r, st.wc_l, st.wc_r
    w_comp16, b_comp = st.compose_front()
    P2 = torch.empty((B, T, Dm), dtype=F32, device=dev)
    C2 = torch.empty((B, T, Dm), dtype=F32, device=dev)
    cb = max(1, min(B, 32768 // max(T, 1)))
    for b0 in range(0, B, cb):
        b1 = min(B, b0 + cb)
        x2, _, _ = K.embed_ln_fwd(masked_perf[b0:b1].reshape(-1, F).contiguous(), table, sizes, ln_w, ln_b)
        x2p = K.gemm(x2, wp16, bias=bp, out_dtype=BF16)
        K.gemm(x2p, wm_r, bias=bm + b_comp, out=P2[b0:b1].view(-1, Dm))
        K.gemm(ctx16[b0:b1].reshape(-1, ctx16.shape[-1]), wc_r, bias=bc, out=C2[b0:b1].view(-1, Dm))
        del x2, x2p
    # ... and the AdaLN terms of every position for the stack kernel (one GEMM instead of a tile phase per step), memory permitting
    gb_all = None
    if plan is not None and B * T * plan.gb.shape[1] * 2 <= ADALN_TERMS_MAX_BYTES:
        gb_all = plan.prepare_adaln(style_f)
    # one launch per step reads what the step needs at the device-side position: tuple i, and the prepared terms / style of note i+1
    tok_buf = torch.empty((B, F), dtype=feed.dtype, device=dev)
    p2_buf = torch.empty((B, Dm), dtype=F32, device=dev)
    c2_buf = torch.empty((B, Dm), dtype=F32, device=dev)
    gather_src, gather_dst = [feed, P2, C2], [tok_buf, p2_buf, c2_buf]
    st_buf = None
    if gb_all is None:
        st_buf = torch.empty((B, style_f.shape[-1]), dtype=F32, device=dev)
        gather_src.append(style_f)
        gather_dst.append(st_buf)
    gather_shift = [0] + [1] * (len(gather_src) - 1)
    ln_buf = torch.empty((B, Dm), dtype=BF16, device=dev)
    # the rest of the front (te = x1 W^T + p2, emb_norm, project_emb's left half + c2) runs inside the stack kernel when the
    # tuple embedding has the recipe's width; x1 is then a static buffer the embedding kernel fills
    front_in_kernel = gb_all is not None and len(sizes) * 128 == 1536 and Dm == 256
    if front_in_kernel:
        x1_buf = torch.empty((B, 1536), dtype=BF16, device=dev)
        plan.set_front(x1_buf, w_comp16, p2_buf, en_w.float().contiguous(), en_b.float().contiguous(), wc_l.t().contiguous(), c2_buf)

    def sample_on_host(e):
        # heads of the rendered fields, PAD / MASK and per-field bans, logit filter and draw in torch; out[:, i+1, fields] = toks
        toks = []
        for f, k in zip(fields, ks):
            lg = K.gemm(e[:, f * emb:(f + 1) * emb], table16[offs[f]:offs[f] + sizes[f]], out_dtype=F32)
            lg[:, :2] = neg_inf                                                 # PAD / MASK are never emitted
            if f in ban_idx:
                lg.index_fill_(1, ban_idx[f], neg_inf)
            if filtered:
                lg = sampling.top_p(lg, float(top_p)) if top_p is not None else _top_a_rows(lg, *top_a)
                tok = torch.multinomial(torch.softmax(lg / temperature, dim=-1), 1, generator=generator).squeeze(1)
            elif k == 1:
                tok = lg.argmax(dim=-1)
            else:
                val, ind = torch.topk(lg, k)
                probs = torch.softmax(val / temperature, dim=-1)
                tok = ind.gather(1, torch.multinomial(probs, 1, generator=generator)).squeeze(1)
            toks.append(tok)
        dst = (pos_t + 1) * F + field_idx                                       # [n_fields] flat column indices
        out.view(B, T * F).index_copy_(1, dst, torch.stack(toks, dim=1))

    def step():
        # decoder position i: full tuple of note i, masked tuple / context / style of note i+1 (wrappers.py:409-431)
        K.gather_at_pos(gather_src, gather_dst, gather_shift, pos_t)
        if front_in_kernel:
            K.embed_ln_fwd(tok_buf, table, sizes, ln_w, ln_b, out=x1_buf)
            x = None
        else:
            x1, _, _ = K.embed_ln_fwd(tok_buf, table, sizes, ln_w, ln_b)
            te = K.gemm(x1, w_comp16, residual=p2_buf, out_dtype=F32)
            K.layer_norm_fwd(te, en_w, en_b, out=ln_buf, need_stats=False)
            x = K.gemm(ln_buf, wc_l, residual=c2_buf, out_dtype=F32)
        if plan is not None:
            # the stack kernel leaves a bf16 copy of its output, the head projection's operand
            plan.step(x, st_buf, km, pos_t, gb_all=gb_all, use_front=front_in_kernel, barrier_is_zero=sampler_ends_step)
            hid16 = plan.out16
        else:
            hid16 = K.cast_bf16(_stack_step(sw, x, st_buf, kv_caches, km, 0, pos_dev=pos_t))
        # tied head for the masked fields only (wrappers.py:364-380)
        e_raw = K.gemm(hid16, whead16, trans_b=True, out_dtype=BF16)
        e, _, _ = K.layer_norm_fwd(e_raw, hn_w, hn_b, out_dtype=BF16, need_stats=False)
        if fused_sampling:
            # heads of the rendered fields, PAD / MASK and per-field bans, logit filter, draw and token write: one launch
            K.sample_fields(e, table16, fields, [offs[f] for f in fields], [sizes[f] for f in fields], ks, out, pos_t,
                            temperature=temperature, seed=seed, advance=plan.advance if sampler_ends_step else None, **filt_kw)
        else:
            sample_on_host(e)
        if not sampler_ends_step:
            pos_t.add_(1)

    n_steps = T - 1 - start
    # host-side filters sort and mask with data-dependent shapes: that step runs eagerly
    graph_ok = use_graph and generator is None and n_steps > 4 and (fused_sampling or not filtered)
    if not graph_ok:
        for _ in range(n_steps):
            step()
        return (out, kv_caches) if return_kv else out
    # two eager steps warm every lazily-initialised path, then one step is captured and replayed for the rest
    step()
    step()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    before = K.LAUNCHES
    with torch.cuda.graph(graph):
        step()                                   # recorded, not executed
    per_step = K.LAUNCHES - before
    K.LAUNCHES = before                          # the recording itself launched nothing ...
    for _ in range(n_steps - 2):
        graph.replay()
    K.LAUNCHES += per_step * (n_steps - 2)       # ... each replay launches every recorded kernel
    return (out, kv_caches) if return_kv else out


def _top_a_rows(logits: Tensor, min_p_pow: float, min_p_ratio: float) -> Tensor:
    """modules.sampling.top_a with the limit taken per row (per score) instead of over the whole [B, V] tensor, as the sampling
    kernel does; the most probable token is always kept."""
    probs = torch.softmax(logits, dim=-1)
    top = probs.max(dim=-1, keepdim=True).values
    limit = torch.minimum(top.pow(min_p_pow) * min_p_ratio, top)
    return torch.where(probs < limit, float("-inf"), logits)


# ----------------------------------------------------------------------------- reference-signature entry points
# `unmask_tokens` / `generate` of the LM wrappers (models/scoreperformer/wrappers.py:200-307, 324-407 of the reference) keep their
# argument lists and their cache contract, so inference/generators.py works unchanged -- but they are adapters over this file:
# a window goes through `render_decoder`'s device-resident loop whenever the request is expressible there (any batch size,
# top-k / greedy sampling, no per-key bans) -- from note 1 for a fresh window, or from the end of caller-held caches whose length
# is the known prefix (the streaming calls of inference/generators.py); everything else runs the general stepper below, which
# advances one note per iteration through the cached stack step and samples on the host side of the logits.
def _sampling_plan(filter_logits_fn, filter_kwargs, sizes: Sequence[int], fields: Sequence[int]):
    """k per field if the filter is the reference's `top_k` (sampling.py:28-33), else None (host sampling)."""
    from .modules import sampling
    if filter_logits_fn is not sampling.top_k:
        return None
    kw = dict(filter_kwargs or {})
    if set(kw) - {"k", "thres"}:
        return None
    ks = [int(kw["k"]) if kw.get("k") is not None else math.ceil((1 - kw.get("thres", 0.9)) * sizes[f]) for f in fields]
    return ks if all(1 <= k <= 32 for k in ks) else None


def _draw(logits: Dict[str, Tensor], banned: Sequence[int], filter_key_ids, filter_logits_fn, filter_kwargs, temperature: float) -> Tensor:
    """One token per field from fp32 logits [B, V]: bans, the caller's filter, softmax at the temperature, a draw."""
    from .modules.sampling import filter_logits_and_sample
    cols = []
    for key, lg in logits.items():
        lg = lg.clone()
        lg[:, list(banned)] = -float("inf")
        extra = (filter_key_ids or {}).get(key)
        if extra is not None:
            lg[:, extra] = -float("inf")
        cols.append(filter_logits_and_sample(lg, filter_logits_fn, filter_kwargs=filter_kwargs, temperature=temperature))
    return torch.cat(cols, dim=-1)


def _masked_columns(tokens: Tensor, mask_token_id: int):
    """(note indices that contain a MASK, bool [F] of the masked fields) -- the same fields at every note of the window, as the
    collator produces them; raises otherwise."""
    hit = tokens == mask_token_id
    notes = torch.nonzero(hit.any(dim=2).any(dim=0)).flatten()
    cols = hit.any(dim=1).any(dim=0)
    return notes, cols, hit


@torch.inference_mode()
def unmask_mixlm(wrapper, tokens: Tensor, tokens_masked: Tensor, temperature: float, filter_logits_fn, filter_kwargs, filter_key_ids,
                 caches, return_caches: bool, **kwargs):
    """MixedLM rendering with the reference's signature (wrappers.py:324-407): fill the MASKed fields of `tokens` note by note;
    position i of the decoder sees the full tuple of note i and the masked tuple of note i+1."""
    dec = wrapper.model
    was_training = dec.training
    dec.eval()
    squeeze = tokens.dim() == 2
    if squeeze:
        tokens, tokens_masked = tokens[None], tokens_masked[None]
    out = tokens.clone()
    mask = kwargs.pop("mask", None)
    notes, cols, hit = _masked_columns(out, wrapper.mask_token_id)
    fields = torch.nonzero(cols).flatten().tolist()
    sizes = dec.token_emb.field_sizes
    ks = _sampling_plan(filter_logits_fn, filter_kwargs, sizes, fields)
    context, style = kwargs.get("context"), kwargs.get("style_embeddings")
    T = out.shape[1]
    contiguous_tail = notes.numel() > 0 and int(notes[0]) >= 1 and torch.equal(notes, torch.arange(int(notes[0]), T, device=notes.device))
    uniform = bool(hit[:, notes][..., cols].all()) if notes.numel() else False
    expressible = (ks is not None and not filter_key_ids and contiguous_tail and uniform and context is not None and style is not None
                   and len(set(ks)) == 1 and set(kwargs) <= {"context", "style_embeddings"})
    fast = expressible and caches is None and not return_caches and int(notes[0]) == 1
    start = int(notes[0]) - 1 if notes.numel() else 0
    att = _stream_prefix(dec, caches, start, context, style, T) if expressible and not fast else None
    session = _session_for(dec, out, fields, ks[0], style) if att is not None else None
    kv_init = None if att is None or session is not None else _streamable(dec, caches, start, context, style, T)
    if fast:
        res = render_decoder(dec, out, tokens_masked, context, style, mask=mask, fields=fields, temperature=temperature, top_k=ks[0])
    elif session is not None:
        # the streaming call of inference/generators.py on the decoder's render session: staged weights, stack plan and buffers are
        # kept between calls, the keys / values of a prefix the session handed out are continued in place
        res, caches = session.render(dec, out, tokens_masked, context, style, mask, fields, temperature, ks[0], start, caches)
    elif kv_init is not None:
        # the streaming call of inference/generators.py: a few new notes behind a prefix whose keys / values the caller holds.  Same
        # device-resident note-step as a whole-window rendering (persistent stack kernel, fused heads + sampling), started at the
        # first new note; eager launches, a chord is too short to pay for a graph capture
        res, kvs = render_decoder(dec, out, tokens_masked, context, style, mask=mask, fields=fields, temperature=temperature,
                                  top_k=ks[0], use_graph=False, start=int(notes[0]) - 1, kv_init=kv_init, return_kv=True)
        caches = _kv_only_caches(dec, kvs, T - 1)
    else:
        res, caches = _unmask_stepwise(wrapper, out, tokens_masked, mask, notes, hit, temperature, filter_logits_fn, filter_kwargs,
                                       filter_key_ids, caches, kwargs)
    dec.train(was_training)
    res = res[0] if squeeze else res
    return (res, caches) if return_caches else res


def _stream_prefix(dec, caches, start: int, context: Tensor, style: Tensor, T: int):
    """The per-layer AttentionIntermediates of the prefix ([] when nothing is cached) if the request can continue on the
    device-resident note-step: nothing cached and the first note is the one to render, or caches whose length is exactly the known
    prefix (the check inference/generators.py:222-226 makes as well).  None sends the request to the general stepper.
    SPB_STREAM=legacy switches this path off."""
    if K._os.environ.get("SPB_STREAM", "fused") != "fused" or context.shape[1] != T or style.shape[1] != T or start < 0:
        return None
    if caches is None:
        return [] if start == 0 else None
    att = caches.transformer.attention if caches.transformer is not None else None
    if not att or len(att) != dec.transformer.depth or caches.token_emb.shape[1] != start or start == 0:
        return None
    if any(a.keys is None or a.values is None or a.keys.shape[-2] != start for a in att):
        return None
    return att


def _streamable(dec, caches, start: int, context: Tensor, style: Tensor, T: int):
    """Per-layer [B, start, 128] keys | values of `_stream_prefix`, or None."""
    att = _stream_prefix(dec, caches, start, context, style, T)
    return None if att is None else [torch.cat([a.keys, a.values], dim=-1).to(BF16).contiguous() for a in att]


def _kv_only_caches(dec, kvs: Sequence[Tensor], length: int, zeros: Optional[Tensor] = None):
    """Caches in the reference's layout (TupleTransformerCaches / TransformerIntermediates / AttentionIntermediates, every tensor
    [B, length, .]) after a device-resident rendering.  Keys and values are views of the working buffers.  `token_emb` and `hiddens`
    are ZERO placeholders of the right shapes (views of `zeros` [B, >= length, dim] when given): the cached step of this
    implementation needs the keys and values of the prefix and the last position only (the reference recomputes emb_norm /
    project_emb over the whole prefix from `token_emb` at every step, transformer.py:171-185, and carries the per-layer hiddens
    without reading them)."""
    from .models.scoreperformer.transformer import TupleTransformerCaches
    from .modules.transformer.attend import AttentionIntermediates
    from .modules.transformer.transformer import TransformerIntermediates
    B = kvs[0].shape[0]
    z = torch.zeros((B, length, dec.dim), dtype=F32, device=kvs[0].device) if zeros is None else zeros[:, :length]
    att = [AttentionIntermediates(keys=kv[:, :length, :64], values=kv[:, :length, 64:]) for kv in kvs]
    return TupleTransformerCaches(token_emb=z, transformer=TransformerIntermediates(hiddens=[z] * (len(kvs) + 1), attention=att))


# ----------------------------------------------------------------------------- render sessions (streaming calls)
# A real-time rendering calls `unmask_tokens` once per chord: 1 to 10 note-steps of ~0.2 ms each.  Staging the weights, building the
# stack plan and preparing the per-position terms of the whole window on every call would cost more than the notes, so the decoder
# keeps a session between calls: staged weights, the stack plan with its input front, KV buffer sets of `cap` rows and the prepared
# term buffers, all with row stride `cap`.  A call prepares the terms of its new rows only and continues a prefix the session handed
# out in place.  The session is keyed by the decoder module (weakly) and (B, style width); a window longer than `cap` replaces it.
_SESSIONS: "weakref.WeakKeyDictionary" = weakref.WeakKeyDictionary()
SESSION_MIN_CAP = 256          # smallest window capacity a session is built with (capacities are powers of two up to 2048)
SESSION_POOL = 4               # KV buffer sets a session keeps for renderings that alternate on one decoder


def _session_for(dec, tokens: Tensor, fields: Sequence[int], k: int, style: Tensor) -> Optional["_RenderSession"]:
    """The decoder's render session for a streaming call of this shape, or None when the note-step of the session cannot express
    the call (the call then runs `render_decoder` as a one-off): the persistent stack kernel with its input front and the fused
    sampling kernel must both apply."""
    B, T, F = tokens.shape
    S = style.shape[-1]
    if not tokens.is_cuda or K._os.environ.get("SPB_DECODE", "fused") != "fused":
        return None
    tr, sizes = dec.transformer, dec.token_emb.field_sizes
    hidden = tr.layers[1][1].ff[3].weight.shape[1]
    if not K.decode_stack_ok(tr.depth, tr.dim, tr.heads, hidden, tr.ada_norm, S, T):
        return None
    cap = max(SESSION_MIN_CAP, 1 << (T - 1).bit_length())
    if (B * cap * (2 * tr.depth + 1) * 512 * 2 > ADALN_TERMS_MAX_BYTES or len(sizes) * 128 != 1536 or dec.dim != 256
            or dec.lm_head.split_dims[0] != 128 or len(fields) > 8 or any(sizes[f] > 256 for f in fields) or not 1 <= k <= 32):
        return None
    per_shape = _SESSIONS.setdefault(dec, {})
    session = per_shape.get((B, S))
    if session is None or session.cap < T:
        session = per_shape[(B, S)] = _RenderSession(dec, B, S, min(cap, 2048), tokens.device)
    return session


class _KVSet:
    """One set of per-layer KV buffers [B, cap, 128] of a render session, with weak references to the caches handed out from it."""

    def __init__(self, depth: int, B: int, cap: int, dev):
        self.kv = [torch.zeros((B, cap, 128), dtype=BF16, device=dev) for _ in range(depth)]
        self._bases = {kv.untyped_storage().data_ptr() for kv in self.kv}
        self.handed: List[weakref.ref] = []

    def rows_in_use(self) -> int:
        """The end row of the longest prefix an alive cache object handed out from this set still views (0: the set is free)."""
        rows, alive = 0, []
        for ref in self.handed:
            c = ref()
            if c is None:
                continue
            alive.append(ref)
            for a in (c.transformer.attention or []) if c.transformer is not None else []:
                for t in (a.keys, a.values):
                    if t is not None and t.dim() == 3 and t.untyped_storage().data_ptr() in self._bases:
                        rows = max(rows, (t.storage_offset() % t.stride(0)) // 128 + t.shape[1])
        self.handed = alive
        return rows

    def holds_prefix(self, att, start: int) -> bool:
        """Whether `att` are exactly rows [0, start) of this set's buffers (the caches of a call this set served, cut from the right)."""
        for a, kv in zip(att, self.kv):
            k, v = a.keys, a.values
            if k.shape != (kv.shape[0], start, 64) or v.shape != k.shape or k.stride() != kv.stride() or v.stride() != kv.stride():
                return False
            if k.data_ptr() != kv.data_ptr() or v.data_ptr() != kv.data_ptr() + 64 * kv.element_size():
                return False
        return True


class _RenderSession:
    """Streaming calls of `unmask_mixlm` on one decoder for one (B, style width, capacity); see the comment above `_SESSIONS`.

    Staleness: every call starts with session_begin (csrc/decode_stack.cu), which hashes all parameters and buffers of the decoder
    on the device and compares the fingerprint with the one of the staged weights; the host reads the flag (one 8-byte copy) and
    restages if it is set or if the parameters' addresses changed.  The fingerprint catches what torch's version counters miss: the
    flat AdamW kernel of TrainStep, `p.data` edits, `load_state_dict`."""

    def __init__(self, dec, B: int, S: int, cap: int, dev):
        tr = dec.transformer
        self.B, self.S, self.cap, self.depth, self.dim = B, S, cap, tr.depth, dec.dim
        F = len(dec.token_emb.field_sizes)
        D, n_gb = dec.dim, (2 * tr.depth + 1) * 512
        self.P2 = torch.empty((B, cap, D), dtype=F32, device=dev)
        self.C2 = torch.empty((B, cap, D), dtype=F32, device=dev)
        self.gb_all = torch.empty((B, cap, n_gb), dtype=BF16, device=dev)
        self.tok = torch.zeros((B, cap, F), dtype=torch.int64, device=dev)
        self.mask = torch.ones((B, cap), dtype=torch.bool, device=dev)
        self.zeros = torch.zeros((B, cap, D), dtype=F32, device=dev)       # token_emb / hiddens placeholders of the returned caches
        self.tok_buf = torch.empty((B, F), dtype=torch.int64, device=dev)
        self.p2_buf = torch.empty((B, D), dtype=F32, device=dev)
        self.c2_buf = torch.empty((B, D), dtype=F32, device=dev)
        self.x1_buf = torch.empty((B, F * 128), dtype=BF16, device=dev)
        self.pos_t = torch.zeros(1, dtype=torch.int64, device=dev)
        self.advance = torch.zeros(2, dtype=torch.int32, device=dev)
        self.state = torch.zeros(4, dtype=torch.int64, device=dev)          # session_begin: fingerprint, 2 scratch words, stale flag
        self.sets: List[_KVSet] = [_KVSet(tr.depth, B, cap, dev)]
        self.w: Optional[_DecoderWeights] = None
        self.plan: Optional[K.DecodeStackPlan] = None
        self._ptrs: Optional[Tuple[int, ...]] = None
        self._table: Optional[Tensor] = None
        self.restages = 0

    def _stage(self, dec) -> None:
        w = _DecoderWeights(dec)
        sw = w.sw
        self.w_comp16, b_comp = w.compose_front()
        self.b_p2 = w.bm + b_comp
        self.plan = K.DecodeStackPlan(sw.layers, sw.w_ada, sw.b_ada, self.sets[0].kv, self.B, self.S, advance=self.advance)
        self.plan.set_front(self.x1_buf, self.w_comp16, self.p2_buf, w.en_w.float().contiguous(), w.en_b.float().contiguous(),
                            w.wc_l.t().contiguous(), self.c2_buf)
        self.w = w
        self.restages += 1

    def _kv_set(self, att, start: int) -> _KVSet:
        """The buffer set this call writes rows >= start of: the set `att` is a prefix of when no other alive cache of it reaches
        beyond `start`, else a free set (allocated if none) that the prefix is copied into."""
        if start > 0:
            for s in self.sets:
                if s.holds_prefix(att, start) and s.rows_in_use() <= start:
                    return s
        free = next((s for s in self.sets if s.rows_in_use() == 0), None)
        if free is None:
            free = _KVSet(self.depth, self.B, self.cap, self.P2.device)
            self.sets.append(free)
            if len(self.sets) > SESSION_POOL:      # forgetting a set never overwrites it: its caches keep their buffers alive
                self.sets.pop(0)
        for a, kv in zip(att, free.kv):
            kv[:, :start, :64] = a.keys
            kv[:, :start, 64:] = a.values
        return free

    def render(self, dec, perf: Tensor, masked_perf: Tensor, context: Tensor, style: Tensor, mask: Optional[Tensor],
               fields: Sequence[int], temperature: float, k: int, start: int, caches):
        """`render_decoder(start=start, kv_init=keys | values of caches, return_kv=True, use_graph=False)` plus the caches in the
        reference's layout, with the same tokens and keys / values."""
        B, T, F = perf.shape
        s, n = start, T - start
        sizes = dec.token_emb.field_sizes
        tensors = list(dec.parameters()) + list(dec.buffers())
        ptrs = tuple(t.data_ptr() for t in tensors)
        if ptrs != self._ptrs:                     # `.to()`, re-allocation: hash the new tensors, restage below
            self._table, self._ptrs, self.w = K.fingerprint_table([t.detach() for t in tensors]), ptrs, None
        K.session_begin(self._table, self.state, self.advance, self.pos_t, s)
        if bool(self.state[3].item()) or self.w is None:
            self._stage(dec)
        w, plan, Dm = self.w, self.plan, self.dim
        seed = K.seed_from_torch() if k > 1 else 0
        kvset = self._kv_set(caches.transformer.attention if s > 0 else [], s)
        plan.set_kv(kvset.kv)

        # the per-position terms of the new rows s..T-1 (a row of these launches does not depend on the other rows)
        self.tok[:, s:T] = perf[:, s:T]
        km = None
        if mask is not None:
            self.mask[:, :T] = mask
            km = self.mask
        x2, _, _ = K.embed_ln_fwd(masked_perf[:, s:T].reshape(-1, F), w.table, sizes, w.ln_w, w.ln_b)
        x2p = K.gemm(x2, w.wp16, bias=w.bp, out_dtype=BF16)
        self.P2[:, s:T] = K.gemm(x2p, w.wm_r, bias=self.b_p2, out_dtype=F32).view(B, n, Dm)
        ctx16 = K.cast_bf16(context[:, s:T].float().contiguous().view(B * n, -1))
        self.C2[:, s:T] = K.gemm(ctx16, w.wc_r, bias=w.bc, out_dtype=F32).view(B, n, Dm)
        self.gb_all[:, s:T] = plan.prepare_adaln(style[:, s:T].float().contiguous())

        offs, vocab, ks = [w.offs[f] for f in fields], [sizes[f] for f in fields], [k] * len(fields)
        gather_src, gather_dst = [self.tok, self.P2, self.C2], [self.tok_buf, self.p2_buf, self.c2_buf]
        for _ in range(T - 1 - s):
            # the note-step of render_decoder with the stack kernel, its input front and the sampling kernel that ends the step
            K.gather_at_pos(gather_src, gather_dst, [0, 1, 1], self.pos_t)
            K.embed_ln_fwd(self.tok_buf, w.table, sizes, w.ln_w, w.ln_b, out=self.x1_buf)
            plan.step(None, None, km, self.pos_t, gb_all=self.gb_all, use_front=True, barrier_is_zero=True)
            e_raw = K.gemm(plan.out16, w.whead16, trans_b=True, out_dtype=BF16)
            e, _, _ = K.layer_norm_fwd(e_raw, w.hn_w, w.hn_b, out_dtype=BF16, need_stats=False)
            K.sample_fields(e, w.table16, fields, offs, vocab, ks, self.tok, self.pos_t, temperature=temperature, seed=seed,
                            advance=plan.advance)
        res = perf.clone()
        res[:, s + 1:T] = self.tok[:, s + 1:T]
        out_caches = _kv_only_caches(dec, kvset.kv, T - 1, zeros=self.zeros)
        kvset.handed.append(weakref.ref(out_caches))
        return res, out_caches


def _unmask_stepwise(wrapper, out, tokens_masked, mask, notes, hit, temperature, filter_logits_fn, filter_kwargs, filter_key_ids, caches, kwargs):
    """General stepper: one cached forward per note (the wrapper's own `forward` slices context / style / masks the way training
    does), logits of the note's masked fields from the tied head, host-side filter + draw."""
    names = list(wrapper.model.lm_head.embs.keys())
    if mask is None:
        mask = torch.ones(out.shape[:2], dtype=torch.bool, device=out.device)
    for idx in notes.tolist():
        keys = torch.nonzero(hit[0, idx]).flatten().tolist()
        step = wrapper(out[:, :idx + 1], seq_masked=tokens_masked[:, :idx + 1], mask=mask[:, :idx + 1], return_embeddings=True,
                       return_caches=True, caches=caches, **kwargs)
        caches = step.caches
        logits = wrapper.model.lm_head(step.hidden_state[:, idx - 1], keys=keys)
        out[:, idx, keys] = _draw(logits, (wrapper.pad_token_id, wrapper.mask_token_id), filter_key_ids, filter_logits_fn, filter_kwargs,
                                  temperature)
    return out, caches


@torch.inference_mode()
def unmask_mlm(wrapper, tokens: Tensor, single_run: bool, temperature: float, filter_logits_fn, filter_kwargs, filter_key_ids, **kwargs):
    """Masked-LM unmasking (wrappers.py:131-198 of the reference): every MASK at once from one forward (`single_run`, arg-max),
    or note by note re-running the (uncached, bidirectional) model."""
    dec = wrapper.model
    was_training = dec.training
    dec.eval()
    squeeze = tokens.dim() == 2
    out = (tokens[None] if squeeze else tokens).clone()
    mask = kwargs.pop("mask", None)
    if mask is None:
        mask = torch.ones(out.shape[:2], dtype=torch.bool, device=out.device)
    notes, _, hit = _masked_columns(out, wrapper.mask_token_id)
    if single_run:
        logits = dec(out, mask=mask, **kwargs).logits
        best = torch.stack([lg.argmax(dim=-1) for lg in logits.values()], dim=-1)
        out = torch.where(hit, best, out)
    else:
        for idx in notes.tolist():
            keys = torch.nonzero(hit[0, idx]).flatten().tolist()
            step = wrapper(out[:, :idx + 1], mask=mask[:, :idx + 1], return_embeddings=True, **kwargs)
            logits = dec.lm_head(step.hidden_state[:, idx - 1], keys=keys)
            out[:, idx, keys] = _draw(logits, range(wrapper.num_special_tokens), filter_key_ids, filter_logits_fn, filter_kwargs, temperature)
    dec.train(was_training)
    return out[0] if squeeze else out


@torch.inference_mode()
def generate_ar(wrapper, start_tokens: Tensor, seq_len: int, max_bar, temperature: float, filter_logits_fn, filter_kwargs, caches,
                return_caches: bool, tokenizer, fix_errors: bool, **kwargs):
    """Causal-LM continuation (wrappers.py:200-307 of the reference): append one sampled tuple per step through the cached stack
    step until `seq_len`, EOS, or a bar beyond `max_bar`.  With a tokenizer and `fix_errors` the bar never decreases and the
    tempo / time signature are held inside a bar."""
    dec = wrapper.model
    was_training = dec.training
    dec.eval()
    squeeze = start_tokens.dim() == 2
    out = start_tokens[None] if squeeze else start_tokens
    t0 = out.shape[1]
    mask = kwargs.pop("mask", None)
    if mask is None:
        mask = torch.ones(out.shape[:2], dtype=torch.bool, device=out.device)
    col = getattr(tokenizer, "vocab_types_idx", None) if fix_errors else None
    for _ in range(t0, seq_len + 1):
        window, wmask = out[:, -wrapper.max_seq_len:], mask[:, -wrapper.max_seq_len:]
        step = wrapper(window, mask=wmask, caches=caches, return_embeddings=True, return_caches=True, **kwargs)
        caches = step.caches
        logits = dec.lm_head(step.hidden_state[:, -1])
        last = out[:, -1]
        new, bar_tok = [], None
        for key, lg in logits.items():
            if col is not None and key == "Bar":
                lg = lg.clone()
                lg[:, 4:int(last[0, col["Bar"]])] = -float("inf")           # bars only move forward
            held = col is not None and (key == "TimeSig" or (key == "Tempo" and bar_tok is not None and bool((bar_tok == last[:, col["Bar"]]).all())))
            tok = last[:, col[key]][:, None] if held else _draw({key: lg}, (0, 1), None, filter_logits_fn, filter_kwargs, temperature)
            if key == "Bar":
                bar_tok = tok[:, 0]
            new.append(tok)
        out = torch.cat([out, torch.cat(new, dim=-1)[:, None]], dim=1)
        mask = torch.nn.functional.pad(mask, (0, 1), value=True)
        if wrapper.eos_token_id is not None:
            if bool((out[:, -1, 0] == wrapper.eos_token_id).any()):
                out[:, -1, 1:] = wrapper.pad_token_id
                break
        elif max_bar is not None and bool((out[:, -1, 0] > max_bar).any()):
            out = out[:, :-1]
            break
    out = out[:, t0:]
    dec.train(was_training)
    out = out[0] if squeeze else out
    return (out, caches) if return_caches else out
