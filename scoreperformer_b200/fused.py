"""Autograd boundaries of the B200 path: each Function below is a hand-scheduled forward + backward over the
C-ABI kernels (scoreperformer_b200.kernels).  PyTorch only owns the tensors and the graph edges between
these few coarse nodes; no arithmetic on activations happens in Python.

Numerics: bf16 tensor-core operands, fp32 accumulation, fp32 residual stream / LayerNorm statistics / softmax /
losses -- i.e. what `torch.autocast(bfloat16)` does to the reference modules (SURVEY.md section 7, "fp16+GradScaler vs bf16").
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import kernels as K

BF16, F32 = torch.bfloat16, torch.float32

# ----------------------------------------------------------------------------- step-level plumbing (set by train_step.TrainStep)
# DIRECT_GRAD: weight-gradient kernels accumulate straight into `param.grad` (a view of the flat gradient buffer) and the
#   autograd node returns None for that input -- no temporary, no AccumulateGrad add kernel.
# SHADOW_ACTIVE: parameters carry `_spb_shadow`, a bf16 view of the flat weight shadow that ONE cast kernel refreshed at the
#   start of this step.  Both flags are only True inside TrainStep's forward/backward, so stale shadows are never read.
DIRECT_GRAD = False
SHADOW_ACTIVE = False
# STACK_BACKWARD_DONE: callable(params) or None.  TransformerStackFn.backward calls it once every weight gradient of its stack has
#   been written: TrainStep launches that stack's gradient bucket on NCCL.
STACK_BACKWARD_DONE = None


def _shadow(param: Tensor) -> Optional[Tensor]:
    return getattr(param, "_spb_shadow", None) if SHADOW_ACTIVE else None


def w16(param: Tensor) -> Tensor:
    """bf16 copy of a weight: the per-step shadow when active, else a fresh cast."""
    t = _shadow(param)
    return t if t is not None else K.cast_bf16(param.detach().contiguous())


def w16_cat(params: Sequence[Tensor]) -> Tensor:
    """bf16 copy of the row-concatenation of weights; free when their shadows are adjacent in the flat buffer."""
    shadows = [_shadow(p) for p in params]
    if all(t is not None for t in shadows):
        ok = all(shadows[i].data_ptr() + shadows[i].numel() * 2 == shadows[i + 1].data_ptr() for i in range(len(shadows) - 1))
        if ok:
            rows = sum(t.shape[0] for t in shadows)
            return torch.as_strided(shadows[0], (rows, shadows[0].shape[1]), (shadows[0].shape[1], 1))
        return torch.cat(shadows, dim=0)
    return K.cast_bf16(torch.cat([p.detach() for p in params], dim=0))


def direct_grad(param: Tensor) -> Optional[Tensor]:
    if not DIRECT_GRAD:
        return None
    g = param.grad
    if g is None or g.dtype != F32 or not g.is_contiguous() or g.shape != param.shape:
        return None
    return g


def direct_grad_cat(params: Sequence[Tensor]) -> Optional[Tensor]:
    """One [sum rows, cols] view over adjacent gradient slots (to_q | to_k | to_v), or None."""
    gs = [direct_grad(p) for p in params]
    if any(g is None for g in gs):
        return None
    if not all(gs[i].data_ptr() + gs[i].numel() * 4 == gs[i + 1].data_ptr() for i in range(len(gs) - 1)):
        return None
    rows = sum(g.shape[0] for g in gs)
    return torch.as_strided(gs[0], (rows, gs[0].shape[1]), (gs[0].shape[1], 1))


def wgrad(param: Tensor, a: Tensor, b: Tensor, alpha: Optional[Tensor] = None) -> Optional[Tensor]:
    """dW[M, N] = a^T b for a stored [K, M], b stored [K, N]: accumulated into param.grad (returns None) or returned."""
    g = direct_grad(param)
    if g is not None:
        K.gemm(a, b, trans_a=True, trans_b=True, out=g, split_k=0, accumulate=True, alpha=alpha)
        return None
    return K.gemm(a, b, trans_a=True, trans_b=True, out_dtype=F32, split_k=0, alpha=alpha)


def vgrad(param: Tensor) -> Tuple[Tensor, bool]:
    """Accumulate-into buffer for a vector gradient: (param.grad.view(-1), True) in direct mode, else (zeros, False)."""
    g = direct_grad(param)
    if g is not None:
        return g.view(-1), True
    return torch.zeros(param.numel(), dtype=F32, device=param.device), False



# ----------------------------------------------------------------------------- generic Linear
class LinearFn(torch.autograd.Function):
    """y = x W^T + b with bf16 operands (nn.Linear under autocast).  x: [n, in] fp32 or bf16; W fp32 [out, in].

    `w_is_kn=True` multiplies by a weight stored [in, out] (the tied head's `x @ project_emb.weight`,
    models/scoreperformer/embeddings.py:346)."""

    @staticmethod
    def forward(ctx, x, weight, bias, out_fp32: bool, w_is_kn: bool):
        x16 = K.cast_bf16(x.contiguous()) if x.dtype == F32 else x
        w_16 = w16(weight)
        y = K.gemm(x16, w_16, trans_b=w_is_kn, bias=bias, out_dtype=F32 if out_fp32 else BF16)
        ctx.saved = (x16, w_16, weight, bias)
        ctx.meta = (x.dtype, w_is_kn, bias is not None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x16, w_16, weight, bias = ctx.saved
        x_dtype, w_is_kn, has_bias = ctx.meta
        dy = dy.contiguous()
        dy16 = K.cast_bf16(dy) if dy.dtype == F32 else dy
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            # dx[n, in] = dy[n, out] @ W[out, in]   (B operand must be [in, out]-indexed: MN-major unless stored [in, out])
            dx = K.gemm(dy16, w_16, trans_b=not w_is_kn, out_dtype=x_dtype)
        if ctx.needs_input_grad[1]:
            dw = wgrad(weight, x16, dy16) if w_is_kn else wgrad(weight, dy16, x16)     # [in,out] = x^T dy  |  [out,in] = dy^T x
        if has_bias and ctx.needs_input_grad[2]:
            buf, direct = vgrad(bias)
            K.colsum(dy16, out=buf)
            db = None if direct else buf
        return dx, dw, db, None, None


def linear(x: Tensor, weight: Tensor, bias: Optional[Tensor] = None, out_fp32: bool = False, w_is_kn: bool = False) -> Tensor:
    shape = x.shape
    y = LinearFn.apply(x.reshape(-1, shape[-1]), weight, bias, out_fp32, w_is_kn)
    return y.view(*shape[:-1], y.shape[-1])


# ----------------------------------------------------------------------------- LayerNorm
class LayerNormFn(torch.autograd.Function):
    """nn.LayerNorm(dim) with fp32 statistics; x fp32 or bf16 [n, dim]; output dtype selectable."""

    @staticmethod
    def forward(ctx, x, weight, bias, out_fp32: bool, eps: float):
        x = x.contiguous()
        y, mean, rstd = K.layer_norm_fwd(x, weight, bias, out_dtype=F32 if out_fp32 else BF16, eps=eps)
        ctx.saved = (x, mean, rstd, weight, bias)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, mean, rstd, weight, bias = ctx.saved
        dy = dy.contiguous()
        dy16 = K.cast_bf16(dy) if dy.dtype == F32 else dy
        dw, d1 = vgrad(weight)
        db, d2 = vgrad(bias)
        dx = K.layer_norm_bwd(dy16, x, mean, rstd, weight, dx_dtype=BF16, dw=dw, db=db)
        if x.dtype == F32:
            dx = dx.float()
        return dx, None if d1 else dw, None if d2 else db, None, None


def layer_norm(x: Tensor, weight: Tensor, bias: Tensor, out_fp32: bool = False, eps: float = 1e-5) -> Tensor:
    shape = x.shape
    return LayerNormFn.apply(x.reshape(-1, shape[-1]), weight, bias, out_fp32, eps).view(shape)


# ----------------------------------------------------------------------------- computed per-field tables (a1)
class TableBuildFn(torch.autograd.Function):
    """table [sum V_f, 128] = cat_f ( index rows of the discrete ids | MLP(token_values_f) elsewhere ), one launch for all fields.

    modules/transformer/embeddings.py:124-143 (token_weight + value_weight) with the dense value MLP of :199-211.
    params: per field (index_weight, W0 [128,1], b0, W1 [128,128], b1); consts: per field (token_values [V,1], discrete mask [V,1])."""

    @staticmethod
    def forward(ctx, sizes: Tuple[int, ...], consts: Tuple[Tensor, ...], *params):
        nf = len(sizes)
        per_field = []
        for f in range(nf):
            iw, w0, b0, w1, b1 = params[5 * f:5 * f + 5]
            per_field.append((iw.detach(), consts[2 * f], consts[2 * f + 1], w0.detach(), b0.detach(), w1.detach(), b1.detach()))
        ctx.sizes, ctx.consts, ctx.params = sizes, consts, params
        return K.table_build_fwd(sizes, per_field)

    @staticmethod
    def backward(ctx, dtable):
        sizes, consts, params = ctx.sizes, ctx.consts, ctx.params
        nf = len(sizes)
        per_field, grads = [], []
        for f in range(nf):
            ps = params[5 * f:5 * f + 5]
            bufs = []
            for p_ in ps:
                g = direct_grad(p_)
                if g is not None:
                    bufs.append(g)
                    grads.append(None)
                else:
                    z = torch.zeros_like(p_)
                    bufs.append(z)
                    grads.append(z)
            per_field.append((ps[0].detach(), consts[2 * f], consts[2 * f + 1], ps[1].detach(), ps[2].detach(), ps[3].detach(),
                              ps[4].detach(), *bufs))
        K.table_build_bwd(sizes, per_field, dtable.contiguous())
        return (None, None) + tuple(grads)


# ----------------------------------------------------------------------------- tuple-token embedding (a1/a2)
class TupleEmbedFn(torch.autograd.Function):
    """project_emb(LayerNorm(cat_f table_f[tokens_f])) -> bf16 [n, dim]  (models/scoreperformer/embeddings.py:121-143)."""

    @staticmethod
    def forward(ctx, tokens, table, ln_w, ln_b, proj_w, proj_b, sizes: Tuple[int, ...]):
        x16, mean, rstd = K.embed_ln_fwd(tokens, table.contiguous(), sizes, ln_w, ln_b)
        w_16 = w16(proj_w)
        y = K.gemm(x16, w_16, bias=proj_b, out_dtype=BF16)
        ctx.saved = (tokens, table, ln_w, ln_b, proj_w, proj_b, mean, rstd, x16, w_16)
        ctx.sizes = sizes
        return y

    @staticmethod
    def backward(ctx, dy):
        tokens, table, ln_w, ln_b, proj_w, proj_b, mean, rstd, x16, w_16 = ctx.saved
        dy16 = dy if dy.stride(-1) == 1 else dy.contiguous()
        assert dy16.dtype == BF16
        dproj_w = wgrad(proj_w, dy16, x16)
        dpb, d0 = vgrad(proj_b)
        K.colsum(dy16, out=dpb)
        dx16 = K.gemm(dy16, w_16, trans_b=True, out_dtype=BF16)
        dtable = torch.zeros_like(table)
        dln_w, d1 = vgrad(ln_w)
        dln_b, d2 = vgrad(ln_b)
        K.embed_ln_bwd(dx16, tokens, table, ctx.sizes, ln_w, mean, rstd, dtable, dln_w, dln_b)
        return None, dtable, None if d1 else dln_w, None if d2 else dln_b, dproj_w, None if d0 else dpb, None


# ----------------------------------------------------------------------------- stand-alone attention core / GLU
class AttentionCoreFn(torch.autograd.Function):
    """softmax(scale q k^T - slope|i-j| + masks) v for MQA; qkv bf16 [B*T, H*64+128] (modules/transformer/attend.py:58-126)."""

    @staticmethod
    def forward(ctx, qkv, mask, logslopes, B, T, H, causal, dropout_p, seed):
        ls = logslopes.detach().reshape(-1).contiguous()
        o, lse, aux = K.attention_fwd(qkv, mask, ls, B, T, H, causal, dropout_p, seed)
        ctx.saved = (qkv, mask, ls, o, lse, aux)
        ctx.meta = (B, T, H, causal, dropout_p, seed, logslopes.shape)
        return o

    @staticmethod
    def backward(ctx, do):
        qkv, mask, ls, o, lse, aux = ctx.saved
        B, T, H, causal, dropout_p, seed, ls_shape = ctx.meta
        dls = torch.zeros(H, dtype=F32, device=qkv.device)
        dqkv = K.attention_bwd(qkv, mask, ls, o, do.contiguous(), lse, dls, B, T, H, causal, dropout_p, seed, aux=aux)
        return dqkv, None, dls.view(ls_shape), None, None, None, None, None, None


class GLUFn(torch.autograd.Function):
    """value * silu(gate) with dropout; u bf16 [n, 2H] (modules/transformer/feedforward.py:13-22,59)."""

    @staticmethod
    def forward(ctx, u, dropout_p, seed):
        u = u.contiguous()
        ctx.saved = (u, dropout_p, seed)
        return K.glu_fwd(u, dropout_p, seed)

    @staticmethod
    def backward(ctx, dh):
        u, dropout_p, seed = ctx.saved
        return K.glu_bwd(dh.contiguous(), u, None, dropout_p, seed), None, None


# ----------------------------------------------------------------------------- transformer stack (a4-a7)
@dataclass(frozen=True)
class StackSpec:
    depth: int
    heads: int
    dim: int
    dim_head: int
    ff_inner: int
    causal: bool
    ada: bool
    attn_dropout: float
    ff_dropout: float
    training: bool
    eps: float = 1e-5
    return_hiddens: bool = False

    @property
    def n_norms(self) -> int:
        return 2 * self.depth + 1


PARAMS_PER_ATTN = 7   # norm_a, norm_b, to_q, to_k, to_v, to_out, logslopes
PARAMS_PER_FF = 5     # norm_a, norm_b, proj_w, proj_b, out_w


class TransformerStackFn(torch.autograd.Function):
    """Pre-norm ('a','f') x depth stack + final norm (modules/transformer/transformer.py:139-232) as ONE graph node.

    x fp32 [B, T, D] (the residual stream stays fp32), mask bool [B, T] or None, style fp32 [B, T, S] (AdaLN) or None.
    params: per layer pair (norm_a, norm_b, to_q, to_k, to_v, to_out, logslopes), (norm_a, norm_b, proj_w, proj_b, out_w),
    then the final norm (a, b); for AdaLN (norm_a, norm_b) are the `linear.weight [2D, S]` / `linear.bias [2D]` of each
    AdaptiveLayerNorm (modules/layers.py:31-47) -- all of them are evaluated by one batched GEMM.
    Returns (out fp32 [B,T,D], hiddens fp32 [depth, B, T, D] = attention-layer inputs, kv bf16 [depth, B*T, 128]).
    """

    @staticmethod
    def forward(ctx, spec: StackSpec, x, mask, style, seeds, *params):
        B, T, D = x.shape
        N = B * T
        H, dh = spec.heads, spec.dim_head
        x2 = x.contiguous().view(N, D)
        keep = any(ctx.needs_input_grad)
        layers: List[dict] = []
        gb_all = style16 = w_ada16 = None
        if spec.ada:
            norm_w = [params[_norm_index(spec, i)] for i in range(spec.n_norms)]
            norm_b = [params[_norm_index(spec, i) + 1] for i in range(spec.n_norms)]
            style16 = K.cast_bf16(style.contiguous().view(N, -1))
            w_ada16 = w16_cat(norm_w)
            # (gamma - 1 | beta) per norm: the kernels add the 1 back in fp32 (gamma stays near its initial value 1)
            gb_all = K.gemm(style16, w_ada16, bias=ada_bias_minus_one(norm_b, D), out_dtype=BF16)   # [N, n_norms * 2D]

        def norm_fwd(i_norm, xin, out_dtype=BF16):
            if spec.ada:
                gb = gb_all[:, i_norm * 2 * D:(i_norm + 1) * 2 * D]
                y, mean, rstd = K.layer_norm_fwd(xin, None, None, gb, out_dtype=out_dtype, eps=spec.eps)
            else:
                j = _norm_index(spec, i_norm)
                y, mean, rstd = K.layer_norm_fwd(xin, params[j], params[j + 1], out_dtype=out_dtype, eps=spec.eps)
            return y, mean, rstd

        n_keep = spec.depth if spec.return_hiddens else 0
        hiddens = torch.empty((n_keep, N, D), dtype=F32, device=x.device)
        kvs = torch.empty((n_keep, N, 2 * dh), dtype=BF16, device=x.device)
        cur = x2
        p_attn = spec.attn_dropout if spec.training else 0.0
        p_ff = spec.ff_dropout if spec.training else 0.0
        for l in range(spec.depth):
            base = l * (PARAMS_PER_ATTN + PARAMS_PER_FF)
            # ---- attention sub-layer
            if spec.return_hiddens:
                hiddens[l].copy_(cur)
            to_q, to_k, to_v, to_out, logslopes = params[base + 2:base + 7]
            xn, mean, rstd = norm_fwd(2 * l, cur)
            wqkv16 = w16_cat([to_q, to_k, to_v])
            qkv = K.gemm(xn, wqkv16, out_dtype=BF16)
            ls = logslopes.detach().reshape(-1).contiguous()
            o, lse, aux = K.attention_fwd(qkv, mask, ls, B, T, H, spec.causal, p_attn, seeds[2 * l], need_aux=keep)
            wo16 = w16(to_out)
            nxt = K.gemm(o, wo16, residual=cur, rowmask=None if mask is None else mask.view(-1), out_dtype=F32)
            if spec.return_hiddens:
                kvs[l].copy_(qkv[:, H * dh:])
            rec_a = dict(x=cur, mean=mean, rstd=rstd, xn=xn, wqkv16=wqkv16, qkv=qkv, ls=ls, o=o, lse=lse, wo16=wo16, aux=aux) if keep else None
            cur = nxt
            # ---- feed-forward sub-layer
            proj_w, proj_b, out_w = params[base + PARAMS_PER_ATTN + 2:base + PARAMS_PER_ATTN + 5]
            xn, mean, rstd = norm_fwd(2 * l + 1, cur)
            w1_16 = w16(proj_w)
            w2_16 = w16(out_w)
            if K.ffn_fused_ok(D, out_w.shape[1]):
                # one kernel: GEMM1 -> GLU -> dropout -> GEMM2 -> +residual; u / h leave only as the backward's side outputs
                nxt, u, h = K.ffn_fwd(xn, w1_16, proj_b, w2_16, cur, p_ff, seeds[2 * l + 1], save=keep)
            else:
                u = K.gemm(xn, w1_16, bias=proj_b, out_dtype=BF16)
                h = K.glu_fwd(u, p_ff, seeds[2 * l + 1])
                nxt = K.gemm(h, w2_16, residual=cur, out_dtype=F32)
            rec_f = dict(x=cur, mean=mean, rstd=rstd, xn=xn, w1_16=w1_16, u=u, h=h, w2_16=w2_16) if keep else None
            cur = nxt
            layers.append((rec_a, rec_f))
        out, mean, rstd = norm_fwd(2 * spec.depth, cur, out_dtype=F32)
        if keep:
            ctx.spec, ctx.shape, ctx.mask, ctx.seeds = spec, (B, T, D), mask, seeds
            ctx.layers, ctx.final = layers, dict(x=cur, mean=mean, rstd=rstd)
            ctx.ada = (gb_all, style16, w_ada16)
            ctx.params = params
            ctx.style_shape = None if style is None else style.shape
        ctx.mark_non_differentiable(hiddens, kvs)
        return out.view(B, T, D), hiddens.view(n_keep, B, T, D), kvs

    @staticmethod
    def backward(ctx, g_out, _g_hiddens, _g_kvs):
        spec: StackSpec = ctx.spec
        B, T, D = ctx.shape
        N = B * T
        H = spec.heads
        params = ctx.params
        mask = ctx.mask
        gb_all, style16, w_ada16 = ctx.ada
        grads: List[Optional[Tensor]] = [None] * len(params)
        dgb_all = torch.empty_like(gb_all) if spec.ada else None
        p_attn = spec.attn_dropout if spec.training else 0.0
        p_ff = spec.ff_dropout if spec.training else 0.0

        # small accumulate-into gradients: straight into param.grad in direct mode, else ONE zero-initialised buffer (one fill)
        n_small = spec.depth * (2 * spec.ff_inner + H) + (0 if spec.ada else spec.n_norms * 2 * D)
        small = None
        small_off = [0]

        def take(param):
            nonlocal small
            g_direct = direct_grad(param)
            if g_direct is not None:
                return g_direct.view(-1), True
            if small is None:
                small = torch.zeros(n_small, dtype=F32, device=g_out.device)
            n = param.numel()
            v = small[small_off[0]:small_off[0] + n]
            small_off[0] += n
            return v, False

        rowmask = None if mask is None else mask.view(-1)

        def norm_bwd(i_norm, dy16, rec, dres):
            """LN backward (+ residual gradient); also returns the bf16 copy of the result the NEXT backward GEMM consumes:
            row-masked when that consumer is an attention sub-layer (its output was multiplied by the mask)."""
            next_is_attn = (i_norm % 2 == 1)              # after a feed-forward norm comes the attention sub-layer of that layer
            want16 = i_norm > 0
            rm16 = rowmask if next_is_attn else None
            if spec.ada:
                sl = slice(i_norm * 2 * D, (i_norm + 1) * 2 * D)
                res = K.layer_norm_bwd(dy16, rec["x"], rec["mean"], rec["rstd"], None, gb_all[:, sl], dres=dres, dx_dtype=F32,
                                       dgb=dgb_all[:, sl], want_dx16=want16, dx16_rowmask=rm16)
                return res if want16 else (res, None)
            j = _norm_index(spec, i_norm)
            dw, d1 = take(params[j])
            db, d2 = take(params[j + 1])
            res = K.layer_norm_bwd(dy16, rec["x"], rec["mean"], rec["rstd"], params[j], dres=dres, dx_dtype=F32, dw=dw, db=db,
                                   want_dx16=want16, dx16_rowmask=rm16)
            grads[j], grads[j + 1] = (None if d1 else dw), (None if d2 else db)
            return res if want16 else (res, None)

        g, g16 = norm_bwd(2 * spec.depth, K.cast_bf16(g_out.contiguous().view(N, D)), ctx.final, None)
        w2t_all = None
        if K.ffn_bwd_fused_ok(D, spec.ff_inner):       # out-projection weights of every layer, transposed in one launch
            w2t_all = K.transpose_bf16([ctx.layers[l][1]["w2_16"] for l in range(spec.depth)])
        for l in reversed(range(spec.depth)):
            base = l * (PARAMS_PER_ATTN + PARAMS_PER_FF)
            rec_a, rec_f = ctx.layers[l]
            # ---- feed-forward backward:  x_out = x + W2 glu(W1 LN(x) + b1)
            p_w1, p_b1, p_w2 = params[base + PARAMS_PER_ATTN + 2:base + PARAMS_PER_ATTN + 5]
            grads[base + PARAMS_PER_ATTN + 4] = wgrad(p_w2, g16, rec_f["h"])
            db1, d_b1 = take(p_b1)
            if K.ffn_bwd_fused_ok(D, spec.ff_inner):
                # one kernel: dh = dy W2 (on chip) -> GLU' . mask -> du (written over u) -> dxn = du W1, db1 += colsum(du)
                if rec_f["u"] is None:
                    raise RuntimeError("TransformerStackFn: second backward through the same graph (the saved pre-activations were "
                                       "overwritten in place by the first)")
                dxn, du = K.ffn_bwd(g16, w2t_all[l], rec_f["w1_16"], rec_f["u"], db1, p_ff, ctx.seeds[2 * l + 1])
                rec_f["u"] = None
            else:
                dh = K.gemm(g16, rec_f["w2_16"], trans_b=True, out_dtype=BF16)
                du = K.glu_bwd(dh, rec_f["u"], db1, p_ff, ctx.seeds[2 * l + 1])
                dxn = None
            grads[base + PARAMS_PER_ATTN + 3] = None if d_b1 else db1
            grads[base + PARAMS_PER_ATTN + 2] = wgrad(p_w1, du, rec_f["xn"])
            if dxn is None:
                dxn = K.gemm(du, rec_f["w1_16"], trans_b=True, out_dtype=BF16)
            g, g16 = norm_bwd(2 * l + 1, dxn, rec_f, g)
            # ---- attention backward:  x_out = x + mask * Wo attn(Wqkv LN(x))
            p_q, p_k, p_v, p_o, p_ls = params[base + 2:base + 7]
            grads[base + 5] = wgrad(p_o, g16, rec_a["o"])
            # dO = dY Wo and delta = rowsum(dO * O) in one GEMM (the epilogue owns whole rows of a head)
            do, delta = K.gemm_rowdot(g16, rec_a["wo16"], rec_a["o"], T, H, trans_b=True)
            dls, d_ls = take(p_ls)
            dqkv = K.attention_bwd(rec_a["qkv"], mask, rec_a["ls"], rec_a["o"], do, rec_a["lse"], dls, B, T, H, spec.causal, p_attn,
                                   ctx.seeds[2 * l], delta=delta, aux=rec_a["aux"])
            grads[base + 6] = None if d_ls else dls.view(p_ls.shape)
            g_qkv = direct_grad_cat([p_q, p_k, p_v])
            if g_qkv is not None:
                K.gemm(dqkv, rec_a["xn"], trans_a=True, trans_b=True, out=g_qkv, split_k=0, accumulate=True)
            else:
                dwqkv = K.gemm(dqkv, rec_a["xn"], trans_a=True, trans_b=True, out_dtype=F32, split_k=0)
                hq = H * spec.dim_head
                grads[base + 2], grads[base + 3], grads[base + 4] = dwqkv[:hq], dwqkv[hq:hq + spec.dim_head], dwqkv[hq + spec.dim_head:]
            dxn = K.gemm(dqkv, rec_a["wqkv16"], trans_b=True, out_dtype=BF16)
            g, g16 = norm_bwd(2 * l, dxn, rec_a, g)
        d_style = None
        if spec.ada:
            dw_ada = K.gemm(dgb_all, style16, trans_a=True, trans_b=True, out_dtype=F32, split_k=0)   # [n_norms*2D, S]
            db_ada = K.colsum(dgb_all)
            add_dst, add_src = [], []
            for i in range(spec.n_norms):
                j = _norm_index(spec, i)
                gw, gb = dw_ada[i * 2 * D:(i + 1) * 2 * D], db_ada[i * 2 * D:(i + 1) * 2 * D]
                dw_direct, db_direct = direct_grad(params[j]), direct_grad(params[j + 1])
                if dw_direct is not None and db_direct is not None:
                    # straight into the gradient buffers, all norms in one launch (and under data parallelism nothing may be left
                    # for autograd's AccumulateGrad: the stack's gradient bucket leaves for NCCL at the end of this node)
                    add_dst += [dw_direct, db_direct]
                    add_src += [gw, gb]
                else:
                    grads[j], grads[j + 1] = gw, gb
            K.multi_add(add_dst, add_src)
            if ctx.needs_input_grad[3]:
                d_style = K.gemm(dgb_all, w_ada16, trans_b=True, out_dtype=F32).view(ctx.style_shape)
        if STACK_BACKWARD_DONE is not None and DIRECT_GRAD:
            STACK_BACKWARD_DONE(params)
        return (None, g.view(B, T, D), None, d_style, None) + tuple(grads)


_ADA_ONES = {}


def ada_bias_minus_one(norm_b: Sequence[Tensor], D: int) -> Tensor:
    """cat of the AdaLN linear biases with 1 subtracted from every gamma half: the batched GEMM then produces (gamma - 1 | beta),
    which is what spb_layer_norm_fwd / _bwd expect in `gb`."""
    key = (len(norm_b), D, str(norm_b[0].device))
    ones = _ADA_ONES.get(key)
    if ones is None:
        ones = torch.zeros(len(norm_b), 2, D, dtype=F32, device=norm_b[0].device)
        ones[:, 0] = 1.0
        ones = _ADA_ONES[key] = ones.view(-1)
    return torch.cat(list(norm_b), dim=0).float() - ones


def _norm_index(spec: StackSpec, i_norm: int) -> int:
    """Index into the flat params tuple of the first tensor of norm number i_norm (0 .. 2*depth)."""
    if i_norm == 2 * spec.depth:
        return spec.depth * (PARAMS_PER_ATTN + PARAMS_PER_FF)
    l, is_ff = divmod(i_norm, 2)
    return l * (PARAMS_PER_ATTN + PARAMS_PER_FF) + (PARAMS_PER_ATTN if is_ff else 0)


# ----------------------------------------------------------------------------- hierarchical latents (a8)
class LatentLevelsFn(torch.autograd.Function):
    """All VAE levels of MMDTupleTransformer._forward_latents (mmd_transformer.py:242-278, 304-368), hierarchical with context.

    hidden fp32 [B,T,D]; mask bool [B,T]; segments: per level int64 [B,T] or None ('mean'); S: per-level slot count.
    Returns style fp32 [B,T,sum z] (the un-dropped, masked embeddings) followed by per level (latents [B,S,z], lmask [B,S]).
    """

    @staticmethod
    def forward(ctx, hidden, mask, segments: Sequence[Optional[Tensor]], slots: Sequence[int], zs: Sequence[int], *wb):
        B, T, D = hidden.shape
        hidden = hidden.contiguous()
        total = int(sum(zs))
        style = torch.zeros((B, T, total), dtype=F32, device=hidden.device)
        outs, saved = [], []
        col = 0
        for lvl, (seg, S, z) in enumerate(zip(segments, slots, zs)):
            W, b = wb[2 * lvl].contiguous(), wb[2 * lvl + 1].contiguous()
            lat, lmask, pooled, counts = K.latent_level_fwd(hidden, style, mask, seg, W, b, col, S, z)
            outs += [lat, lmask]
            saved.append((seg, S, z, col, W, pooled, counts, lmask))
            col += z
        ctx.saved = saved
        ctx.wb = wb
        ctx.mask = mask
        ctx.shape = (B, T, D)
        ctx.mark_non_differentiable(*[o for o in outs[1::2]])
        return (style, *outs)

    @staticmethod
    def backward(ctx, d_style, *d_outs):
        B, T, D = ctx.shape
        d_style = d_style.contiguous().clone() if d_style is not None else None
        if d_style is None:
            d_style = torch.zeros((B, T, sum(s[2] for s in ctx.saved)), dtype=F32, device=ctx.mask.device)
        d_hidden = torch.zeros((B, T, D), dtype=F32, device=d_style.device)
        grads_wb: List[Optional[Tensor]] = [None] * (2 * len(ctx.saved))
        for lvl in reversed(range(len(ctx.saved))):
            seg, S, z, col, W, pooled, counts, lmask = ctx.saved[lvl]
            d_lat = d_outs[2 * lvl]
            d_lat = None if d_lat is None else d_lat.contiguous()
            p_w, p_b = ctx.wb[2 * lvl], ctx.wb[2 * lvl + 1]
            g_w = direct_grad(p_w)
            dW = g_w if g_w is not None else torch.zeros_like(W)
            db, d_b = vgrad(p_b)
            K.latent_level_bwd(d_style, col, d_lat, ctx.mask, seg, W, pooled, counts, lmask, d_hidden, dW, db, S, z)
            grads_wb[2 * lvl], grads_wb[2 * lvl + 1] = (None if g_w is not None else dW), (None if d_b else db)
        return (d_hidden, None, None, None, None) + tuple(grads_wb)


class MMDFn(torch.autograd.Function):
    """Fused pairwise-RBF MMD between the prior sample z and the valid latents (mmd_transformer.py:505-534)."""

    @staticmethod
    def forward(ctx, y, w, z_prior):
        loss, grad = K.mmd_fwd_bwd(z_prior.contiguous(), y.contiguous(), w.contiguous())
        ctx.saved = grad
        return loss.view(())

    @staticmethod
    def backward(ctx, g):
        return ctx.saved * g, None, None


# ----------------------------------------------------------------------------- tied LM head + masked CE (a10)
def _eval_stats_from_logits(logits: Tensor, labels: Tensor, tv: Optional[Tensor], ignore_index: int) -> Tensor:
    """(hits, sum |tv[argmax]-tv[label]|, sum_v p_v |tv[label]-tv[v]|) over the labelled rows, from materialised logits: the
    statement of what spb_head_ce accumulates in tensor memory (fields too wide for it take this path)."""
    use = labels != ignore_index
    lab = labels.clamp(min=0)
    pred = logits.argmax(dim=-1)
    hits = ((pred == lab) & use).sum().float()
    if tv is None:
        return torch.stack([hits, hits.new_zeros(()), hits.new_zeros(())])
    tv = tv.to(logits.device, F32)
    dist = ((tv[pred] - tv[lab]).abs() * use).sum()
    wdist = ((logits.float().softmax(-1) * (tv[lab][:, None] - tv[None, :]).abs()).sum(-1) * use).sum()
    return torch.stack([hits, dist, wdist])


class TiedHeadCEFn(torch.autograd.Function):
    """loss = mean over labelled fields of CE(LN(h @ Wp)[field] @ table_field^T, labels[field]).

    models/scoreperformer/embeddings.py:345-353 + wrappers.py:49-59.  Only the `fields` that carry labels are contracted;
    the gradient wrt logits (softmax - onehot) is produced in the same pass as the loss, so fp32 logits are consumed
    where they are produced and only the bf16 dlogits of the labelled fields are kept for the two backward GEMMs.
    Returns (loss, per_field_loss [n_fields_total] (nan where inactive), counts).
    """

    @staticmethod
    def forward(ctx, hidden, proj_w, ln_w, ln_b, table, labels, sizes: Tuple[int, ...], fields: Tuple[int, ...], emb: int,
                ignore_index: int, token_values=None):
        """`token_values`: None, or one fp32 [V_f] tensor (or None) per field -- the value each token stands for.  When given,
        the head kernel also accumulates the evaluator's statistics of the labelled rows (evaluator.py:38-46,72-104) while
        the logits are in tensor memory: stats[f] = (hits, sum |tv[argmax]-tv[label]|, sum_v p_v |tv[label]-tv[v]|)."""
        n = hidden.shape[0]
        dev = hidden.device
        h16 = K.cast_bf16(hidden.contiguous()) if hidden.dtype == F32 else hidden.contiguous()
        wp16 = w16(proj_w)                                          # [dim, F*emb]
        # the projection stays fp32 until its LayerNorm (one bf16 rounding less in front of the logits; 1536 columns only)
        e_raw = K.gemm(h16, wp16, trans_b=True, out_dtype=F32)     # [n, F*emb]
        e, mean, rstd = K.layer_norm_fwd(e_raw, ln_w, ln_b, out_dtype=BF16)
        table16 = K.cast_bf16(table.contiguous())
        offs = [0]
        for v in sizes[:-1]:
            offs.append(offs[-1] + v)
        nf = len(sizes)
        acc = torch.zeros((2, nf), dtype=F32, device=dev)           # one fill: loss sums, counts
        loss_sum, count = acc[0], acc[1]
        stats_buf = torch.zeros((nf, 3), dtype=F32, device=dev) if token_values is not None else None
        dlogits = {}
        need_grad = any(ctx.needs_input_grad)
        for f in fields:
            V = sizes[f]
            dl = torch.empty((n, (V + 7) // 8 * 8), dtype=BF16, device=dev) if need_grad else None
            tv = token_values[f] if token_values is not None else None
            if emb == 128 and V <= 256:
                # logits stay in tensor memory: GEMM + masked CE + gradient rows (+ evaluator sums) in one kernel
                K.head_ce(e[:, f * emb:(f + 1) * emb], table16[offs[f]:offs[f] + V], labels[:, f], loss_sum[f:f + 1], count[f:f + 1],
                          dl, None, ignore_index, token_values=tv, stats=None if stats_buf is None else stats_buf[f])
            else:
                logits = K.gemm(e[:, f * emb:(f + 1) * emb], table16[offs[f]:offs[f] + V], out_dtype=F32)
                K.ce_rows(logits, labels[:, f], V, loss_sum[f:f + 1], count[f:f + 1], dl, None, ignore_index)
                if stats_buf is not None:
                    stats_buf[f] = _eval_stats_from_logits(logits[:, :V], labels[:, f], tv, ignore_index)
            dlogits[f] = dl
        active = count > 0
        per_field = loss_sum / count.clamp(min=1.0)
        n_active = active.sum().clamp(min=1)
        loss = (per_field * active).sum() / n_active
        ctx.saved = (h16, wp16, e_raw, e, mean, rstd, ln_w, table16, dlogits, count, active, n_active)
        ctx.params = (proj_w, ln_w, ln_b)
        ctx.meta = (sizes, fields, emb, offs, hidden.dtype)
        if stats_buf is None:
            stats_buf = torch.zeros((0, 3), dtype=F32, device=dev)
        ctx.mark_non_differentiable(per_field, count, stats_buf)
        return loss, per_field, count, stats_buf

    @staticmethod
    def backward(ctx, g, _g1, _g2, _g3):
        h16, wp16, e_raw, e, mean, rstd, ln_w, table16, dlogits, count, active, n_active = ctx.saved
        sizes, fields, emb, offs, h_dtype = ctx.meta
        n = h16.shape[0]
        coef = (g * active.float() / (count.clamp(min=1.0) * n_active)).contiguous()       # [n_fields] device scalars
        de = torch.zeros_like(e)
        dtable = torch.zeros((sum(sizes), emb), dtype=F32, device=h16.device)
        for f in fields:
            V, dl = sizes[f], dlogits[f]
            a = dl[:, :V] if dl.shape[1] != V else dl
            K.gemm(a, table16[offs[f]:offs[f] + V], trans_b=True, out=de[:, f * emb:(f + 1) * emb], alpha=coef[f:f + 1])
            K.gemm(a, e[:, f * emb:(f + 1) * emb], trans_a=True, trans_b=True, out=dtable[offs[f]:offs[f] + V], split_k=0,
                   alpha=coef[f:f + 1])
        p_proj, p_lnw, p_lnb = ctx.params
        dln_w, d1 = vgrad(p_lnw)
        dln_b, d2 = vgrad(p_lnb)
        de_raw = K.layer_norm_bwd(de, e_raw, mean, rstd, ln_w, dx_dtype=BF16, dw=dln_w, db=dln_b)
        dproj = wgrad(p_proj, h16, de_raw) if p_proj.dim() == 2 and p_proj.is_contiguous() else \
            K.gemm(h16, de_raw, trans_a=True, trans_b=True, out_dtype=F32, split_k=0)             # [dim, F*emb]
        dh = K.gemm(de_raw, wp16, out_dtype=h_dtype)                                               # [n, dim]
        return dh, dproj, None if d1 else dln_w, None if d2 else dln_b, dtable, None, None, None, None, None, None


class UntiedHeadCEFn(torch.autograd.Function):
    """Per-field `nn.Linear(dim, V_f)` heads + masked cross-entropy, mean over the fields that carry labels
    (models/scoreperformer/embeddings.py:287-313 `lm` head, wrappers.py:45-59): the variant of recipes/.../ablation/no_io_tie.yaml.

    hidden [n, dim] fp32 / bf16; labels int64 [n, F]; fields = indices into the label columns, params = (weight [V_f, dim],
    bias [V_f]) per listed field.  Returns (loss, per-field losses [len(fields)], counts).  One GEMM + one CE-rows kernel per field
    (logits live for one field at a time); backward: dW_f = c_f dlogits^T h, db_f = c_f colsum(dlogits), dh = sum_f c_f dlogits W_f."""

    @staticmethod
    def forward(ctx, hidden, labels, ignore_index: int, fields: Tuple[int, ...], *params):
        dev = hidden.device
        n = hidden.shape[0]
        h16 = K.cast_bf16(hidden.contiguous()) if hidden.dtype == F32 else hidden.contiguous()
        nf = len(fields)
        acc = torch.zeros((2, nf), dtype=F32, device=dev)
        loss_sum, count = acc[0], acc[1]
        need_grad = any(ctx.needs_input_grad)
        dlogits, w16s = [], []
        for i, f in enumerate(fields):
            W, b = params[2 * i], params[2 * i + 1]
            V = W.shape[0]
            w_16 = w16(W)
            logits = K.gemm(h16, w_16, bias=b.detach().float().contiguous(), out_dtype=F32)                 # [n, V]
            dl = torch.empty((n, (V + 7) // 8 * 8), dtype=BF16, device=dev) if need_grad else None
            K.ce_rows(logits, labels[:, f], V, loss_sum[i:i + 1], count[i:i + 1], dl, None, ignore_index)
            dlogits.append(dl)
            w16s.append(w_16)
        active = count > 0
        per_field = loss_sum / count.clamp(min=1.0)
        n_active = active.sum().clamp(min=1)
        loss = (per_field * active).sum() / n_active
        ctx.saved = (h16, dlogits, w16s, count, active, n_active)
        ctx.params, ctx.h_dtype = params, hidden.dtype
        ctx.mark_non_differentiable(per_field, count)
        return loss, per_field, count

    @staticmethod
    def backward(ctx, g, _g1, _g2):
        h16, dlogits, w16s, count, active, n_active = ctx.saved
        params = ctx.params
        coef = (g * active.float() / (count.clamp(min=1.0) * n_active)).contiguous()
        dh = torch.zeros((h16.shape[0], h16.shape[1]), dtype=F32, device=h16.device)
        grads = []
        for i, dl in enumerate(dlogits):
            W, b = params[2 * i], params[2 * i + 1]
            V = W.shape[0]
            a = dl[:, :V] if dl.shape[1] != V else dl
            grads.append(wgrad(W, a, h16, alpha=coef[i:i + 1]))                                             # [V, dim]
            db, direct = vgrad(b)
            cs = K.colsum(a) * coef[i]
            if direct:
                db.add_(cs)
                grads.append(None)
            else:
                grads.append(cs)
            K.gemm(a, w16s[i], trans_b=True, out=dh, accumulate=True, alpha=coef[i:i + 1])                 # dh += c dlogits W
        if ctx.h_dtype != F32:
            dh = dh.to(ctx.h_dtype)
        return (dh, None, None, None) + tuple(grads)


def tied_head_logits(hidden: Tensor, proj_w: Tensor, ln_w: Tensor, ln_b: Tensor, table: Tensor, sizes: Sequence[int],
                     fields: Sequence[int], emb: int) -> List[Tensor]:
    """Inference-side logits (fp32 [n, V_f] per requested field); no autograd."""
    with torch.no_grad():
        h16 = K.cast_bf16(hidden.contiguous()) if hidden.dtype == F32 else hidden.contiguous()
        e_raw = K.gemm(h16, K.cast_bf16(proj_w.contiguous()), trans_b=True, out_dtype=F32)
        e, _, _ = K.layer_norm_fwd(e_raw, ln_w, ln_b, out_dtype=BF16, need_stats=False)
        table16 = K.cast_bf16(table.contiguous())
        offs = [0]
        for v in sizes[:-1]:
            offs.append(offs[-1] + v)
        return [K.gemm(e[:, f * emb:(f + 1) * emb], table16[offs[f]:offs[f] + sizes[f]], out_dtype=F32) for f in fields]


# ----------------------------------------------------------------------------- classifier heads (a11)
class ClassifierHeadsFn(torch.autograd.Function):
    """loss_weight * mean_g weightedCE(Linear_g(dropout(x[rowmask])), labels[rowmask, g])  (models/classifiers/model.py:202-223).

    x fp32 [n, in_dim] is treated as detached (detach_inputs: true in every recipe); W/bias are the concatenated heads.
    Returns (loss, per_head_loss [n_heads])."""

    @staticmethod
    def forward(ctx, x, rowmask, labels, W, bias, class_w, n_classes: Tuple[int, ...], dropout_p: float, seed: int, loss_weight: float):
        x = x.detach().contiguous()
        W, bias = W.contiguous(), bias.contiguous()
        g = len(n_classes)
        num = torch.zeros(g, dtype=F32, device=x.device)
        den = torch.zeros(g, dtype=F32, device=x.device)
        K.clf_heads(x, rowmask, labels, W, bias, class_w, n_classes, dropout_p, seed, num=num, den=den)
        per_head = num / den.clamp(min=1e-20)
        loss = loss_weight * per_head.sum() / g
        ctx.saved = (x, rowmask, labels, W, bias, class_w, den)
        ctx.meta = (n_classes, dropout_p, seed, loss_weight)
        ctx.mark_non_differentiable(per_head)
        return loss, per_head

    @staticmethod
    def backward(ctx, gl, _g):
        x, rowmask, labels, W, bias, class_w, den = ctx.saved
        n_classes, dropout_p, seed, loss_weight = ctx.meta
        scale = (gl * loss_weight / len(n_classes)) / den.clamp(min=1e-20)
        dW, db = torch.zeros_like(W), torch.zeros_like(bias)
        K.clf_heads(x, rowmask, labels, W, bias, class_w, n_classes, dropout_p, seed, dlogit_scale=scale.contiguous(), dW=dW, db=db)
        return None, None, None, dW, db, None, None, None, None, None
