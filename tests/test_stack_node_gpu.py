"""The transformer-stack training node (`fused.TransformerStackFn`) against a float64 statement of the stack.

`stack_statement` is the pre-norm ('a', 'f') x depth stack + final norm of `oracle/model_oracle.transformer_stack` (with its
`attention`, `_norm` and `feed_forward`), written over the node's flat parameter list and evaluated in float64 with autograd.
The CPU tests pin it to the oracle, forward and backward, for the three stack kinds of the default model.  The GPU tests run
the node with the modules' parameters and a random output gradient on every row (padded rows included), in both gradient
modes: plain autograd, and the configuration TrainStep runs it in (flat fp32 gradient buffer written in place, bf16 weight
shadow, `DIRECT_GRAD` / `SHADOW_ACTIVE`, `STACK_BACKWARD_DONE`).  They also record every kernel call the node makes and compare
each with a float64 statement of that one operation on its recorded inputs, so a wrong slice, stride, mask or norm index shows
at its call site instead of being diluted over ~40 chained GEMMs.

With `rounded=True` the statement rounds to bf16 exactly where the node stores bf16 in HBM.  Forward: the style rows and the
weight copies; the AdaLN terms gb = bf16(style Wada^T + (b - 1)) (gamma - 1 is rounded, not gamma); every norm output xn; qkv;
the attention output o; and h = GLU(u), evaluated from the fp32 u that the fused feed-forward kernel keeps in tensor memory.
Backward: the output gradient g16; the bf16 copy of every residual gradient that feeds a sub-layer (row-masked in front of an
attention sub-layer); dO, whose row sums delta = rowsum(dO o) are taken from the fp32 dO before it is rounded; dqkv; du (the
GLU derivative is evaluated at the saved bf16 u; db1 sums the fp32 du); every dxn; and the AdaLN gradient dgb.

Left out of the rounded statement, so they are part of what the tight bars allow:
- the on-chip roundings of attention: P before P.V in the forward, P and dS in the backward (bf16 tensor-core operands);
- `tanh.approx.f32` in the SiLU of both feed-forward kernels;
- the order of fp32 sums (split-K, atomics, warp reductions), and the bf16 roundings that these flip.
"""
import copy
import inspect
import math

import pytest
import torch
import torch.nn.functional as F

from tests import parity
import model_oracle as mo

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64
STACKS = {"score_enc": "score_encoder.transformer", "perf_enc": "perf_encoder.transformer",
          "decoder": "perf_decoder.model.transformer"}
FILL = -torch.finfo(F64).max // 2           # the oracle's additive mask fill (attend.py:102-108)


def _bf(t):
    return t.to(BF16).to(t.dtype)


def rel_err(got, want):
    """max |got - want| / max |want|, in float64."""
    got, want = got.detach().double(), want.detach().double()
    return float((got - want).abs().max() / want.abs().max().clamp(min=1e-300))


def cos_dist(got, want):
    got, want = got.detach().double().flatten(), want.detach().double().flatten()
    return float(1 - torch.dot(got, want) / (got.norm() * want.norm()).clamp(min=1e-300))


def norm_ratio(got, want):
    """| ||got|| / ||want|| - 1 |: the scale error that the cosine distance cannot see."""
    return abs(float(got.detach().double().norm() / want.detach().double().norm().clamp(min=1e-300)) - 1.0)


# ------------------------------------------------------------------ the float64 statement
class _RoundGrad(torch.autograd.Function):
    """Identity in the forward; rounds the incoming gradient to bf16 (a gradient the node stores as bf16)."""

    @staticmethod
    def forward(ctx, t):
        return t.clone()

    @staticmethod
    def backward(ctx, g):
        return _bf(g)


def _rf(t):
    """Rounded to bf16 in the forward, gradient passed through unchanged (a value the node stores as bf16)."""
    return t + (_bf(t) - t).detach()


def _rg(t):
    return _RoundGrad.apply(t)


def _ident(t):
    return t


def _allowed(mask, T, causal, dev, diag=True):
    """[b, 1, T, T] keys each query may attend to: key padding, and j <= i when causal (j < i without `diag`)."""
    ok = torch.ones(mask.shape[0], 1, T, T, dtype=torch.bool, device=dev)
    if mask is not None:
        ok = ok & mask[:, None, None, :].bool()
    if causal:
        ok = ok & torch.ones(T, T, dtype=torch.bool, device=dev).tril(0 if diag else -1)
    return ok


def _chunks(B, H, T):
    """Samples per float64 attention chunk: keeps the [b, H, T, T] score tensors near 2^25 elements."""
    return max(1, (1 << 25) // (H * T * T))


class _Attention(torch.autograd.Function):
    """MQA + learned ALiBi over qkv [B, T, H*64 + 128] (q heads | k | v), modules/transformer/attend.py:58-126.

    Forward: o [B, T, H*64], rounded to bf16 when `rounded`.  Backward, as csrc/attention_bwd_tc.cu with delta from
    spb_gemm_bf16_rowdot: dP = dO16 v^T with dO16 = bf16(dO), delta = rowsum(dO o) from the fp32 dO and the stored o, and
    dS = P (dP - delta).  Without `rounded` this is the exact gradient.  P is recomputed chunk by chunk of samples."""

    @staticmethod
    def forward(ctx, qkv, ls, mask, H, causal, rounded, diag):
        B, T, _ = qkv.shape
        o = torch.empty(B, T, H * 64, dtype=qkv.dtype, device=qkv.device)
        for b0 in range(0, B, _chunks(B, H, T)):
            sl = slice(b0, b0 + _chunks(B, H, T))
            p, _, _, v = _Attention._probs(qkv[sl], ls, None if mask is None else mask[sl], H, causal, diag)
            o[sl] = torch.einsum("bhij,bjd->bihd", p, v).reshape(p.shape[0], T, H * 64)
        if rounded:
            o = _bf(o)
        ctx.save_for_backward(qkv, ls, o)
        ctx.meta = (mask, H, causal, rounded, diag)
        return o

    @staticmethod
    def _probs(qkv, ls, mask, H, causal, diag):
        b, T, _ = qkv.shape
        q = qkv[..., :H * 64].reshape(b, T, H, 64).transpose(1, 2)
        k, v = qkv[..., H * 64:H * 64 + 64], qkv[..., H * 64 + 64:]
        pos = torch.arange(T, device=qkv.device)
        dist = (pos[None, :] - pos[:, None]).abs().to(qkv.dtype)
        s = torch.einsum("bhid,bjd->bhij", q, k) * 0.125 - ls.reshape(-1).exp()[None, :, None, None] * dist
        ok = _allowed(mask if mask is not None else torch.ones(b, T, dtype=torch.bool, device=qkv.device), T, causal,
                      qkv.device, diag)
        return s.masked_fill(~ok, FILL).softmax(dim=-1), q, k, v

    @staticmethod
    def backward(ctx, do):
        qkv, ls, o = ctx.saved_tensors
        mask, H, causal, rounded, diag = ctx.meta
        B, T, _ = qkv.shape
        delta = (do * o).reshape(B, T, H, 64).sum(-1).transpose(1, 2)                   # [B, H, T]
        dqkv, dls = attention_grads(qkv, ls, mask, H, causal, _bf(do) if rounded else do, delta, diag)
        return dqkv, dls.view_as(ls), None, None, None, None, None


def attention_grads(qkv, ls, mask, H, causal, do, delta, diag=True):
    """dqkv [B, T, H*64 + 128] and dlogslopes [H] of _Attention from dO [B, T, H*64] and delta [B, H, T]."""
    B, T, _ = qkv.shape
    dqkv = torch.zeros_like(qkv)
    dls = torch.zeros(H, dtype=qkv.dtype, device=qkv.device)
    pos = torch.arange(T, device=qkv.device)
    dist = (pos[None, :] - pos[:, None]).abs().to(qkv.dtype)
    for b0 in range(0, B, _chunks(B, H, T)):
        sl = slice(b0, b0 + _chunks(B, H, T))
        p, q, k, v = _Attention._probs(qkv[sl], ls, None if mask is None else mask[sl], H, causal, diag)
        b = p.shape[0]
        dOh = do[sl].reshape(b, T, H, 64).transpose(1, 2)
        dp = torch.einsum("bhid,bjd->bhij", dOh, v)
        ds = p * (dp - delta[sl][..., None])
        dqkv[sl, :, :H * 64] = (torch.einsum("bhij,bjd->bihd", ds, k) * 0.125).reshape(b, T, H * 64)
        dqkv[sl, :, H * 64:H * 64 + 64] = torch.einsum("bhij,bhid->bjd", ds, q) * 0.125
        dqkv[sl, :, H * 64 + 64:] = torch.einsum("bhij,bhid->bjd", p, dOh)
        dls -= (ds * dist).sum(dim=(0, 2, 3)) * ls.reshape(-1).exp()
    return dqkv, dls


class _GLU(torch.autograd.Function):
    """value * silu(gate) of u = [value | gate] (modules/transformer/feedforward.py:13-22).  The backward evaluates the
    derivative at bf16(u) when `at_bf16_u`: the saved pre-activation that csrc/ffn_bwd.cu reads."""

    @staticmethod
    def forward(ctx, u, at_bf16_u):
        ctx.save_for_backward(u)
        ctx.at_bf16_u = at_bf16_u
        a, g = u.chunk(2, dim=-1)
        return a * F.silu(g)

    @staticmethod
    def backward(ctx, dh):
        (u,) = ctx.saved_tensors
        a, g = (_bf(u) if ctx.at_bf16_u else u).chunk(2, dim=-1)
        sig = torch.sigmoid(g)
        silu = g * sig
        return torch.cat([dh * silu, dh * a * (sig + silu * (1 - sig))], dim=-1), None


def norm_index(spec, i_norm):
    """Index into the node's flat parameter list of the first tensor of norm number i_norm (fused._norm_index)."""
    if i_norm == 2 * spec.depth:
        return spec.depth * 12
    l, is_ff = divmod(i_norm, 2)
    return l * 12 + (7 if is_ff else 0)


def stack_statement(spec, params, x, mask, style, rounded, mutation=None):
    """float64 stack over the node's flat parameter list `params` (per layer: norm a, norm b, to_q, to_k, to_v, to_out,
    logslopes, norm a, norm b, proj_w, proj_b, out_w; then the final norm).  x [B, T, D], mask bool [B, T] or None, style
    [B, T, S] or None.  Returns (out [B, T, D], hiddens [depth, B, T, D], kvs [depth, B, T, 128]).

    `mutation` names a deliberately wrong statement, for the resolution test: "no_attn_mask" (the attention branch is not
    row-masked), "ada_neighbour" (norm 1 reads the AdaLN slice of norm 2), "causal_no_diag" (a causal query does not see its
    own key), "glu_fp32_u" (GLU' at the fp32 u instead of the saved bf16 u)."""
    rf, rg = (_rf, _rg) if rounded else (_ident, _ident)
    B, T, D = x.shape
    H = spec.heads
    m = torch.ones(B, T, 1, dtype=x.dtype, device=x.device) if mask is None else mask[..., None].to(x.dtype)
    gb_all = None
    if spec.ada:
        nw = torch.cat([params[norm_index(spec, i)] for i in range(spec.n_norms)])
        nb = torch.cat([params[norm_index(spec, i) + 1] for i in range(spec.n_norms)])
        ones = torch.cat([torch.ones(D), torch.zeros(D)]).to(nb).repeat(spec.n_norms)
        gb_all = rg(rf(rf(style) @ rf(nw).t() + (nb - ones)))

    def norm(i, xin):
        if spec.ada:
            k = i + 1 if (mutation == "ada_neighbour" and i == 1) else i
            gb = gb_all[..., k * 2 * D:(k + 1) * 2 * D]
            return F.layer_norm(xin, (D,), eps=spec.eps) * (1 + gb[..., :D]) + gb[..., D:]
        j = norm_index(spec, i)
        return F.layer_norm(xin, (D,), params[j], params[j + 1], spec.eps)

    cur, hiddens, kvs = x, [], []
    for l in range(spec.depth):
        to_q, to_k, to_v, to_out, ls, = params[12 * l + 2:12 * l + 7]
        w1, b1, w2 = params[12 * l + 9:12 * l + 12]
        hiddens.append(cur)
        xn = rg(rf(norm(2 * l, cur)))
        qkv = rg(rf(xn @ rf(torch.cat([to_q, to_k, to_v])).t()))
        kvs.append(qkv[..., H * 64:])
        o = _Attention.apply(qkv, ls, mask, H, spec.causal, rounded, mutation != "causal_no_diag")
        y = o @ rf(to_out).t()
        cur = cur + rg(y if mutation == "no_attn_mask" else y * m)
        xn = rg(rf(norm(2 * l + 1, cur)))
        u = rg(xn @ rf(w1).t()) + b1                  # db1 sums the fp32 du, dW1 and dxn read the bf16 du
        h = rf(_GLU.apply(u, rounded and mutation != "glu_fp32_u"))
        cur = cur + rg(h @ rf(w2).t())
    out = rg(norm(2 * spec.depth, cur))
    return out, torch.stack(hiddens), torch.stack(kvs)


def statement_grads(spec, params, x, mask, style, g_out, rounded, mutation=None):
    """Forward + backward of the statement on float64 leaf copies of (params, x, style).  Returns a dict name -> tensor:
    out, hiddens, kvs, dx, dstyle (AdaLN only) and p<i> for every flat parameter i."""
    leaves = [p.detach().double().requires_grad_() for p in params]
    xd = x.detach().double().requires_grad_()
    sd = style.detach().double().requires_grad_() if style is not None else None
    out, hid, kv = stack_statement(spec, leaves, xd, mask, sd, rounded, mutation)
    inputs = leaves + [xd] + ([sd] if sd is not None else [])
    grads = torch.autograd.grad(out, inputs, g_out.double())
    res = {"out": out.detach(), "hiddens": hid.detach(), "kvs": kv.detach(), "dx": grads[len(leaves)]}
    if sd is not None:
        res["dstyle"] = grads[-1]
    for i in range(len(leaves)):
        res[f"p{i}"] = grads[i]
    return res


# ------------------------------------------------------------------ the stacks of the default model
@pytest.fixture(scope="module")
def cpu_model():
    return parity.build_model(dropout=False, device="cpu")


def stack_of(model, kind):
    mod = model.get_submodule(STACKS[kind])
    return mod, mod.stack_spec(return_hiddens=True)


def param_labels(mod):
    """Readable name of every flat parameter: the module's parameter name with the layer number replaced by '*'."""
    names = {id(p): n for n, p in mod.named_parameters()}
    out = []
    for p in mod.flat_params():
        parts = names[id(p)].split(".")
        if parts[0] == "layers":
            parts[1] = "*"
        out.append(".".join(parts))
    return out


def ragged_mask(B, T, dev, seed):
    """Sample 0 complete; sample 1 padded at the end; from sample 2 on holes everywhere, position 0 among them."""
    g = torch.Generator().manual_seed(seed)
    m = torch.rand(B, T, generator=g) > 0.25
    m[0] = True
    if B > 1:
        m[1] = True
        m[1, T - T // 3:] = False
    if B > 2:
        m[2, 0] = False
    m[:, T // 2] = True                           # every sample keeps at least one valid position (DESIGN section 4)
    return m.to(dev)


def make_inputs(spec, B, T, masked, dev, seed, style_dim):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, spec.dim, generator=g).to(dev)
    style = (0.5 * torch.randn(B, T, style_dim, generator=g)).to(dev) if spec.ada else None
    g_out = torch.randn(B, T, spec.dim, generator=g).to(dev)
    mask = ragged_mask(B, T, dev, seed) if masked else None
    return x, mask, style, g_out


# ------------------------------------------------------------------ CPU: the statement against the oracle
@pytest.mark.parametrize("kind", list(STACKS))
def test_statement_matches_oracle_stack(cpu_model, kind):
    """The plain statement (with its hand-written attention and GLU backward) equals oracle.transformer_stack in float64:
    output, hiddens, k|v and the gradients of x, style and every parameter, on a ragged mask (holes, a padded tail, position
    0 padded).  The bound only has to separate reordered float64 sums (~1e-15) from a different statement (>= 1e-8)."""
    mod, spec = stack_of(cpu_model, kind)
    names = {id(p): n for n, p in mod.named_parameters()}
    leaves = {n: p.detach().double().requires_grad_() for n, p in mod.named_parameters()}
    flat = [leaves[names[id(p)]] for p in mod.flat_params()]
    sd = {f"t.{n}": t for n, t in leaves.items()}
    ospec = parity.oracle_spec(cpu_model)
    B, T = 3, 19
    x, mask, style, g_out = make_inputs(spec, B, T, True, "cpu", 11, ospec.style_dim)
    x, g_out = x.double().requires_grad_(), g_out.double()
    style = style.double().requires_grad_() if style is not None else None
    want, w_hid, w_kv = mo.transformer_stack(sd, "t", x, mask, spec.depth, spec.causal, ospec, style=style)
    got, g_hid, g_kv = stack_statement(spec, flat, x, mask, style, rounded=False)
    assert rel_err(got, want) < 1e-12
    for l in range(spec.depth):
        assert rel_err(g_hid[l], w_hid[l]) < 1e-12, l
        assert rel_err(g_kv[l], torch.cat(w_kv[l], dim=-1)) < 1e-12, l
    inputs = [x] + ([style] if style is not None else []) + list(leaves.values())
    g_want = torch.autograd.grad(want, inputs, g_out)
    g_got = torch.autograd.grad(got, inputs, g_out)
    labels = ["x"] + (["style"] if style is not None else []) + list(leaves)
    for name, a, b in zip(labels, g_got, g_want):
        assert rel_err(a, b) < 1e-12, name


def test_rounded_statement_rounds_where_stated(cpu_model):
    """The rounded statement stays within bf16 storage noise of the plain one, and it is not the plain one: its kvs are
    bf16 values and its gradients differ from the exact ones."""
    mod, spec = stack_of(cpu_model, "decoder")
    params = list(mod.flat_params())
    x, mask, style, g_out = make_inputs(spec, 2, 13, True, "cpu", 3, parity.oracle_spec(cpu_model).style_dim)
    r = statement_grads(spec, params, x, mask, style, g_out, rounded=True)
    p = statement_grads(spec, params, x, mask, style, g_out, rounded=False)
    assert torch.equal(r["kvs"], _bf(r["kvs"]))
    for name in ("out", "dx", "dstyle", "p2"):
        assert 1e-6 < rel_err(r[name], p[name]) < 5e-2, name


# ------------------------------------------------------------------ GPU: the node against the statement
# Bars, per tensor: (rel, cos, ratio) against the rounded statement (TIGHT), then against the plain one (LOOSE).  rel_err is a
# max-abs statistic, set by single flipped bf16 roundings of large elements; the cosine distance sees the whole tensor; the norm
# ratio | |got| / |want| - 1 | sees a wrong scale, which the cosine distance cannot.  Each bar is the largest value measured
# on a B200 (1000 W) over every case and both gradient modes of this file in three runs (the comment beside it: tight |
# loose), times 1.5 (rel) or 2 (cos, ratio), rounded up.  The encoders' final LayerNorm bias gradient is the column sum of
# g16, which the rounded statement mirrors exactly: its tight bars only leave room for the order of the fp32 atomics.
#
# Why the gradient cosine bars sit near 1e-4 and not near 1e-5: every single kernel call agrees with its own float64 statement
# to bf16 storage (cos <= 2.8e-6, test_every_kernel_call_matches_its_statement), but end to end the node and the rounded
# statement stop rounding the same values as soon as one unmirrored rounding (P and dS in attention, tanh.approx) or one
# reordered fp32 sum flips a bf16 rounding; from there on each side rounds its own values, so after four layers the rounded
# statement is only about twice as close as the plain one.  The logslopes gradient (4 values per layer) is a sum over every
# score of dS |i - j| that the kernel forms as sum(P dP |i - j|) - sum(delta E[|i - j|]): it cancels to a small fraction of
# its terms, so its bf16 dS noise shows at the percent level (1.1e-2 rel already within one call).  LayerNorm bias and
# AdaLN bias gradients are column sums of the bf16 dxn with the same kind of cancellation, hence their larger norm ratios.
# Even so, a 1e-3 scale error of a large gradient (proj_w, out_w, to_out, ffn bias, ...) breaks its ratio bar, and a wrong
# mask, slice or causal diagonal breaks the bars by orders of magnitude (test_bars_separate_mutated_statements).
BARS = {    # label: (tight rel, cos, ratio, loose rel, cos, ratio)   # measured tight rel cos ratio | loose rel cos ratio
    "out": (1.2e-2, 3.2e-5, 3.4e-5, 1.9e-2, 7.1e-5, 3.9e-5),                        # 7.8e-03 1.6e-05 1.7e-05 | 1.3e-02 3.5e-05 1.9e-05
    "hiddens": (9.1e-3, 1.8e-5, 5.0e-5, 1.4e-2, 4.5e-5, 1.7e-4),                    # 6.0e-03 8.8e-06 2.5e-05 | 9.3e-03 2.2e-05 8.3e-05
    "kvs": (8.9e-3, 1.8e-5, 8.7e-5, 1.6e-2, 3.9e-5, 9.9e-5),                        # 5.9e-03 9.0e-06 4.4e-05 | 1.0e-02 1.9e-05 4.9e-05
    "dx": (2.4e-2, 1.5e-4, 1.1e-3, 3.1e-2, 2.6e-4, 1.6e-3),                         # 1.5e-02 7.3e-05 5.5e-04 | 2.0e-02 1.3e-04 7.8e-04
    "dstyle": (2.1e-2, 1.4e-4, 2.5e-4, 3.0e-2, 2.4e-4, 2.9e-4),                     # 1.4e-02 6.8e-05 1.3e-04 | 2.0e-02 1.2e-04 1.4e-04
    "layers.*.0.0.weight": (1.9e-2, 1.2e-4, 2.6e-3, 2.0e-2, 1.4e-4, 3.7e-3),        # 1.3e-02 5.8e-05 1.3e-03 | 1.3e-02 6.8e-05 1.8e-03
    "layers.*.0.0.bias": (1.7e-2, 6.8e-5, 4.2e-3, 2.2e-2, 1.1e-4, 5.4e-3),          # 1.1e-02 3.4e-05 2.1e-03 | 1.5e-02 5.4e-05 2.7e-03
    "layers.*.0.0.linear.weight": (2.7e-2, 2.2e-4, 1.8e-3, 3.6e-2, 3.6e-4, 2.1e-3), # 1.8e-02 1.1e-04 8.6e-04 | 2.4e-02 1.8e-04 1.0e-03
    "layers.*.0.0.linear.bias": (2.4e-2, 1.7e-4, 2.9e-3, 3.0e-2, 3.1e-4, 4.4e-3),   # 1.6e-02 8.0e-05 1.4e-03 | 2.0e-02 1.5e-04 2.2e-03
    "layers.*.1.to_q.weight": (2.5e-2, 2.5e-4, 1.8e-3, 3.2e-2, 4.4e-4, 2.5e-3),     # 1.6e-02 1.2e-04 8.5e-04 | 2.1e-02 2.2e-04 1.2e-03
    "layers.*.1.to_k.weight": (2.7e-2, 2.6e-4, 2.0e-3, 3.9e-2, 4.5e-4, 2.6e-3),     # 1.7e-02 1.3e-04 9.8e-04 | 2.6e-02 2.2e-04 1.3e-03
    "layers.*.1.to_v.weight": (2.1e-2, 1.6e-4, 1.5e-3, 2.9e-2, 2.8e-4, 1.3e-3),     # 1.4e-02 7.8e-05 7.3e-04 | 1.9e-02 1.4e-04 6.1e-04
    "layers.*.1.to_out.weight": (2.1e-2, 1.5e-4, 7.0e-4, 2.9e-2, 2.7e-4, 1.0e-3),   # 1.4e-02 7.3e-05 3.5e-04 | 1.9e-02 1.3e-04 5.0e-04
    "layers.*.1.rel_pos.learned_logslopes": (1.3e-1, 4.1e-3, 5.8e-2, 1.2e-1, 2.6e-3, 9.6e-2),  # 8.4e-02 2.0e-03 2.9e-02 | 7.5e-02 1.3e-03 4.8e-02
    "layers.*.1.ff.0.proj.weight": (2.0e-2, 1.4e-4, 4.5e-4, 3.1e-2, 2.5e-4, 5.7e-4),  # 1.3e-02 6.7e-05 2.2e-04 | 2.0e-02 1.2e-04 2.8e-04
    "layers.*.1.ff.0.proj.bias": (1.9e-2, 1.3e-4, 9.0e-4, 2.5e-2, 2.1e-4, 2.0e-3),    # 1.3e-02 6.4e-05 4.5e-04 | 1.6e-02 1.1e-04 9.5e-04
    "layers.*.1.ff.3.weight": (2.0e-2, 1.3e-4, 3.7e-4, 2.3e-2, 2.4e-4, 5.1e-4),       # 1.3e-02 6.3e-05 1.8e-04 | 1.5e-02 1.2e-04 2.5e-04
    "final_norm.weight": (6.8e-3, 1.6e-5, 9.0e-4, 1.1e-2, 3.2e-5, 1.6e-3),            # 4.5e-03 7.6e-06 4.5e-04 | 7.3e-03 1.6e-05 8.0e-04
    "final_norm.bias": (2.0e-6, 2.0e-13, 2.0e-7, 3.2e-3, 3.4e-6, 2.5e-4),             # 9.7e-07 5.9e-14 8.7e-08 | 2.1e-03 1.7e-06 1.2e-04
    "final_norm.linear.weight": (1.1e-2, 2.3e-5, 8.5e-5, 1.8e-2, 4.9e-5, 1.7e-4),     # 7.2e-03 1.1e-05 4.2e-05 | 1.2e-02 2.4e-05 8.2e-05
    "final_norm.linear.bias": (9.4e-3, 2.3e-5, 9.2e-4, 1.5e-2, 4.5e-5, 7.4e-4),       # 6.3e-03 1.1e-05 4.6e-04 | 1.0e-02 2.3e-05 3.7e-04
}
WORST = {}


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        print("\nworst over the cases run (statement, tensor): rel / cos / ratio")
        for key in sorted(WORST):
            v = WORST[key]
            print(f"  {key[0]:5s} {key[1]:34s} {v['rel']:.2e} {v['cos']:.2e} {v['ratio']:.2e}")


@pytest.fixture(scope="module")
def gpu_model():
    return parity.build_model(dropout=False, device="cuda")


@pytest.fixture(scope="module")
def K():
    from scoreperformer_b200 import kernels
    return kernels


def run_node(spec, params, x, mask, style, g_out):
    """The node with return_hiddens, backward with g_out.  Returns (out, hiddens, kvs, dx, dstyle); parameter gradients are
    left where autograd or the direct-gradient kernels put them."""
    from scoreperformer_b200 import fused
    xr = x.clone().requires_grad_()
    sr = style.clone().requires_grad_() if style is not None else None
    out, hid, kv = fused.TransformerStackFn.apply(spec, xr, mask, sr, (0,) * (2 * spec.depth), *params)
    torch.autograd.backward(out, g_out)
    torch.cuda.synchronize()
    return out.detach(), hid, kv, xr.grad, None if sr is None else sr.grad


def node_results(spec, out, hid, kv, dx, dstyle, grads):
    B, T, D = out.shape
    res = {"out": out, "hiddens": hid, "kvs": kv.view(spec.depth, B, T, -1), "dx": dx}
    if dstyle is not None:
        res["dstyle"] = dstyle
    for i, g in enumerate(grads):
        res[f"p{i}"] = g
    return res


def compare(got, want, labels, which, record=True):
    """Every tensor of `got` against `want` with the bars of statement `which`; returns the violations."""
    bad = []
    for name, g in got.items():
        w = want[name]
        label = labels[int(name[1:])] if name.startswith("p") else name
        assert g is not None and torch.isfinite(g).all(), (which, label)
        if float(w.abs().max()) == 0.0:
            if float(g.abs().max()) != 0.0:
                bad.append(f"{which} {label}: want exactly zero, got {float(g.abs().max()):.2e}")
            continue
        st = dict(rel=rel_err(g, w), cos=cos_dist(g, w), ratio=norm_ratio(g, w))
        if record:
            cur = WORST.setdefault((which, label), dict(rel=0.0, cos=0.0, ratio=0.0))
            for s, v in st.items():
                cur[s] = max(cur[s], v)
        bars = dict(zip(("rel", "cos", "ratio"), BARS[label][:3] if which == "tight" else BARS[label][3:]))
        for s, v in st.items():
            if not v < bars[s]:
                bad.append(f"{which} {label}: {s} {v:.2e} >= {bars[s]:.1e}")
    return bad


def _cuda_stack(gpu_model, kind):
    mod = copy.deepcopy(gpu_model.get_submodule(STACKS[kind]))
    mod.train()
    return mod, mod.stack_spec(return_hiddens=True)


class _Host(torch.nn.Module):
    """A stack between two other parameters, so that TrainStep's flat buffers hold gradient slots the stack does not own."""

    def __init__(self, stack):
        super().__init__()
        self.pre = torch.nn.Parameter(torch.randn(13, device="cuda"))
        self.stack = stack
        self.post = torch.nn.Parameter(torch.randn(3, 5, device="cuda"))


def run_direct(K, mod, spec, x, mask, style, g_out, plain_grads):
    """The node in TrainStep's configuration: parameters and gradients are views of flat fp32 buffers (offsets padded to 8),
    forward GEMMs read the bf16 shadow, weight gradients accumulate into the buffer.  The buffer is pre-filled with random
    values (per slot at the scale of that parameter's gradient).  Returns (results like node_results with every gradient
    minus its pre-fill, prefill, flat gradient after backward, the clone taken in STACK_BACKWARD_DONE, callback count, owned
    mask of the flat buffer)."""
    from scoreperformer_b200 import fused
    from scoreperformer_b200.train_step import TrainStep
    host = _Host(mod)
    rng_offset = K.RNG_OFFSET
    ts = TrainStep(host, lr=0.0, grad_clip=None, use_graph=False)
    K.RNG_OFFSET = rng_offset
    flat = list(mod.flat_params())
    offs = {id(p): off for p, off in zip(ts.params, ts.offsets)}
    g = torch.Generator(device="cuda").manual_seed(99)
    prefill = torch.randn(ts.flat_grad.numel(), device="cuda", generator=g)
    owned = torch.zeros_like(prefill, dtype=torch.bool)
    for p, pg in zip(flat, plain_grads):
        o = offs[id(p)]
        prefill[o:o + p.numel()] *= pg.float().pow(2).mean().sqrt()
        owned[o:o + p.numel()] = True
    ts.flat_grad.copy_(prefill)
    K.cast_bf16(ts.flat_param, out=ts.flat_shadow)
    calls = []

    def done(params):
        calls.append((list(params), ts.flat_grad.clone()))

    fused.DIRECT_GRAD = fused.SHADOW_ACTIVE = True
    fused.STACK_BACKWARD_DONE = done
    try:
        out, hid, kv, dx, dstyle = run_node(spec, flat, x, mask, style, g_out)
    finally:
        fused.DIRECT_GRAD = fused.SHADOW_ACTIVE = False
        fused.STACK_BACKWARD_DONE = None
    grads = [(ts.flat_grad[offs[id(p)]:offs[id(p)] + p.numel()] - prefill[offs[id(p)]:offs[id(p)] + p.numel()]).view_as(p)
             for p in flat]
    res = node_results(spec, out, hid, kv, dx, dstyle, grads)
    for p in flat:
        assert p.grad.data_ptr() == ts.flat_grad[offs[id(p)]:].data_ptr()      # autograd left the buffer views in place
    return res, prefill, ts.flat_grad.clone(), calls, owned, [offs[id(p)] for p in flat]


CASES = [                       # kind, B, T, masked
    ("score_enc", 3, 130, True), ("score_enc", 2, 47, True),
    ("perf_enc", 3, 130, True), ("perf_enc", 2, 47, True),
    ("decoder", 3, 130, True), ("decoder", 2, 47, True),
    ("decoder", 2, 64, False),
    ("decoder", 64, 512, True), ("decoder", 16, 2048, True), ("perf_enc", 64, 512, True),     # C2, C4: > 1 tile per SM
]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,B,T,masked", CASES)
def test_stack_node_matches_statement(gpu_model, K, kind, B, T, masked):
    """out, hiddens, k|v and the gradients of x, style and every parameter, in both gradient modes, against the rounded
    (tight) and the plain (loose) statement.  The TrainStep configuration must give pre-fill + plain-mode gradient to within
    fp32 rounding in every slot (accumulate, never overwrite), leave every slot the stack does not own untouched, and hand
    its gradients off exactly once, after the last write."""
    mod, spec = _cuda_stack(gpu_model, kind)
    labels = param_labels(mod)
    params = list(mod.flat_params())
    x, mask, style, g_out = make_inputs(spec, B, T, masked, "cuda", B * 1000 + T, 64)
    want = {w: statement_grads(spec, params, x, mask, style, g_out, rounded=(w == "tight")) for w in ("tight", "loose")}

    for p in params:
        p.grad = None
    out, hid, kv, dx, dstyle = run_node(spec, params, x, mask, style, g_out)
    plain = node_results(spec, out, hid, kv, dx, dstyle, [p.grad for p in params])
    bad = compare(plain, want["tight"], labels, "tight") + compare(plain, want["loose"], labels, "loose")

    direct, prefill, flat_after, calls, owned, offs = run_direct(K, mod, spec, x, mask, style, g_out,
                                                                 [plain[f"p{i}"] for i in range(len(params))])
    bad += compare(direct, want["tight"], labels, "tight") + compare(direct, want["loose"], labels, "loose")
    # the same forward from the shadow as from fresh casts.  The backward is not bit-reproducible at the full sizes: fp32
    # atomics (dQ accumulation, split-K weight gradients, bias column sums) add in varying order and a flipped bf16 rounding
    # propagates, so two runs differ at bf16 level (measured up to 4.9e-3 max-abs relative on dx at C2 / C4, 0 at the small
    # sizes).  Every slot must hold pre-fill + plain-mode gradient to within fp32 rounding plus that run-to-run noise (the
    # tensor's tight rel bar): a slot overwritten instead of accumulated is off by the whole pre-fill (~4 rms of its gradient),
    # one accumulated twice by the whole gradient.
    for name in ("out", "hiddens", "kvs"):
        assert rel_err(direct[name], plain[name]) < 1e-5, name
    for i, o in enumerate(offs):
        n = params[i].numel()
        pf, pg = prefill[o:o + n], plain[f"p{i}"].reshape(-1)
        err = float((flat_after[o:o + n] - (pf + pg)).abs().max())
        tol = 1e-5 * float(pf.abs().max() + pg.abs().max()) + BARS[labels[i]][0] * float(pg.abs().max())
        assert err <= tol, (labels[i], err, tol)
    assert torch.equal(flat_after[~owned], prefill[~owned]), "a gradient slot the stack does not own was written"
    assert len(calls) == 1, f"STACK_BACKWARD_DONE called {len(calls)} times"
    assert [id(p) for p in calls[0][0]] == [id(p) for p in params]
    assert torch.equal(calls[0][1], flat_after), "gradients were written after the bucket was handed off"
    print(f"stack node {kind} B={B} T={T} masked={masked}: {len(bad)} violations")
    assert not bad, "\n".join(bad)


# ------------------------------------------------------------------ GPU: resolution
MUTATIONS = ["no_attn_mask", "ada_neighbour", "causal_no_diag", "grad_scale", "glu_fp32_u"]


@pytest.fixture(scope="module")
def decoder_run(gpu_model):
    mod, spec = _cuda_stack(gpu_model, "decoder")
    params = list(mod.flat_params())
    x, mask, style, g_out = make_inputs(spec, 3, 130, True, "cuda", 3130, 64)
    for p in params:
        p.grad = None
    out, hid, kv, dx, dstyle = run_node(spec, params, x, mask, style, g_out)
    got = node_results(spec, out, hid, kv, dx, dstyle, [p.grad for p in params])
    return mod, spec, params, (x, mask, style, g_out), got


@pytest.mark.gpu
@pytest.mark.parametrize("mutation", MUTATIONS)
def test_bars_separate_mutated_statements(decoder_run, mutation):
    """The decoder kind's node results (3 x 130, ragged) against deliberately wrong rounded statements: each of these must
    break a tight bar, or the bars could not see that mistake in the node.  "grad_scale" scales one parameter gradient of
    the statement by 1 + 1e-3 (only the norm ratio can see it).  "glu_fp32_u" is the one rounding of the statement that
    is reported rather than required: the test prints whether the bars separate it and fails only for the others."""
    mod, spec, params, (x, mask, style, g_out), got = decoder_run
    labels = param_labels(mod)
    want = statement_grads(spec, params, x, mask, style, g_out, rounded=True,
                           mutation=None if mutation == "grad_scale" else mutation)
    if mutation == "grad_scale":
        want["p9"] = want["p9"] * (1 + 1e-3)                  # layer 0 proj_w
    bad = compare(got, want, labels, "tight", record=False)
    print(f"mutation {mutation}: {len(bad)} bars broken" + "".join(f"\n  {b}" for b in bad[:6]))
    if mutation != "glu_fp32_u":
        assert bad, f"the bars do not separate the mutation {mutation}"


# ------------------------------------------------------------------ GPU: every kernel call of the node on its own
SPIED = ["gemm", "gemm_rowdot", "layer_norm_fwd", "layer_norm_bwd", "attention_fwd", "attention_bwd", "ffn_fwd", "ffn_bwd",
         "colsum", "multi_add", "transpose_bf16"]


def _clone(v):
    if isinstance(v, torch.Tensor):
        return v.clone()
    if isinstance(v, (list, tuple)):
        return type(v)(_clone(e) for e in v)
    return v


def record_calls(K, monkeypatch):
    """Replace the kernels `fused` calls as K.<fn> with spies.  A spy clones the arguments before the call (ffn_bwd writes du
    over u; accumulate-into outputs change) and again after it, and clones what the call returned."""
    calls = []
    for name in SPIED:
        orig = getattr(K, name)
        sig = inspect.signature(orig)

        def spy(*a, _orig=orig, _sig=sig, _name=name, **kw):
            ba = _sig.bind(*a, **kw)
            ba.apply_defaults()
            before = {k: _clone(v) for k, v in ba.arguments.items()}
            ret = _orig(*a, **kw)
            after = {k: _clone(v) for k, v in ba.arguments.items()}
            calls.append((_name, before, after, _clone(ret)))
            return ret

        monkeypatch.setattr(K, name, spy)
    return calls


def _d(t):
    return None if t is None else t.double()


def _ln_gamma_beta(a, D):
    if a["gb"] is not None:
        gb = _d(a["gb"])
        return 1 + gb[:, :D], gb[:, D:]
    return _d(a["w"]), (_d(a["b"]) if "b" in a else None)


def call_statement(name, a, after, ret):
    """[(output label, got, want float64)] for one recorded kernel call (a: the arguments before the call)."""
    if name == "gemm":
        A = _d(a["a"]).t() if a["trans_a"] else _d(a["a"])
        Bm = _d(a["b"]).t() if a["trans_b"] else _d(a["b"])
        c = A @ Bm.t()
        if a["alpha"] is not None:
            c = c * _d(a["alpha"])
        if a["bias"] is not None:
            c = c + _d(a["bias"])
        if a["rowmask"] is not None:
            c = c * a["rowmask"].double()[:, None]
        if a["residual"] is not None:
            c = c + _d(a["residual"])
        if a["out"] is not None:
            if a["accumulate"]:
                c = c + _d(a["out"])
            return [("C", after["out"], c)]
        return [("C", ret, c)]
    if name == "gemm_rowdot":
        Bm = _d(a["b"]).t() if a["trans_b"] else _d(a["b"])
        c = _d(a["a"]) @ Bm.t()
        T, H = a["T"], a["H"]
        delta = (c * _d(a["x"])).view(-1, T, H, 64).sum(-1).transpose(1, 2)
        return [("C", ret[0], c), ("delta", ret[1], delta)]
    if name == "layer_norm_fwd":
        x = _d(a["x"])
        D = x.shape[1]
        mean = x.mean(-1, keepdim=True)
        rstd = ((x - mean).pow(2).mean(-1, keepdim=True) + a["eps"]).rsqrt()
        gam, bet = _ln_gamma_beta(a, D)
        return [("y", ret[0], (x - mean) * rstd * gam + bet), ("mean", ret[1], mean[:, 0]), ("rstd", ret[2], rstd[:, 0])]
    if name == "layer_norm_bwd":
        x, dy = _d(a["x"]), _d(a["dy"])
        D = x.shape[1]
        xh = (x - _d(a["mean"])[:, None]) * _d(a["rstd"])[:, None]
        gam, _ = _ln_gamma_beta(a, D)
        dyw = dy * gam
        dx = _d(a["rstd"])[:, None] * (dyw - dyw.mean(-1, keepdim=True) - xh * (dyw * xh).mean(-1, keepdim=True))
        if a["dres"] is not None:
            dx = dx + _d(a["dres"])
        res = [("dx", ret[0] if a["want_dx16"] else ret, dx)]
        if a["want_dx16"]:
            m = 1.0 if a["dx16_rowmask"] is None else a["dx16_rowmask"].double()[:, None]
            res.append(("dx16", ret[1], dx * m))
        if a["dgb"] is not None:
            res.append(("dgb", after["dgb"], torch.cat([dy * xh, dy], dim=1)))
        if a["dw"] is not None:
            res += [("dw", after["dw"], _d(a["dw"]) + (dy * xh).sum(0)), ("db", after["db"], _d(a["db"]) + dy.sum(0))]
        return res
    if name in ("attention_fwd", "attention_bwd"):
        B, T, H = a["B"], a["T"], a["H"]
        qkv = _d(a["qkv"]).view(B, T, -1)
        mask = None if a["key_mask"] is None else a["key_mask"].bool()
        ls = _d(a["logslopes"])
        if name == "attention_fwd":
            o = _Attention.apply(qkv, ls, mask, H, a["causal"], False, True).reshape(B * T, -1)
            ok = _allowed(mask if mask is not None else torch.ones(B, T, dtype=torch.bool, device=qkv.device), T, a["causal"],
                          qkv.device).any(-1).reshape(B * T)   # a query without any key attends to nothing in particular
            return [("o", ret[0][ok], o[ok])]
        dqkv, dls = attention_grads(qkv, ls, mask, H, a["causal"], _d(a["dout"]).view(B, T, -1), _d(a["delta"]))
        return [("dqkv", ret, dqkv.reshape(B * T, -1)), ("dls", after["dlogslopes"], _d(a["dlogslopes"]) + dls)]
    if name == "ffn_fwd":
        u = _d(a["xn"]) @ _d(a["w1"]).t() + _d(a["b1"])
        h = _GLU.apply(u, False)
        out = (_d(ret[2]) if a["save"] else _bf(h)) @ _d(a["w2"]).t()     # GEMM2 from the h the kernel stored (tanh.approx)
        if a["resid"] is not None:
            out = out + _d(a["resid"])
        return [("out", ret[0], out)] + ([("u", ret[1], u), ("h", ret[2], h)] if a["save"] else [])
    if name == "ffn_bwd":
        dh = _d(a["dy"]) @ _d(a["w2t"]).t()
        va, g = _d(a["u"]).chunk(2, dim=-1)
        sig = torch.sigmoid(g)
        silu = g * sig
        du = torch.cat([dh * silu, dh * va * (sig + silu * (1 - sig))], dim=-1)
        res = [("dxn", ret[0], _bf(du) @ _d(a["w1"])), ("du", ret[1], du)]
        if a["db1"] is not None:
            res.append(("db1", after["db1"], _d(a["db1"]) + du.sum(0)))
        return res
    if name == "colsum":
        s = _d(a["x"]).sum(0)
        return [("sum", ret, s + (_d(a["out"]) if a["out"] is not None else 0))]
    if name == "multi_add":
        return [(f"dst{i}", after["dsts"][i], _d(d) + _d(s)) for i, (d, s) in enumerate(zip(a["dsts"], a["srcs"]))]
    if name == "transpose_bf16":
        ws = [a["ws"]] if isinstance(a["ws"], torch.Tensor) else a["ws"]
        return [(f"w{i}T", ret[i] if len(ws) > 1 else ret, _d(w).t()) for i, w in enumerate(ws)]
    raise AssertionError(name)


# Bars of one call against its float64 statement, by the dtype the output is stored in.  A bf16 store is off by up to half an
# ulp, 2^-9 of the element, so up to 3.9e-3 of the largest element once fp32 sums flip a rounding; its cosine distance is that
# quantisation noise, ~1.4e-6 for any large tensor.  The attention kernels add the on-chip bf16 roundings of P (and dS); the
# logslopes gradient cancels (see BARS).  Largest values measured on a B200 (1000 W) over every call of both stack kinds and
# both gradient modes: bf16 rel 3.5e-3 cos 1.40e-6; fp32 rel 1.0e-5 (a weight gradient) cos 4.5e-12; attention o / dqkv rel
# 5.4e-3 cos 2.8e-6; dlogslopes rel 1.1e-2 cos 4.5e-5.  The feed-forward output is taken from the h the kernel stored.
CALL_BARS = {"bf16": dict(rel=5e-3, cos=2.5e-6), "fp32": dict(rel=3e-5, cos=1e-10),
             "attention": dict(rel=8e-3, cos=5e-6), "dls": dict(rel=3e-2, cos=1e-4)}
CALL_WORST = {}


@pytest.mark.gpu
@pytest.mark.parametrize("direct", [False, True], ids=["autograd", "trainstep"])
@pytest.mark.parametrize("kind", ["perf_enc", "decoder"])
def test_every_kernel_call_matches_its_statement(gpu_model, K, monkeypatch, kind, direct):
    """Each kernel call of one forward + backward of the node (3 x 130, ragged mask) against the float64 statement of that
    one operation on the inputs the call actually received: the real slices, strides, row masks and norm indices."""
    mod, spec = _cuda_stack(gpu_model, kind)
    params = list(mod.flat_params())
    x, mask, style, g_out = make_inputs(spec, 3, 130, True, "cuda", 77, 64)
    calls = record_calls(K, monkeypatch)
    if direct:
        run_direct(K, mod, spec, x, mask, style, g_out, [torch.ones_like(p) for p in params])
    else:
        run_node(spec, params, x, mask, style, g_out)
    monkeypatch.undo()
    seen, bad = {}, []
    for i, (name, a, after, ret) in enumerate(calls):
        for label, got, want in call_statement(name, a, after, ret):
            if name == "transpose_bf16":
                assert torch.equal(got.double(), want), (i, name)
                continue
            key = f"{name}.{label}"
            cls = "dls" if key == "attention_bwd.dls" else "attention" if name.startswith("attention") else \
                "bf16" if got.dtype == BF16 else "fp32"
            seen[key] = seen.get(key, 0) + 1
            assert torch.isfinite(got).all(), (i, key)
            st = dict(rel=rel_err(got, want), cos=cos_dist(got, want)) if float(want.abs().max()) > 0 else \
                dict(rel=float(got.abs().max()), cos=0.0)
            w = CALL_WORST.setdefault((kind, key, cls), dict(rel=0.0, cos=0.0))
            for s, v in st.items():
                w[s] = max(w[s], v)
                if not v < CALL_BARS[cls][s]:
                    bad.append(f"call {i} {key} ({cls}): {s} {v:.2e} >= {CALL_BARS[cls][s]:.1e}")
    for (k_, key, cls), w in sorted(CALL_WORST.items()):
        if k_ == kind:
            print(f"  {kind} {key:28s} {cls:9s} rel {w['rel']:.2e} cos {w['cos']:.2e}")
    assert seen.get("ffn_bwd.du", 0) == spec.depth and seen.get("attention_bwd.dqkv", 0) == spec.depth, seen
    assert not bad, "\n".join(bad)


# ------------------------------------------------------------------ GPU: the whole training step in TrainStep's mode
# Per-parameter bars of TrainStep's gradients against plain autograd on the same weights and batch.  Both run the same
# kernels; they differ in how weight gradients reach memory (accumulated in place vs returned) and in fp32 atomics (split-K,
# segment pooling), whose last-bit differences sometimes flip a bf16 rounding that then propagates.  Largest values measured on
# a B200 (1000 W) over every parameter, eager and replayed, over several runs: cos 2.4e-5, ratio 2.9e-3 (a logslopes
# gradient, see BARS; 7.2e-4 for every other parameter); in runs without such a flip both stay below 1e-14 / 1e-7.  A gradient
# slot that is missed, doubled or overwritten moves cos or ratio by far more than these bars.
STEP_COS, STEP_RATIO = 1e-4, 1e-2


@pytest.mark.gpu
def test_train_step_gradients_match_plain_autograd(K):
    """TrainStep (lr 0, dropout off, fixed prior samples, so every step computes the gradient of the same weights) against
    loss.backward() of an identically built model on the same batch: every parameter's slot of the flat gradient buffer,
    after an eager step and after a CUDA-graph replay.  This covers the direct-gradient paths of every node of the model:
    transformer stacks, linear layers, heads, embeddings, latent levels."""
    from scoreperformer_b200.train_step import TrainStep
    batch = {k: v.cuda() for k, v in parity.make_batch(2, 64, seed=5).items()}
    g = torch.Generator().manual_seed(17)
    z = [torch.randn(256, d, generator=g).cuda() for d in (32, 20, 8, 4)]

    def build():
        m = parity.build_model(dropout=False, device="cuda")
        m.train()
        m.perf_encoder.exact_latent_shapes = False
        m.z_prior = [t.clone() for t in z]
        return m

    ref = build()
    ref(**batch).loss.backward()
    want = {n: p.grad.detach().clone() for n, p in ref.named_parameters() if p.requires_grad}
    m = build()
    rng_offset = K.RNG_OFFSET
    try:
        ts = TrainStep(m, lr=0.0, grad_clip=None, use_graph=True)
        worst = dict(cos=(0.0, ""), ratio=(0.0, ""))
        bad = []
        for step in range(5):                       # 3 eager warm-ups, capture, replay
            ts.step(batch)
            if step not in (0, 4):
                continue
            torch.cuda.synchronize()
            for n, p in m.named_parameters():
                if not p.requires_grad:
                    continue
                got, w = p.grad, want[n]
                assert got.data_ptr() >= ts.flat_grad.data_ptr() and torch.isfinite(got).all(), n
                if float(w.abs().max()) == 0.0:
                    assert float(got.abs().max()) == 0.0, n
                    continue
                c, r = cos_dist(got, w), norm_ratio(got, w)
                worst["cos"] = max(worst["cos"], (c, n))
                worst["ratio"] = max(worst["ratio"], (r, n))
                if not (c < STEP_COS and r < STEP_RATIO):
                    bad.append(f"step {step} {n}: cos {c:.2e} ratio {r:.2e}")
    finally:
        K.RNG_OFFSET = rng_offset
    print(f"train step vs autograd: worst cos {worst['cos'][0]:.2e} ({worst['cos'][1]}), "
          f"worst ratio {worst['ratio'][0]:.2e} ({worst['ratio'][1]})")
    assert not bad, "\n".join(bad)
