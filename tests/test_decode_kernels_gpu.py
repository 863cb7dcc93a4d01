"""The cached decoder-step kernels against a float64 statement of one cached decoder step.

`ref_step` is one new position through the decoder stack, written after `oracle/model_oracle.transformer_stack(...,
caches=...)` (with its `attention`, `_norm` and `feed_forward`) over the weight layout of csrc/decode_stack.cu.  `ref_front` is
the input front of the rendering loop, x = LN(x1 Wf^T + p2) Wc^T + c2.  The CPU tests pin both to the oracle in float64; the
GPU tests compare `spb_attention_decode` and `spb_decode_stack_step` with them.

With `rounded=True` the statement rounds to bf16 exactly where decode_stack.cu stores bf16: the style row and the AdaLN terms
`gb`, every AdaLN output `xn`, `qkv` (which the cache stores), the normalised attention output `o`, the GLU output `hmid` and
the front's LayerNorm output.  The one rounding it leaves out is that of the softmax weights P before P.V (the kernel feeds P
to the tensor cores as bf16).  So the kernel must agree with the rounded statement to within reordered fp32 sums, P's
rounding, and the bf16 roundings those flip; and with the plain float64 statement to within its bf16 storage.
"""
import math

import pytest
import torch
import torch.nn.functional as F

from tests import parity
from tests.test_kernels_gpu import cos_dist, rel_err
import model_oracle as mo

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64
D, H, DH, HID = 256, 4, 64, 1024
EPS = 1e-5
DEC = "perf_decoder.model"


def _bf(t):
    return t.to(BF16).to(t.dtype)


def rel_err64(a, b):
    """rel_err without the fp32 conversion: for statements that must agree to float64 rounding."""
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp(min=1e-300))


# ------------------------------------------------------------------ the float64 statements
def ref_front(x1, wf, p2, ln_w, ln_b, wc_t, c2, rounded=False, eps=EPS):
    """x = LN(x1 wf^T + p2) wc_t + c2 (wc_t input-major), the front decode_stack.cu evaluates with `front`."""
    y = F.layer_norm(x1 @ wf.t() + p2, (D,), ln_w, ln_b, eps)
    return (_bf(y) if rounded else y) @ wc_t + c2


def _adaln(x, gb, eps):
    """AdaLN from the (gamma - 1 | beta) row the kernels use: gamma * LN(x) + beta."""
    return F.layer_norm(x, (D,), eps=eps) * (1 + gb[:, :D]) + gb[:, D:]


def ref_step(W, style, kv, key_mask, x, pos, rounded=False, eps=EPS):
    """One cached step of the decoder stack at position `pos`.

    W: float64 weights in the kernel's layout (`weights_from_state`), style [B, S], kv[l] [B, >= pos, 128] holding k | v of the
    rows < pos, key_mask [B, > pos] (bool, None: no padding), x [B, 256] the stack input of position pos.
    Returns (k | v of position pos per layer [depth, B, 128], attention-layer inputs [depth, B, 256], final AdaLN output [B, 256]).
    Masked keys get the oracle's additive fill; the attention output is zeroed at a padded query (key_mask[:, pos])."""
    r = _bf if rounded else (lambda t: t)
    B = x.shape[0]
    gb = r(r(style) @ W["w_ada"].t() + W["b_ada"])
    valid = torch.ones(B, pos + 1, dtype=torch.bool, device=x.device) if key_mask is None else key_mask[:, :pos + 1].bool()
    dist = (pos - torch.arange(pos + 1, device=x.device)).abs().to(x.dtype)
    fill = -torch.finfo(x.dtype).max // 2
    kv_new, hid = [], []
    for l, L in enumerate(W["layers"]):
        hid.append(x)
        xn = r(_adaln(x, gb[:, 2 * l * 2 * D:(2 * l + 1) * 2 * D], eps))
        qkv = r(xn @ L["wqkv"].t())
        kv_new.append(qkv[:, H * DH:])
        keys = torch.cat([kv[l][:, :pos].to(x.dtype), qkv[:, None, H * DH:]], dim=1)
        s = torch.einsum("bhd,bjd->bhj", qkv[:, :H * DH].view(B, H, DH), keys[..., :DH]) * DH ** -0.5
        s = s - L["ls"].exp()[None, :, None] * dist
        p = s.masked_fill(~valid[:, None, :], fill).softmax(dim=-1)
        o = r(torch.einsum("bhj,bjd->bhd", p, keys[..., DH:]).reshape(B, H * DH))
        x = x + valid[:, pos:pos + 1].to(x.dtype) * (o @ L["wo"].t())
        xn = r(_adaln(x, gb[:, (2 * l + 1) * 2 * D:(2 * l + 2) * 2 * D], eps))
        u = xn @ L["w1"].t() + L["b1"]
        h = r(u[:, :HID] * F.silu(u[:, HID:]))
        x = x + h @ L["w2"].t()
    depth = len(W["layers"])
    return torch.stack(kv_new), torch.stack(hid), _adaln(x, gb[:, 2 * depth * 2 * D:], eps)


def weights_from_state(sd, prefix, depth):
    """The oracle's state dict -> the layout of decode.py's _StackWeights (q|k|v rows concatenated, AdaLN rows of all norms
    concatenated with 1 subtracted from every gamma bias)."""
    layers, nw, nb = [], [], []
    for l in range(depth):
        a, f = f"{prefix}.layers.{2 * l}", f"{prefix}.layers.{2 * l + 1}"
        layers.append(dict(wqkv=torch.cat([sd[f"{a}.1.to_q.weight"], sd[f"{a}.1.to_k.weight"], sd[f"{a}.1.to_v.weight"]]),
                           wo=sd[f"{a}.1.to_out.weight"], ls=sd[f"{a}.1.rel_pos.learned_logslopes"].reshape(-1),
                           w1=sd[f"{f}.1.ff.0.proj.weight"], b1=sd[f"{f}.1.ff.0.proj.bias"], w2=sd[f"{f}.1.ff.3.weight"]))
        nw += [sd[f"{a}.0.0.linear.weight"], sd[f"{f}.0.0.linear.weight"]]
        nb += [sd[f"{a}.0.0.linear.bias"], sd[f"{f}.0.0.linear.bias"]]
    nw.append(sd[f"{prefix}.final_norm.linear.weight"])
    nb.append(sd[f"{prefix}.final_norm.linear.bias"])
    ones = torch.cat([torch.ones(D), torch.zeros(D)]).to(nb[0]).repeat(len(nb))
    return dict(layers=layers, w_ada=torch.cat(nw), b_ada=torch.cat(nb) - ones)


# ------------------------------------------------------------------ CPU: the statements against the oracle
@pytest.fixture(scope="module")
def dec_state():
    model = parity.build_model(dropout=False, device="cpu")
    sd = {k: v.detach().double() for k, v in parity.oracle_state(model, requires_grad=False).items()}
    return sd, parity.oracle_spec(model)


@pytest.mark.parametrize("ragged", [False, True])
def test_reference_step_matches_oracle_stack(dec_state, ragged):
    """P cached steps from an empty cache equal the oracle's uncached causal stack over the whole sequence, position by
    position: output, attention-layer inputs and k|v, to float64 rounding (measured 7.0e-15 plain, 5.3e-15 ragged).  The bound
    sits far above that on purpose: it only has to separate reordered float64 sums (~1e-14) from a different statement, which
    shows at bf16 / fp32 size (>= 1e-8)."""
    sd, spec = dec_state
    prefix, depth = f"{DEC}.transformer", spec.depth_dec
    W = weights_from_state(sd, prefix, depth)
    g = torch.Generator().manual_seed(5)
    B, P = 3, 21
    x = torch.randn(B, P, D, generator=g, dtype=F64)
    style = torch.randn(B, P, spec.style_dim, generator=g, dtype=F64)
    mask = None
    if ragged:                                  # row 1 padded at the end, row 2 with holes (position 0 among them)
        mask = torch.ones(B, P, dtype=torch.bool)
        mask[1, 13:] = False
        mask[2, [0, 4, 5, 11]] = False
    want, hiddens, kvs = mo.transformer_stack(sd, prefix, x, mask, depth, True, spec, style=style)
    kv = [torch.zeros(B, P, 128, dtype=F64) for _ in range(depth)]
    for t in range(P):
        kv_t, hid_t, out_t = ref_step(W, style[:, t], kv, mask, x[:, t], t)
        assert rel_err64(out_t, want[:, t]) < 1e-12, t
        for l in range(depth):
            kv[l][:, t] = kv_t[l]
            assert rel_err64(hid_t[l], hiddens[l][:, t]) < 1e-12, (t, l)
            assert rel_err64(kv_t[l], torch.cat(kvs[l], dim=-1)[:, t]) < 1e-12, (t, l)


def _emb_ln(sd, spec, tokens):
    """tuple embedding up to its LayerNorm (model_oracle.tuple_embed without project_emb): what the rendering loop's x1 holds."""
    keys = list(spec.num_tokens)
    x = torch.cat([mo.field_table(sd, f"{DEC}.token_emb", k, spec.discrete_ids)[tokens[..., i]] for i, k in enumerate(keys)], dim=-1)
    return F.layer_norm(x, (x.shape[-1],), sd[f"{DEC}.token_emb.norm.weight"], sd[f"{DEC}.token_emb.norm.bias"])


def test_front_statement_matches_oracle_decoder_embed(dec_state):
    """ref_front with the operands decode.render_decoder composes (Wf = project_multiemb's left half . project_emb, p2 = the
    masked tuple's half + biases, c2 = the context half of the decoder's project_emb + bias) equals oracle.decoder_embed."""
    sd, spec = dec_state
    g = torch.Generator().manual_seed(7)
    B, T = 2, 6
    tok = lambda: torch.stack([torch.randint(0, n, (B, T), generator=g) for n in spec.num_tokens.values()], dim=-1)
    seq, seq_masked = tok(), tok()
    ctx = torch.randn(B, T, D, generator=g, dtype=F64)
    want, _ = mo.decoder_embed(sd, seq, seq_masked, ctx, spec)
    wp, bp = sd[f"{DEC}.token_emb.project_emb.weight"], sd[f"{DEC}.token_emb.project_emb.bias"]
    wm, bm = sd[f"{DEC}.token_emb.project_multiemb.weight"], sd[f"{DEC}.token_emb.project_multiemb.bias"]
    wc, bc = sd[f"{DEC}.project_emb.weight"], sd[f"{DEC}.project_emb.bias"]
    p2 = (_emb_ln(sd, spec, seq_masked) @ wp.t() + bp) @ wm[:, D:].t() + bm + wm[:, :D] @ bp
    c2 = ctx @ wc[:, D:].t() + bc
    got = ref_front(_emb_ln(sd, spec, seq), wm[:, :D] @ wp, p2, sd[f"{DEC}.emb_norm.weight"], sd[f"{DEC}.emb_norm.bias"],
                    wc[:, :D].t(), c2)
    assert rel_err64(got, want) < 1e-12


# ------------------------------------------------------------------ GPU: spb_attention_decode
@pytest.fixture(scope="module")
def k():
    from scoreperformer_b200 import kernels
    return kernels


def ref_attention_decode(q, kv, key_mask, logslopes, n_heads, n_keys, q_pos):
    """float64 MQA + ALiBi of one query at q_pos over keys j < n_keys with j <= q_pos and key_mask[b, j]; a row without any key
    attends to nothing (zeros)."""
    B = q.shape[0]
    qd = q[:, :n_heads * DH].double().view(B, n_heads, DH)
    kd, vd = kv[:, :n_keys, :DH].double(), kv[:, :n_keys, DH:].double()
    j = torch.arange(n_keys, device=q.device)
    s = torch.einsum("bhd,bjd->bhj", qd, kd) * DH ** -0.5 - logslopes.double().exp()[None, :, None] * (q_pos - j).abs().double()
    ok = (j <= q_pos)[None].expand(B, -1)
    if key_mask is not None:
        ok = ok & key_mask[:, :n_keys].bool()
    p = s.masked_fill(~ok[:, None, :], -math.inf).softmax(dim=-1).nan_to_num(0.0)
    return torch.einsum("bhj,bjd->bhd", p, vd).reshape(B, n_heads * DH)


def _logslopes(n_heads, dev):
    return torch.log(torch.tensor([2.0 ** (-8.0 * (h + 1) / n_heads) for h in range(n_heads)], device=dev)).float()


# The kernel's only rounding is the bf16 store of the output: half an ulp, at most 2^-8 = 3.9e-3 of an element (bf16 carries 8
# significant bits) and so of the largest element; 4.5e-3 leaves room for the fp32 sums over up to 4096 keys.  Largest value
# measured on a B200 (1000 W) over every case of this file: 3.2e-3.
ATT_REL = 4.5e-3


@pytest.mark.gpu
@pytest.mark.parametrize("n_heads,n_keys,q_pos", [
    (1, 200, 199), (16, 1000, 999),
    (4, 1, 0), (4, 31, 30), (4, 32, 31), (4, 33, 32), (4, 1000, 999), (4, 4096, 4095),
    (4, 300, 120), (4, 33, 5),                  # keys after the query are ignored
])
def test_attention_decode_matches_float64(k, n_heads, n_keys, q_pos):
    torch.manual_seed(n_keys * 7 + n_heads)
    dev = "cuda"
    B = 5
    ls = _logslopes(n_heads, dev)
    w = n_heads * DH + 128
    # contiguous operands, no mask
    q = torch.randn(B, w, device=dev).to(BF16)
    kv = torch.randn(B, n_keys, 128, device=dev).to(BF16)
    out = k.attention_decode(q, kv, None, ls, n_heads, n_keys, q_pos)
    want = ref_attention_decode(q, kv, None, ls, n_heads, n_keys, q_pos)
    e = rel_err(out, want)
    print(f"attention_decode H={n_heads} n={n_keys} q_pos={q_pos}: plain {e:.2e}", end="")
    assert e < ATT_REL                                                     # ATT_REL, measured <= 3.2e-3 over this file
    # strided operands: q rows wider than H*64+128, the cache a view into a longer one (kv_batch_stride > cap*128), the mask a
    # view into a wider one (mask_stride > n_keys) with holes, and one row whose keys up to the query are all masked
    qs = torch.randn(B, w + 64, device=dev).to(BF16)[:, :w]
    kvs = torch.randn(B, n_keys + 24, 128, device=dev).to(BF16)[:, :n_keys]
    mask = (torch.rand(B, n_keys + 40, device=dev) > 0.3)[:, :n_keys]
    mask[:, q_pos] = True
    mask[1, :q_pos + 1] = False
    out = k.attention_decode(qs, kvs, mask, ls, n_heads, n_keys, q_pos)
    want = ref_attention_decode(qs, kvs, mask, ls, n_heads, n_keys, q_pos)
    e = rel_err(out, want)
    print(f", strided + holes {e:.2e}")
    assert e < ATT_REL                                                     # ATT_REL, measured <= 3.2e-3 over this file
    assert torch.equal(out[1], torch.zeros_like(out[1]))
    # the position read on the device (n_keys is then the capacity) computes exactly what the host position does
    host = k.attention_decode(qs, kvs, mask, ls, n_heads, q_pos + 1, q_pos)
    dev_pos = k.attention_decode(qs, kvs, mask, ls, n_heads, n_keys, 0, pos_dev=torch.tensor([q_pos], device=dev))
    assert torch.equal(dev_pos, host)


@pytest.mark.gpu
@pytest.mark.parametrize("n_heads,cap,q_pos", [(4, 64, 0), (4, 64, 37), (4, 64, 63), (16, 700, 411)])
def test_attention_decode_append_kv(k, n_heads, cap, q_pos):
    """append_kv with a device position: cache row q_pos becomes q[:, H*64:H*64+128] bit for bit, every other row is unchanged,
    and the query attends to the appended row."""
    torch.manual_seed(cap + q_pos)
    B, w = 3, n_heads * DH + 128
    q = torch.randn(B, w + 32, device="cuda").to(BF16)[:, :w]
    kv = torch.randn(B, cap, 128, device="cuda").to(BF16)
    before = kv.clone()
    mask = torch.rand(B, cap, device="cuda") > 0.2
    mask[:, q_pos] = True
    ls = _logslopes(n_heads, "cuda")
    out = k.attention_decode(q, kv, mask, ls, n_heads, cap, 0, pos_dev=torch.tensor([q_pos], device="cuda"), append_kv=True)
    assert torch.equal(kv[:, q_pos], q[:, n_heads * DH:])
    rows = torch.arange(cap, device="cuda") != q_pos
    assert torch.equal(kv[:, rows], before[:, rows])
    assert rel_err(out, ref_attention_decode(q, kv, mask, ls, n_heads, cap, q_pos)) < ATT_REL       # ATT_REL, measured <= 3.2e-3 over this file


@pytest.mark.gpu
@pytest.mark.parametrize("q_pos", [-1, 64, 67])
def test_attention_decode_append_outside_cache_writes_nothing(k, q_pos):
    """A device position outside [0, cap) appends nothing.  The cache is carved out of one buffer with canary rows on both
    sides, so a missing guard would land in memory the test owns (the neighbouring score's rows or a canary), not outside it."""
    torch.manual_seed(11)
    B, cap, pad = 3, 64, 8
    flat = torch.randn((B * cap + 2 * pad) * 128, device="cuda").to(BF16)
    before = flat.clone()
    kv = flat[pad * 128:(pad + B * cap) * 128].view(B, cap, 128)
    q = torch.randn(B, H * DH + 128, device="cuda").to(BF16)
    ls = _logslopes(H, "cuda")
    out = k.attention_decode(q, kv, None, ls, H, cap, 0, pos_dev=torch.tensor([q_pos], device="cuda"), append_kv=True)
    assert torch.equal(flat, before)
    want = ref_attention_decode(q, kv, None, ls, H, cap, q_pos)                  # q_pos < 0: no key, zeros
    assert (out == 0).all() if q_pos < 0 else rel_err(out, want) < ATT_REL     # ATT_REL, measured <= 3.2e-3 over this file


@pytest.mark.gpu
def test_attention_decode_rejects_what_it_cannot_hold(k):
    """H * n_keys fp32 scores above the shared memory of a block, and a host position outside the cache with append_kv, are
    argument errors reported before any launch."""
    q = torch.zeros(1, 16 * DH + 128, dtype=BF16, device="cuda")
    kv = torch.zeros(1, 4096, 128, dtype=BF16, device="cuda")
    with pytest.raises(RuntimeError, match="shared memory"):
        k.attention_decode(q, kv, None, _logslopes(16, "cuda"), 16, 4096, 4095)
    with pytest.raises(RuntimeError, match="append_kv"):
        k.attention_decode(q, kv, None, _logslopes(16, "cuda"), 16, 100, 100, append_kv=True)
    torch.cuda.synchronize()


# ------------------------------------------------------------------ GPU: spb_decode_stack_step
def make_weights(depth, S, seed, dev):
    """Seeded stack weights in the kernel's layout, as float64 values that bf16 (matrices) / fp32 (biases, slopes) hold exactly.
    Scaled so that q.k / 8 and the ALiBi terms are O(1), the AdaLN gammas stay near 1, and the residual stream grows slowly."""
    g = torch.Generator().manual_seed(seed)
    rn = lambda *s, scale: torch.randn(*s, generator=g, dtype=F64) * scale
    b16 = lambda t: _bf(t).to(dev)
    f32 = lambda t: t.float().double().to(dev)
    base = torch.log(torch.tensor([2.0 ** (-2 * (h + 1)) for h in range(H)], dtype=F64))
    layers = [dict(wqkv=b16(rn(H * DH + 128, D, scale=D ** -0.5)), wo=b16(rn(D, D, scale=0.5 * D ** -0.5)),
                   ls=f32(base + rn(H, scale=0.1)), w1=b16(rn(2 * HID, D, scale=D ** -0.5)), b1=f32(rn(2 * HID, scale=0.1)),
                   w2=b16(rn(D, HID, scale=0.5 * HID ** -0.5))) for _ in range(depth)]
    n = 2 * depth + 1
    return dict(layers=layers, w_ada=b16(rn(n * 2 * D, S, scale=0.3 * S ** -0.5)), b_ada=f32(rn(n * 2 * D, scale=0.1)))


def kernel_weights(W):
    layers = [dict(wqkv=L["wqkv"].to(BF16).contiguous(), wo=L["wo"].to(BF16).contiguous(), ls=L["ls"].float().contiguous(),
                   w1=L["w1"].to(BF16).contiguous(), b1=L["b1"].float().contiguous(), w2=L["w2"].to(BF16).contiguous())
              for L in W["layers"]]
    return layers, W["w_ada"].to(BF16).contiguous(), W["b_ada"].float().contiguous()


def make_front(B, seed, dev):
    """Front operands: te = x1 Wf^T + p2 has rms ~0.01, so LN's eps is 1 % of the row variance and a wrong eps shows."""
    g = torch.Generator().manual_seed(seed)
    rn = lambda *s, scale=1.0: torch.randn(*s, generator=g) * scale
    return dict(x1=rn(B, 1536).to(BF16).to(dev), wf=rn(D, 1536, scale=0.01 / math.sqrt(1536)).to(BF16).to(dev),
                p2=rn(B, D, scale=0.003).to(dev), ln_w=(1 + rn(D, scale=0.1)).to(dev), ln_b=rn(D, scale=0.1).to(dev),
                wc_t=rn(D, D, scale=D ** -0.5).to(BF16).to(dev), c2=rn(B, D, scale=0.5).to(dev))


def front_x(fr, rounded):
    d = {n: t.double() for n, t in fr.items()}
    return ref_front(d["x1"], d["wf"], d["p2"], d["ln_w"], d["ln_b"], d["wc_t"], d["c2"], rounded=rounded)


def ragged_mask(B, cap, pos, dev):
    """Holes everywhere, row 0 complete; every third row (2, 5, ...) has its query position padded."""
    m = torch.rand(B, cap, device=dev) > 0.2
    m[:, pos] = True
    m[2::3, pos] = False
    if B > 1:
        m[0] = True
    return m.to(torch.uint8)


# Bounds of the stack step.  TIGHT: against the rounded statement (what is left is fp32 summation order, the bf16 rounding of
# P, and the bf16 roundings that these flip); LOOSE: against plain float64 (the bf16 storage of xn, qkv, o, hmid, gb, style).
# rel_err is a max-abs statistic, so one flipped bf16 rounding of a large element sets it: a k|v element carries up to a full
# ulp, 2^-7 = 7.8e-3, against either statement; the cosine distance sees the whole tensor and is where the rounded statement
# is closer.  Largest values measured on a B200 (1000 W) over every case, path and step of this file:
#   tight rel  out 4.7e-3  hid 3.9e-3  kv 7.2e-3      tight cos  out 4.9e-6  hid 2.6e-6  kv 5.0e-6
#   loose rel  out 4.5e-3  hid 3.6e-3  kv 4.6e-3      loose cos  out 7.8e-6  hid 4.1e-6  kv 6.4e-6
TIGHT_REL, TIGHT_COS = 1e-2, 1e-5
LOOSE_REL, LOOSE_COS = 1.5e-2, 2e-5


def _errs(got, want):
    return rel_err(got, want), cos_dist(got, want)


class _Case:
    """One (B, pos, cap, depth, S) configuration: weights, caches, plan, inputs, and the four references."""

    def __init__(self, k, B, pos, cap, depth, S, seed=0):
        dev = "cuda"
        torch.manual_seed(1000 * seed + B + pos)
        self.B, self.pos, self.cap, self.depth = B, pos, cap, depth
        self.W = make_weights(depth, S, seed=depth * 1000 + S, dev=dev)
        layers, w_ada, b_ada = kernel_weights(self.W)
        self.kv0 = [torch.randn(B, cap, 128, device=dev).to(BF16) for _ in range(depth)]
        self.caches = [c.clone() for c in self.kv0]
        self.plan = k.DecodeStackPlan(layers, w_ada, b_ada, self.caches, B, S, keep_hiddens=True)
        self.x = torch.randn(B, D, device=dev)
        self.style = torch.randn(B, S, device=dev)
        self.mask = ragged_mask(B, cap, pos, dev)
        self.pos_dev = torch.tensor([pos], device=dev)
        # prepared AdaLN terms: this step's style at position pos + 1; and with T_all = pos + 1, where pos + 1 is clamped to pos
        sa = torch.randn(B, pos + 3, S, device=dev)
        sa[:, pos + 1] = self.style
        self.gb_all = self.plan.prepare_adaln(sa.contiguous())
        sc = torch.randn(B, pos + 1, S, device=dev)
        sc[:, pos] = self.style
        self.gb_clamped = self.plan.prepare_adaln(sc.contiguous())
        self.front = make_front(B, seed + pos, dev)
        f = self.front
        self.plan.set_front(f["x1"], f["wf"], f["p2"], f["ln_w"], f["ln_b"], f["wc_t"], f["c2"])
        kvd = [c.double() for c in self.kv0]
        self.ref = {}
        for src, xs in (("x", lambda r: self.x.double()), ("front", lambda r: front_x(f, r))):
            for rounded in (True, False):
                self.ref[src, rounded] = ref_step(self.W, self.style.double(), kvd, self.mask, xs(rounded), pos, rounded=rounded)

    def launch(self, path, barrier_is_zero=False):
        p = self.plan
        for t in (p.out, p.hid):
            t.fill_(float("nan"))
        p.out16.fill_(float("nan"))
        for c, c0 in zip(self.caches, self.kv0):
            c.copy_(c0)
        x = None if path.startswith("front") else self.x
        gb_all = {"gb_all": self.gb_all, "front_gb_all": self.gb_all, "gb_all_clamped": self.gb_clamped}.get(path)
        p.step(x, None if gb_all is not None else self.style, self.mask, self.pos_dev, gb_all=gb_all,
               use_front=path.startswith("front"), barrier_is_zero=barrier_is_zero)
        torch.cuda.synchronize()

    def check(self, path, worst):
        p, pos = self.plan, self.pos
        src = "front" if path.startswith("front") else "x"
        kv_r, hid_r, out_r = self.ref[src, True]
        kv_x, hid_x, out_x = self.ref[src, False]
        assert torch.equal(p.out16, p.out.to(BF16)), path
        got = {"out": (p.out, out_r, out_x), "hid": (p.hid, hid_r, hid_x),
               "kv": (torch.stack([c[:, pos] for c in self.caches]), kv_r, kv_x)}
        for name, (g, r, x) in got.items():
            assert torch.isfinite(g).all(), (path, name)
            t_rel, t_cos = _errs(g, r)
            l_rel, l_cos = _errs(g, x)
            for key, v in ((f"{name} tight rel", t_rel), (f"{name} tight cos", t_cos), (f"{name} loose rel", l_rel),
                           (f"{name} loose cos", l_cos)):
                worst[key] = max(worst.get(key, 0.0), v)
            assert t_rel < TIGHT_REL and t_cos < TIGHT_COS, (path, name, t_rel, t_cos)
            assert l_rel < LOOSE_REL and l_cos < LOOSE_COS, (path, name, l_rel, l_cos)
        for c, c0 in zip(self.caches, self.kv0):                 # only row pos of each cache is written
            assert torch.equal(c[:, :pos], c0[:, :pos]) and torch.equal(c[:, pos + 1:], c0[:, pos + 1:]), path


STACK_CASES = [                 # B, pos, cap, depth, S: key counts at the 16-key / per-warp split edges, odd B, B > 2 x 148 SMs
    (1, 0, 64, 4, 64),
    (2, 15, 64, 1, 16),
    (3, 16, 80, 8, 256),
    (33, 17, 128, 4, 64),
    (2, 63, 64, 4, 64),
    (3, 64, 96, 4, 16),
    (33, 65, 200, 1, 256),
    (297, 511, 512, 4, 64),
    (5, 2047, 2048, 8, 64),
]
PATHS = ["style", "gb_all", "gb_all_clamped", "front", "front_gb_all"]


@pytest.mark.gpu
@pytest.mark.parametrize("B,pos,cap,depth,S", STACK_CASES)
def test_decode_stack_step_matches_reference(k, B, pos, cap, depth, S):
    """One step through every input path on the same data: AdaLN terms from `style` (phase 0) or prepared (`gb_all`, also where
    position pos + 1 is clamped to T_all - 1), stack input `x_in` or the in-kernel front.  out, its bf16 copy, hid_out and the
    appended k|v rows against the rounded (tight) and the plain (loose) float64 statement."""
    case = _Case(k, B, pos, cap, depth, S)
    worst = {}
    for path in PATHS:
        case.launch(path)
        case.check(path, worst)
    print(f"decode_stack B={B} pos={pos} cap={cap} depth={depth} S={S}: " + ", ".join(f"{n} {v:.2e}" for n, v in worst.items()))


@pytest.mark.gpu
def test_decode_stack_step_repeatable_and_barrier_is_zero(k):
    """Nothing in the kernel uses atomics on data: a second identical launch is bit-identical (out, hid_out, caches); so is a
    launch that trusts the grid-barrier word to be zero already (`barrier_is_zero`, as after the sampling kernel's advance)."""
    case = _Case(k, 33, 65, 128, 4, 64)
    p = case.plan
    results = []
    for barrier_is_zero in (False, False, True):
        if barrier_is_zero:
            p.barrier.zero_()
        case.launch("front_gb_all", barrier_is_zero=barrier_is_zero)
        results.append([p.out.clone(), p.out16.clone(), p.hid.clone()] + [c.clone() for c in case.caches])
    for other in results[1:]:
        for a, b in zip(results[0], other):
            assert torch.equal(a, b)
    case.check("front_gb_all", {})


@pytest.mark.gpu
def test_decode_stack_graph_steps_match_eager_and_reference(k):
    """P consecutive steps from zeroed caches, the position advanced on the device, captured once in a CUDA graph and replayed
    as decode.render_decoder does: the replays are bit-identical to eager steps, every step matches the rounded statement run
    step by step on its own caches, and the final caches match its k|v in every row."""
    dev = "cuda"
    B, P, cap, depth, S = 7, 40, 64, 4, 64
    torch.manual_seed(3)
    W = make_weights(depth, S, seed=77, dev=dev)
    layers, w_ada, b_ada = kernel_weights(W)
    caches = [torch.zeros(B, cap, 128, dtype=BF16, device=dev) for _ in range(depth)]
    plan = k.DecodeStackPlan(layers, w_ada, b_ada, caches, B, S, keep_hiddens=True)
    xs = torch.randn(B, P, D, device=dev)
    style_all = torch.randn(B, P + 1, S, device=dev)
    gb_all = plan.prepare_adaln(style_all)
    mask = torch.ones(B, cap, dtype=torch.uint8, device=dev)
    mask[1, 30:] = 0                             # padded tail
    mask[2, [3, 17, 18]] = 0                     # holes
    mask[3, 0] = 0
    x_buf = torch.empty(B, D, device=dev)
    pos_t = torch.zeros(1, dtype=torch.int64, device=dev)

    def step():
        k.gather_at_pos([xs], [x_buf], [0], pos_t)
        plan.step(x_buf, None, mask, pos_t, gb_all=gb_all, barrier_is_zero=True)
        plan.barrier.zero_()
        pos_t.add_(1)

    eager = []
    for _ in range(P):
        step()
        eager.append((plan.out.clone(), plan.hid.clone()))
    kv_eager = [c.clone() for c in caches]
    for c in caches:
        c.zero_()
    pos_t.zero_()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    replay = []
    for _ in range(P):
        graph.replay()
        replay.append((plan.out.clone(), plan.hid.clone()))
    torch.cuda.synchronize()
    assert int(pos_t) == P
    for (eo, eh), (ro, rh) in zip(eager, replay):
        assert torch.equal(eo, ro) and torch.equal(eh, rh)
    for c, ce in zip(caches, kv_eager):
        assert torch.equal(c, ce)
    kvd = [torch.zeros(B, cap, 128, dtype=F64, device=dev) for _ in range(depth)]
    worst = {}
    for t in range(P):
        kv_t, hid_t, out_t = ref_step(W, style_all[:, t + 1].double(), kvd, mask, xs[:, t].double(), t, rounded=True)
        for l in range(depth):
            kvd[l][:, t] = kv_t[l]
        for name, g, r in (("out", eager[t][0], out_t), ("hid", eager[t][1], hid_t)):
            e_rel, e_cos = _errs(g, r)
            worst[name + " rel"] = max(worst.get(name + " rel", 0.0), e_rel)
            worst[name + " cos"] = max(worst.get(name + " cos", 0.0), e_cos)
            assert e_rel < TIGHT_REL and e_cos < TIGHT_COS, (t, name, e_rel, e_cos)
    for l in range(depth):
        e_rel, e_cos = _errs(caches[l][:, :P], kvd[l][:, :P])
        worst["kv rel"] = max(worst.get("kv rel", 0.0), e_rel)
        assert e_rel < TIGHT_REL and e_cos < TIGHT_COS, (l, e_rel, e_cos)
        assert torch.equal(caches[l][:, P:], torch.zeros_like(caches[l][:, P:]))
    print("decode_stack graph steps: " + ", ".join(f"{n} {v:.2e}" for n, v in worst.items()))
