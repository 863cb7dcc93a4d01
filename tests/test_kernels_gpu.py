"""Per-kernel parity: every C-ABI entry point against a plain PyTorch fp32 statement of the same op (on the GPU)."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

BF16, F32 = torch.bfloat16, torch.float32


@pytest.fixture(scope="module")
def k():
    from scoreperformer_b200 import kernels
    return kernels


def rel_err(a, b):
    a, b = a.float(), b.float()
    return float((a - b).abs().max() / b.abs().max().clamp(min=1e-6))


def cos_dist(a, b):
    a, b = a.float().flatten(), b.float().flatten()
    return float(1 - torch.dot(a, b) / (a.norm() * b.norm()).clamp(min=1e-12))


def randn(*shape, dtype=F32, scale=1.0):
    return (torch.randn(*shape, device="cuda") * scale).to(dtype)


# ------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("M,N,K", [(257, 384, 256), (1022, 132, 128), (64, 1536, 512)])
def test_gemm_variants(k, ta, tb, M, N, K):
    torch.manual_seed(0)
    A, B = randn(M, K, dtype=BF16), randn(N, K, dtype=BF16)
    a = A.t().contiguous() if ta else A
    b = B.t().contiguous() if tb else B
    if (ta and M % 8) or (tb and N % 8):
        pytest.skip("MN-major operands need a 16-byte aligned row stride")
    ref = A.float() @ B.float().t()
    out = k.gemm(a, b, trans_a=bool(ta), trans_b=bool(tb), out_dtype=F32)
    assert rel_err(out, ref) < 2e-5
    bias, res = randn(N), randn(M, N)
    mask = torch.rand(M, device="cuda") > 0.3
    alpha = torch.tensor([0.37], device="cuda")
    out = k.gemm(a, b, trans_a=bool(ta), trans_b=bool(tb), bias=bias, residual=res, rowmask=mask, out_dtype=BF16, alpha=alpha)
    ref2 = (0.37 * ref + bias) * mask[:, None] + res
    assert rel_err(out, ref2) < 1e-2


def test_gemm_splitk_wgrad(k):
    torch.manual_seed(1)
    dy, x = randn(4090 * 2, 384, dtype=BF16), randn(4090 * 2, 256, dtype=BF16)
    ref = dy.float().t() @ x.float()
    out = k.gemm(dy, x, trans_a=True, trans_b=True, out_dtype=F32, split_k=0)
    assert rel_err(out, ref) < 1e-4
    out2 = k.gemm(dy, x, trans_a=True, trans_b=True, out=out.clone(), split_k=0, accumulate=True)
    assert rel_err(out2, 2 * ref) < 1e-4


@pytest.mark.parametrize("mode", [{"SPB_GEMM_EPI": "direct"}, {"SPB_GEMM_BN": "128"}])
def test_gemm_alternate_paths(k, mode, monkeypatch):
    """Forced tile widths and the direct (non-TMA) epilogue fallback must agree with the default path on every epilogue
    variant, including ragged M / N and split-K."""
    torch.manual_seed(7)
    cases = [(1000, 384, 256, False, False), (2048, 512, 512, False, True), (515, 256, 1024, False, False)]
    wg_dy, wg_x = randn(8200, 384, dtype=BF16), randn(8200, 256, dtype=BF16)
    outs = {}
    for tag in ("default", "alt"):
        if tag == "alt":
            for kk, vv in mode.items():
                monkeypatch.setenv(kk, vv)
        res = []
        for (M, N, K_, ta, tb) in cases:
            g = torch.Generator(device="cuda").manual_seed(M + N)
            A = torch.randn(M, K_, device="cuda", generator=g).to(BF16)
            B = torch.randn(N, K_, device="cuda", generator=g).to(BF16)
            b = B.t().contiguous() if tb else B
            bias = torch.randn(N, device="cuda", generator=g)
            resid = torch.randn(M, N, device="cuda", generator=g)
            mask = torch.rand(M, device="cuda", generator=g) > 0.3
            res.append(k.gemm(A, b, trans_b=tb, bias=bias, out_dtype=BF16))
            res.append(k.gemm(A, b, trans_b=tb, residual=resid, rowmask=mask, out_dtype=F32))
        res.append(k.gemm(wg_dy, wg_x, trans_a=True, trans_b=True, out_dtype=F32, split_k=0))
        outs[tag] = res
    for i, (d, a_) in enumerate(zip(outs["default"], outs["alt"])):
        tol = 1e-4 if i == len(outs["default"]) - 1 else 0.0      # split-K sums in a different order
        assert rel_err(a_, d) <= tol, (mode, i)
    ref = wg_dy.float().t() @ wg_x.float()
    assert rel_err(outs["alt"][-1], ref) < 1e-4


@pytest.mark.parametrize("B,T", [(3, 130), (2, 512)])
def test_gemm_rowdot_delta(k, B, T):
    """dO = dY Wo with the attention-backward delta = rowsum(dO * O) per head emitted by the same epilogue."""
    torch.manual_seed(8)
    H = 4
    dy, wo, o = randn(B * T, 256, dtype=BF16), randn(256, 256, dtype=BF16) * 0.1, randn(B * T, 256, dtype=BF16)
    do, delta = k.gemm_rowdot(dy, wo, o, T, H, trans_b=True)
    ref_do = dy.float() @ wo.float()
    assert torch.equal(do, k.gemm(dy, wo, trans_b=True, out_dtype=BF16))          # same values as the plain GEMM
    ref_delta = (ref_do * o.float()).view(B, T, H, 64).sum(-1).permute(0, 2, 1)
    assert delta.shape == (B, H, T) and rel_err(delta, ref_delta) < 2e-3


def test_gemm_strided_views(k):
    torch.manual_seed(2)
    big = randn(300, 1536, dtype=BF16)
    w = randn(165, 128, dtype=BF16)
    a = big[:, 256:384]
    out = k.gemm(a, w, out_dtype=F32)
    assert rel_err(out, a.float() @ w.float().t()) < 2e-5
    buf = torch.zeros(300, 512, dtype=BF16, device="cuda")
    k.gemm(a, randn(256, 128, dtype=BF16), out=buf[:, 256:])
    assert float(buf[:, :256].abs().max()) == 0 and float(buf[:, 256:].abs().max()) > 0


def test_cast_and_colsum(k):
    x = randn(777, 256)
    mask = torch.rand(777, device="cuda") > 0.5
    assert torch.equal(k.cast_bf16(x), x.to(BF16))
    assert torch.equal(k.cast_bf16(x, mask), (x * mask[:, None]).to(BF16))
    y = randn(3001, 507)
    assert rel_err(k.colsum(y), y.sum(0)) < 1e-5
    assert rel_err(k.colsum(y.to(BF16)), y.to(BF16).float().sum(0)) < 1e-5


# ------------------------------------------------------------------ LayerNorm
@pytest.mark.parametrize("dim,x_dtype,y_dtype,ada", [(256, F32, BF16, False), (256, F32, BF16, True), (256, F32, F32, False),
                                                     (1536, BF16, BF16, False), (256, BF16, BF16, False)])
def test_layer_norm(k, dim, x_dtype, y_dtype, ada):
    torch.manual_seed(3)
    n = 517
    x = randn(n, dim, dtype=x_dtype, scale=2.0) + 0.5
    w, b = randn(dim) * 0.2 + 1, randn(dim) * 0.1
    # adaptive form: `gb` holds (gamma - 1 | beta) -- gamma lives near 1 (layers.py:38-40) and bf16 keeps the deviation
    gb = (randn(n, 2 * dim) * 0.3 - 0.2).to(BF16) if ada else None
    xr = x.float().requires_grad_(True)
    if ada:
        gbr = gb.float().requires_grad_(True)
        ref = (1.0 + gbr[:, :dim]) * F.layer_norm(xr, (dim,)) + gbr[:, dim:]
    else:
        wr, br = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
        ref = F.layer_norm(xr, (dim,), wr, br)
    y, mean, rstd = k.layer_norm_fwd(x, None if ada else w, None if ada else b, gb, out_dtype=y_dtype)
    assert rel_err(y, ref) < (1e-5 if y_dtype == F32 else 1e-2)
    dy = randn(n, dim, dtype=BF16)
    dres = randn(n, dim)
    ref.backward(dy.float())
    if not ((x_dtype == F32 and not ada) or (x_dtype == F32 and ada) or x_dtype == BF16):
        return
    dx_dtype = F32 if (x_dtype == F32 and y_dtype == BF16) else (BF16 if x_dtype == BF16 else BF16)
    if ada:
        dgb = torch.empty(n, 2 * dim, dtype=BF16, device="cuda")
        dx = k.layer_norm_bwd(dy, x, mean, rstd, None, gb, dres=dres, dx_dtype=F32, dgb=dgb)
        assert rel_err(dx, xr.grad + dres) < 1e-4
        assert rel_err(dgb, gbr.grad) < 1e-2
    else:
        dw, db = torch.zeros(dim, device="cuda"), torch.zeros(dim, device="cuda")
        use_res = dx_dtype == F32
        dx = k.layer_norm_bwd(dy, x, mean, rstd, w, dres=dres if use_res else None, dx_dtype=dx_dtype, dw=dw, db=db)
        assert rel_err(dx, xr.grad + (dres if use_res else 0)) < (1e-4 if dx_dtype == F32 else 1e-2)
        assert rel_err(dw, wr.grad) < 1e-4 and rel_err(db, br.grad) < 1e-4


# ------------------------------------------------------------------ GLU
@pytest.mark.parametrize("H", [1024, 64])
def test_glu(k, H):
    torch.manual_seed(4)
    u = randn(333, 2 * H, dtype=BF16)
    ur = u.float().requires_grad_(True)
    a, g = ur.chunk(2, dim=-1)
    ref = a * F.silu(g)
    h = k.glu_fwd(u, 0.0, 0)
    assert rel_err(h, ref) < 1e-2
    dh = randn(333, H, dtype=BF16)
    ref.backward(dh.float())
    db = torch.zeros(2 * H, device="cuda")
    du = k.glu_bwd(dh, u, db, 0.0, 0)
    assert rel_err(du, ur.grad) < 1e-2
    assert rel_err(db, ur.grad.sum(0)) < 1e-2
    # dropout: same mask in forward and backward, keep-rate close to 1-p
    hd = k.glu_fwd(u, 0.25, 1234)
    kept = (hd != 0).float().mean()
    assert abs(float(kept) - 0.75) < 0.02
    dud = k.glu_bwd(dh, u, None, 0.25, 1234)
    m = (hd != 0)
    assert rel_err(dud[:, :H][m], (ur.grad[:, :H] / 0.75)[m]) < 2e-2
    assert float(dud[:, :H][~m & (ref != 0)].abs().max()) == 0


# ------------------------------------------------------------------ fused feed-forward sub-layer
@pytest.mark.parametrize("n", [128, 333, 4099, 32768])
def test_ffn_fused_forward(k, n):
    """spb_ffn_fwd (one tcgen05 kernel, u / h on chip) against the fp32 statement of feedforward.py:13-22,56-64 plus the residual,
    and against the unfused kernel chain it replaces: same side outputs u / h, same dropout mask."""
    torch.manual_seed(11)
    D, H = 256, 1024
    xn = randn(n, D, dtype=BF16)
    w1, b1, w2 = randn(2 * H, D, dtype=BF16, scale=D ** -0.5), randn(2 * H, scale=0.1), randn(D, H, dtype=BF16, scale=H ** -0.5)
    resid = randn(n, D)
    u_ref = xn.float() @ w1.float().t() + b1
    a, g = u_ref.chunk(2, dim=-1)
    h_ref = a * F.silu(g)
    ref = resid + h_ref @ w2.float().t()
    out, u, h = k.ffn_fwd(xn, w1, b1, w2, resid, 0.0, 0)
    assert rel_err(u, u_ref) < 1e-2 and rel_err(h, h_ref) < 1e-2
    assert rel_err(out, ref) < 1e-2
    out2, _, _ = k.ffn_fwd(xn, w1, b1, w2, None, 0.0, 0, save=False)
    assert rel_err(out2, ref - resid) < 1e-2
    # the unfused chain on the same inputs (its u is rounded to bf16 before the GLU; the fused kernel keeps fp32 there)
    u2 = k.gemm(xn, w1, bias=b1, out_dtype=BF16)
    h2 = k.glu_fwd(u2, 0.0, 0)
    out3 = k.gemm(h2, w2, residual=resid, out_dtype=F32)
    assert rel_err(u, u2) < 1e-2 and rel_err(out, out3) < 1e-2
    # dropout: the mask is the function spb_glu_fwd / spb_glu_bwd evaluate
    outd, ud, hd = k.ffn_fwd(xn, w1, b1, w2, resid, 0.25, 77)
    hd2 = k.glu_fwd(ud, 0.25, 77)
    assert torch.equal(hd == 0, hd2 == 0) and rel_err(hd, hd2) < 1e-2
    assert abs(float((hd != 0).float().mean()) - 0.75) < 0.02
    assert rel_err(outd, resid + hd.float() @ w2.float().t()) < 1e-2


@pytest.mark.parametrize("n", [256, 333, 4099, 32768])
@pytest.mark.parametrize("p_drop", [0.0, 0.25])
def test_ffn_fused_backward(k, n, p_drop):
    """spb_ffn_bwd (one tcgen05 kernel: dh on chip, du in place, dxn, bias gradient) against autograd of the fp32 statement of
    feedforward.py:13-22,56-64 with the kernel's own dropout mask, and against the unfused chain (gemm -> glu_bwd -> gemm)."""
    torch.manual_seed(13)
    D, H = 256, 1024
    dy = randn(n, D, dtype=BF16)
    u = randn(n, 2 * H, dtype=BF16)
    w1, w2 = randn(2 * H, D, dtype=BF16, scale=D ** -0.5), randn(D, H, dtype=BF16, scale=H ** -0.5)
    w2t = k.transpose_bf16(w2)
    assert torch.equal(w2t, w2.t().contiguous())
    keep = (k.glu_fwd(u, p_drop, 77) != 0) | (u[:, :H].float() * F.silu(u[:, H:].float()) == 0)     # the mask function of the forward
    ur = u.float().requires_grad_(True)
    a, g = ur.chunk(2, dim=-1)
    hr = a * F.silu(g) * keep / (1 - p_drop)
    hr.backward(dy.float() @ w2.float())
    du_ref = ur.grad
    db, db2 = torch.zeros(2 * H, device="cuda"), torch.zeros(2 * H, device="cuda")
    dxn, du = k.ffn_bwd(dy, w2t, w1, u, db, p_drop, 77, in_place=False)
    assert rel_err(du, du_ref) < 1e-2
    assert rel_err(dxn, du_ref @ w1.float()) < 1e-2
    assert rel_err(db, du_ref.sum(dim=0)) < 1e-2
    # the chain it replaces: same mask, same numbers up to the bf16 rounding of dh the fused kernel does not do
    dh = k.gemm(dy, w2, trans_b=True, out_dtype=BF16)
    du2 = k.glu_bwd(dh, u, db2, p_drop, 77)
    assert torch.equal(du == 0, du2 == 0) and rel_err(du, du2) < 1e-2
    assert rel_err(dxn, k.gemm(du2, w1, trans_b=True, out_dtype=BF16)) < 1e-2 and rel_err(db, db2) < 1e-2
    # in place: du over u, bias gradient accumulated on top of what is there
    u2 = u.clone()
    dxn3, du3 = k.ffn_bwd(dy, w2t, w1, u2, db, p_drop, 77)
    assert du3.data_ptr() == u2.data_ptr() and torch.equal(du3, du) and torch.equal(dxn3, dxn)
    assert rel_err(db, 2 * db2) < 1e-2


# ------------------------------------------------------------------ tuple embedding
@pytest.mark.parametrize("F_", [12, 10])
def test_embed_ln(k, F_):
    torch.manual_seed(5)
    sizes = [260, 132, 92, 132, 133, 125, 26, 69, 16, 16, 165, 85][:F_]
    n = 1000
    table = randn(sum(sizes), 128)
    tokens = torch.stack([torch.randint(0, v, (n,), device="cuda") for v in sizes], dim=-1)
    tokens[::7] = 0
    w, b = randn(F_ * 128) * 0.2 + 1, randn(F_ * 128) * 0.1
    tr = table.clone().requires_grad_(True)
    wr, br = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    offs = [0]
    for v in sizes[:-1]:
        offs.append(offs[-1] + v)
    parts = []
    for f in range(F_):
        blk = tr[offs[f]:offs[f] + sizes[f]]
        parts.append(F.embedding(tokens[:, f], blk, padding_idx=0))
    ref = F.layer_norm(torch.cat(parts, -1), (F_ * 128,), wr, br)
    out, mean, rstd = k.embed_ln_fwd(tokens, table, sizes, w, b)
    assert rel_err(out, ref) < 1e-2
    dy = randn(n, F_ * 128, dtype=BF16)
    ref.backward(dy.float())
    dtable, dw, db = torch.zeros_like(table), torch.zeros_like(w), torch.zeros_like(b)
    k.embed_ln_bwd(dy, tokens, table, sizes, w, mean, rstd, dtable, dw, db)
    assert rel_err(dtable, tr.grad) < 4e-3        # dx is rounded to bf16 (like dy itself) before the tensor-core scatter
    assert rel_err(dw, wr.grad) < 1e-4 and rel_err(db, br.grad) < 1e-4


# ------------------------------------------------------------------ attention
def ref_attention(qkv, mask, logslopes, B, T, H, causal):
    qkv = qkv.view(B, T, -1)
    q = qkv[..., :H * 64].view(B, T, H, 64).transpose(1, 2)
    kk, v = qkv[..., H * 64:H * 64 + 64], qkv[..., H * 64 + 64:]
    pos = torch.arange(T, device=qkv.device)
    bias = -(pos[None, :] - pos[:, None]).abs().float()[None] * logslopes.exp().view(H, 1, 1)
    allowed = mask[:, None, None, :].expand(B, 1, T, T)
    if causal:
        allowed = allowed & (pos[None, :] <= pos[:, None])[None, None]
    s = torch.einsum("bhid,bjd->bhij", q, kk) * 0.125 + bias[None]
    s = s.masked_fill(~allowed, -1e30)
    p = s.softmax(-1)
    return torch.einsum("bhij,bjd->bhid", p, v).transpose(1, 2).reshape(B * T, H * 64)


@pytest.mark.parametrize("impl", ["tcgen05", "mma"])
@pytest.mark.parametrize("B,T,causal", [(2, 64, False), (3, 47, True), (2, 200, False), (2, 511, True), (1, 130, True), (2, 511, False),
                                        (2, 2048, True), (1, 2048, False)])
def test_attention_fwd_bwd(k, B, T, causal, impl):
    """Both implementations (tcgen05/TMEM/TMA default, legacy mma.sync) against the fp32 statement of attend.py:58-126: ragged
    key-padding masks, causal and not, sequence lengths off the tile grid (47, 130, 511) and the long-context length."""
    torch.manual_seed(6)
    H = 4
    qkv = randn(B * T, H * 64 + 128, dtype=BF16)
    lengths = torch.randint(T // 2, T + 1, (B,), device="cuda")
    lengths[0] = T
    mask = torch.arange(T, device="cuda")[None] < lengths[:, None]
    logslopes = torch.log(torch.tensor([0.25, 0.0625, 0.015625, 0.00390625], device="cuda")) + 0.1
    qr = qkv.float().requires_grad_(True)
    lr = logslopes.clone().requires_grad_(True)
    ref = ref_attention(qr, mask, lr, B, T, H, causal)
    out, lse, aux = k.attention_fwd(qkv, mask, logslopes, B, T, H, causal, 0.0, 0, impl=impl)
    assert rel_err(out, ref) < 1.5e-2
    dout = randn(B * T, H * 64, dtype=BF16)
    ref.backward(dout.float())
    dls = torch.zeros(H, device="cuda")
    dqkv = k.attention_bwd(qkv, mask, logslopes, out, dout, lse, dls, B, T, H, causal, 0.0, 0, aux=aux)
    if impl == "tcgen05":      # the fp32 dQ accumulator must be handed back zeroed
        assert float(k._dq_accumulator(B * T, H * 64, qkv.device).abs().max()) == 0.0
    assert cos_dist(dqkv[:, :256], qr.grad[:, :256]) < 1e-3
    assert cos_dist(dqkv[:, 256:320], qr.grad[:, 256:320]) < 1e-3
    assert cos_dist(dqkv[:, 320:], qr.grad[:, 320:]) < 1e-3
    assert rel_err(dqkv, qr.grad) < 3e-2
    assert rel_err(dls, lr.grad) < 3e-2


@pytest.mark.parametrize("impl", ["tcgen05", "mma"])
def test_attention_dropout_consistency(k, impl):
    """Backward must regenerate the forward's dropout mask: finite-difference-free check via linearity in V."""
    torch.manual_seed(7)
    B, T, H = 2, 96, 4
    qkv = randn(B * T, H * 64 + 128, dtype=BF16)
    mask = torch.ones(B, T, dtype=torch.bool, device="cuda")
    ls = torch.log(torch.tensor([0.25, 0.0625, 0.015625, 0.00390625], device="cuda"))
    out, lse, aux = k.attention_fwd(qkv, mask, ls, B, T, H, False, 0.3, 99, impl=impl)
    out2, _, _ = k.attention_fwd(qkv, mask, ls, B, T, H, False, 0.3, 99, impl=impl)
    assert torch.equal(out, out2)
    out3, _, _ = k.attention_fwd(qkv, mask, ls, B, T, H, False, 0.3, 100, impl=impl)
    assert not torch.equal(out, out3)
    # O is linear in V: <dO, O> == <dV, V> when dO is the upstream gradient
    dout = randn(B * T, H * 64, dtype=BF16)
    dqkv = k.attention_bwd(qkv, mask, ls, out, dout, lse, torch.zeros(H, device="cuda"), B, T, H, False, 0.3, 99, aux=aux)
    lhs = float((dout.float() * out.float()).sum())
    rhs = float((dqkv[:, 320:].float() * qkv[:, 320:].float()).sum())
    assert abs(lhs - rhs) / abs(lhs) < 3e-2


# ------------------------------------------------------------------ latent levels
def test_latent_level(k):
    torch.manual_seed(8)
    B, T, D, z, col0 = 3, 70, 256, 8, 52
    hidden = randn(B, T, D)
    lengths = torch.tensor([70, 50, 61], device="cuda")
    mask = torch.arange(T, device="cuda")[None] < lengths[:, None]
    seg = 4 + torch.cumsum((torch.rand(B, T, device="cuda") < 0.4).long(), 1)
    seg = seg * mask
    S = T + 4
    style = torch.zeros(B, T, 64, device="cuda")
    style[..., :col0] = randn(B, T, col0) * mask[..., None]
    W, bias = randn(z, D + col0) * 0.1, randn(z) * 0.1
    hr, sr = hidden.clone().requires_grad_(True), style[..., :col0].clone().requires_grad_(True)
    Wr, br = W.clone().requires_grad_(True), bias.clone().requires_grad_(True)
    x = torch.cat([hr * mask[..., None], sr], -1)
    onehot = F.one_hot(seg, S).float()
    counts = onehot.sum(1).clamp(min=1)
    pooled = torch.einsum("bts,btd->bsd", onehot, x) / counts[..., None]
    lm = (pooled != 0).all(-1)
    lat_ref = (pooled @ Wr.t() + br) * lm[..., None]
    emb_ref = torch.gather(lat_ref, 1, seg[..., None].expand(-1, -1, z)) * mask[..., None]
    st = style.clone()
    lat, lmask, pooled_k, counts_k = k.latent_level_fwd(hidden, st, mask, seg, W, bias, col0, S, z)
    assert torch.equal(lmask, lm)
    assert torch.equal(counts_k.view(B, S).long(), onehot.sum(1).long())
    assert rel_err(lat, lat_ref) < 1e-5
    assert rel_err(st[..., col0:col0 + z], emb_ref) < 1e-5
    # backward
    d_emb, d_lat_direct = randn(B, T, z), randn(B, S, z)
    (emb_ref * d_emb).sum().add((lat_ref * d_lat_direct).sum()).backward()
    d_style = torch.zeros(B, T, 64, device="cuda")
    d_style[..., col0:col0 + z] = d_emb
    d_hidden = torch.zeros(B, T, D, device="cuda")
    dW, db = torch.zeros_like(W), torch.zeros_like(bias)
    k.latent_level_bwd(d_style, col0, d_lat_direct, mask, seg, W, pooled_k, counts_k, lmask, d_hidden, dW, db, S, z)
    assert rel_err(d_hidden, hr.grad) < 1e-4
    assert rel_err(d_style[..., :col0], sr.grad) < 1e-4
    assert rel_err(dW, Wr.grad) < 1e-4 and rel_err(db, br.grad) < 1e-4


def test_latent_level_mean_mode(k):
    torch.manual_seed(9)
    B, T, D, z = 2, 40, 256, 32
    hidden = randn(B, T, D)
    mask = torch.arange(T, device="cuda")[None] < torch.tensor([40, 25], device="cuda")[:, None]
    W, bias = randn(z, D) * 0.1, randn(z) * 0.1
    style = torch.zeros(B, T, 64, device="cuda")
    lat, lmask, _, _ = k.latent_level_fwd(hidden, style, mask, None, W, bias, 0, 2, z)
    pooled = (hidden * mask[..., None]).sum(1) / mask.sum(1, keepdim=True)
    ref = pooled @ W.t() + bias
    assert rel_err(lat[:, 1], ref) < 1e-5
    assert rel_err(style[..., :z], ref[:, None] * mask[..., None]) < 1e-5


@pytest.mark.parametrize("d,n_y", [(4, 700), (8, 300), (20, 129), (32, 5)])
def test_mmd(k, d, n_y):
    torch.manual_seed(10)
    z = randn(256, d)
    y = randn(n_y, d) * 0.7 + 0.2
    w = torch.rand(n_y, device="cuda") > 0.2
    yr = y.clone().requires_grad_(True)

    def kern(a, b):
        return torch.exp(-((a[:, None] - b[None]) ** 2).mean(-1) / d).mean()
    ys = yr[w]
    ref = kern(z, z) + kern(ys, ys) - 2 * kern(z, ys)
    ref.backward()
    loss, grad = k.mmd_fwd_bwd(z, y, w)
    assert abs(float(loss) - float(ref)) < 1e-5 + 1e-4 * abs(float(ref))
    assert rel_err(grad, yr.grad) < 1e-4


# ------------------------------------------------------------------ heads
@pytest.mark.parametrize("V", [132, 165, 85, 260])
def test_ce_rows(k, V):
    torch.manual_seed(11)
    n = 999
    logits = randn(n, V, scale=3.0)
    labels = torch.randint(4, V, (n,), device="cuda")
    labels[::3] = -100
    lr = logits.clone().requires_grad_(True)
    ref = F.cross_entropy(lr, labels, ignore_index=-100, reduction="sum")
    ref.backward()
    ls, cnt = torch.zeros(1, device="cuda"), torch.zeros(1, device="cuda")
    vpad = (V + 7) // 8 * 8
    dl = torch.empty(n, vpad, dtype=BF16, device="cuda")
    am = torch.empty(n, dtype=torch.int32, device="cuda")
    k.ce_rows(logits, labels, V, ls, cnt, dl, am)
    assert abs(float(ls) - float(ref)) / float(ref) < 1e-5
    assert int(cnt) == int((labels != -100).sum())
    assert rel_err(dl[:, :V], lr.grad) < 1e-2
    assert float(dl[:, V:].abs().max()) == 0 if vpad > V else True
    assert torch.equal(am.long(), logits.argmax(-1))


@pytest.mark.parametrize("V,n", [(132, 999), (125, 4096), (165, 130), (85, 777), (256, 300), (16, 64)])
def test_head_ce_fused(k, V, n):
    """Tied head + CE in one kernel (logits stay in TMEM) against torch: loss, count, gradient rows, argmax."""
    torch.manual_seed(13)
    e_all = randn(n, 3 * 128, dtype=BF16)                     # the field's 128 columns are a strided slice
    e = e_all[:, 128:256]
    table = (randn(V + 5, 128) * 0.3).to(BF16)[2:2 + V]     # row-offset slice of a bigger table
    labels2 = torch.randint(0, V, (n, 2), device="cuda")
    labels2[::3, 1] = -100
    labels = labels2[:, 1]
    logits = (e.float() @ table.float().t()).requires_grad_(True)
    ref = F.cross_entropy(logits, labels, ignore_index=-100, reduction="sum")
    ref.backward()
    ls, cnt = torch.zeros(1, device="cuda"), torch.zeros(1, device="cuda")
    vpad = (V + 7) // 8 * 8
    dl = torch.full((n, vpad), 7.0, dtype=BF16, device="cuda")
    am = torch.empty(n, dtype=torch.int32, device="cuda")
    k.head_ce(e, table, labels, ls, cnt, dl, am)
    assert abs(float(ls) - float(ref)) / abs(float(ref)) < 1e-4
    assert int(cnt) == int((labels != -100).sum())
    assert rel_err(dl[:, :V], logits.grad) < 1e-2
    if vpad > V:
        assert float(dl[:, V:].abs().max()) == 0
    top2 = logits.detach().topk(2, dim=-1).values
    clear = (top2[:, 0] - top2[:, 1]) > 1e-3                # argmax may differ only on near ties (fp32 accumulation order)
    assert torch.equal(am.long()[clear], logits.detach().argmax(-1)[clear])
    # loss only (inference / evaluation): no gradient buffer
    ls2, cnt2 = torch.zeros(1, device="cuda"), torch.zeros(1, device="cuda")
    k.head_ce(e, table, labels, ls2, cnt2)
    assert abs(float(ls2) - float(ls)) <= 1e-6 * abs(float(ls))


@pytest.mark.parametrize("world", [1, 4])
def test_adamw_flat_matches_torch(k, world):
    """csrc/optim.cu against clip_grad_norm_ + torch.optim.AdamW (the reference's Optimizer.step) over five steps."""
    torch.manual_seed(14)
    n = 40_008
    p0 = randn(n) * 0.1
    ref_p = torch.nn.Parameter(p0.clone())
    opt = torch.optim.AdamW([ref_p], lr=2e-3, weight_decay=1e-2, betas=(0.9, 0.99), eps=1e-8)
    p, m, v = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    shadow = torch.empty(n, dtype=BF16, device="cuda")
    step = torch.zeros(1, dtype=torch.int64, device="cuda")
    for it in range(5):
        g = randn(n) * (10.0 if it % 2 == 0 else 1e-3)           # alternately clipped / not clipped
        ref_p.grad = g.clone()
        torch.nn.utils.clip_grad_norm_([ref_p], 2.0)
        opt.step()
        g_sum = g * world                                       # what an all-reduce SUM over `world` ranks would hold
        norm = torch.linalg.vector_norm(g_sum)
        step.add_(1)
        k.adamw_step(p, g_sum, m, v, shadow, norm, step, lr=2e-3, betas=(0.9, 0.99), eps=1e-8, weight_decay=1e-2, max_norm=2.0,
                     grad_scale=1.0 / world)
        assert rel_err(p, ref_p.data) < 2e-6, it
        assert torch.equal(shadow, p.to(BF16))
    st = opt.state[ref_p]
    assert rel_err(m, st["exp_avg"]) < 1e-5 and rel_err(v, st["exp_avg_sq"]) < 1e-5


def test_clf_heads(k):
    torch.manual_seed(12)
    n, in_dim = 1500, 64
    ncls = [10, 3, 3, 14, 11, 2, 2, 2, 2]
    tot = sum(ncls)
    x = randn(n, in_dim)
    rowmask = torch.rand(n, device="cuda") > 0.3
    labels = torch.stack([torch.randint(0, c, (n,), device="cuda") for c in ncls], -1)
    W, b = randn(tot, in_dim) * 0.2, randn(tot) * 0.1
    cw = torch.rand(tot, device="cuda") + 0.5
    Wr, br = W.clone().requires_grad_(True), b.clone().requires_grad_(True)
    off, total = 0, 0
    per_head = []
    for g, c in enumerate(ncls):
        lg = x[rowmask] @ Wr[off:off + c].t() + br[off:off + c]
        l = F.cross_entropy(lg, labels[rowmask][:, g], weight=cw[off:off + c])
        per_head.append(l)
        total = total + l
        off += c
    loss_ref = total / len(ncls)
    loss_ref.backward()
    num, den = torch.zeros(len(ncls), device="cuda"), torch.zeros(len(ncls), device="cuda")
    k.clf_heads(x, rowmask, labels, W, b, cw, ncls, 0.0, 0, num=num, den=den)
    assert rel_err(num / den, torch.stack(per_head)) < 1e-5
    scale = (1.0 / len(ncls)) / den
    dW, db = torch.zeros_like(W), torch.zeros_like(b)
    k.clf_heads(x, rowmask, labels, W, b, cw, ncls, 0.0, 0, dlogit_scale=scale, dW=dW, db=db)
    assert rel_err(dW, Wr.grad) < 1e-4 and rel_err(db, br.grad) < 1e-4
    assert rel_err(k.clf_logits(x, W, b), x @ W.t() + b) < 1e-5


def test_table_build_matches_module_arithmetic():
    """Fused table kernel (forward + backward) against the per-field module arithmetic (the reference's token_weight + value MLP)."""
    from scoreperformer_b200 import fused
    from scoreperformer_b200.modules.transformer import DiscreteDenseContinuousEmbedding
    torch.manual_seed(13)
    sizes = [260, 16, 85]
    embs = torch.nn.ModuleDict()
    for i, v in enumerate(sizes):
        tv = [0.0] * 4 + torch.linspace(0, 1, v - 4).tolist()
        e = DiscreteDenseContinuousEmbedding(v, 128, discrete=False, continuous=True, discrete_ids=[0, 1, 2, 3], token_values=tv, padding_idx=0)
        for p_ in e.parameters():
            p_.data.normal_(0, 0.5)
        embs[f"f{i}"] = e
    embs = embs.cuda()
    ref = torch.cat([e.weight for e in embs.values()], 0)
    g = randn(sum(sizes), 128)
    ref.backward(g)
    ref_grads = [p_.grad.clone() for p_ in embs.parameters()]
    for p_ in embs.parameters():
        p_.grad = None
    consts, params = [], []
    for e in embs.values():
        consts += [e.token_values, e._discrete_mask]
        params += [e.index_weight, e.value_layer[0][0].weight, e.value_layer[0][0].bias, e.value_layer[1][0].weight, e.value_layer[1][0].bias]
    out = fused.TableBuildFn.apply(tuple(sizes), tuple(consts), *params)
    assert rel_err(out, ref) < 1e-5
    out.backward(g)
    for p_, want in zip(embs.parameters(), ref_grads):
        assert rel_err(p_.grad, want) < 1e-4


# ------------------------------------------------------------------ device-side collator
def test_unpack_batch_matches_reference_collator(k):
    """spb_unpack_batch: (1) the MixedLM masking is bit-exact against MixedLMPerformanceCollator.mask_sequence of the unmodified
    reference (golden vectors, three settings, ragged lengths, every special token); (2) pack -> copy -> unpack reproduces the
    int64 batch of the shapes the model consumes, bit for bit, including writing into preallocated (static-graph) tensors."""
    import numpy as np
    from tests import parity
    from scoreperformer_b200.data import PackedBatchSpec, pack_batch, unpack_batch
    g = parity.golden("collator_mixlm.npz")
    seq = torch.from_numpy(g["seq"])
    lengths = torch.from_numpy(g["lengths"]).to(torch.int32)
    specs = {"recipe": PackedBatchSpec(),
             "all_dims": PackedBatchSpec(mask_ignore_token_ids=(0, 3), mask_ignore_token_dims=(), label_pad_ignored_dims=False),
             "keep_labels": PackedBatchSpec(mask_ignore_token_dims=(0, 5), label_pad_ignored_dims=False)}
    for tag, spec in specs.items():
        packed = {"perf": seq.to(torch.int32).to(torch.uint16).cuda(), "perf_len": lengths.cuda()}
        out = unpack_batch(packed, spec)
        assert torch.equal(out["perf"].cpu(), seq), tag
        assert torch.equal(out["masked_perf"].cpu(), torch.from_numpy(g[f"{tag}/masked"])), tag
        assert torch.equal(out["labels"].cpu(), torch.from_numpy(g[f"{tag}/labels"])), tag
        assert torch.equal(out["perf_mask"].cpu(), torch.arange(seq.shape[1])[None] < lengths[:, None]), tag
    for B, T in ((3, 33), (64, 512)):
        batch = parity.make_batch(B, T, seed=21)
        packed = {kk: v.cuda() for kk, v in pack_batch(batch, check=True).items()}
        got = unpack_batch(packed)
        assert set(got) == set(batch)
        for name, want in batch.items():
            assert got[name].dtype == want.dtype and torch.equal(got[name].cpu(), want), name
        static = {kk: torch.zeros_like(v, device="cuda") for kk, v in batch.items()}
        unpack_batch(packed, out=static)
        for name, want in batch.items():
            assert torch.equal(static[name].cpu(), want), name


# ------------------------------------------------------------------ heads + sampling of the rendered fields
def test_sample_fields_greedy_and_topk(k):
    """spb_sample_fields: k = 1 is torch.argmax of the fp32 statement of the tied head (PAD / MASK banned); k > 1 only ever draws
    from the k largest logits, every one of them, with frequencies that follow the softmax at the temperature."""
    torch.manual_seed(12)
    B, T, F_ = 64, 6, 12
    sizes = [260, 132, 92, 132, 133, 125, 26, 69, 16, 16, 165, 85]
    offs = [0]
    for v in sizes[:-1]:
        offs.append(offs[-1] + v)
    fields = [3, 5, 10, 11]
    table = randn(sum(sizes), 128, dtype=BF16, scale=0.3)
    e = randn(B, F_ * 128, dtype=BF16)
    tokens = torch.zeros(B, T, F_, dtype=torch.int64, device="cuda")
    pos = torch.tensor([2], device="cuda")
    logits = {f: e[:, f * 128:(f + 1) * 128].float() @ table[offs[f]:offs[f] + sizes[f]].float().t() for f in fields}
    for f in fields:
        logits[f][:, :2] = -float("inf")
    k.sample_fields(e, table, fields, [offs[f] for f in fields], [sizes[f] for f in fields], [1] * 4, tokens, pos)
    for f in fields:
        top2 = logits[f].topk(2, dim=-1).values
        clear = (top2[:, 0] - top2[:, 1]) > 1e-3                    # bf16 products summed in a different order: skip numerical ties
        assert torch.equal(tokens[clear, 3, f], logits[f].argmax(-1)[clear]), f
    assert int(tokens[:, :3].abs().sum()) == 0 and int(tokens[:, 4:].abs().sum()) == 0
    untouched = [f for f in range(F_) if f not in fields]
    assert int(tokens[:, 3, untouched].abs().sum()) == 0
    # top-k sampling: one row repeated, many seeds
    kk, temp, n_draw = 5, 0.7, 4096
    e1 = e[:1].repeat(n_draw, 1).contiguous()
    tok = torch.zeros(n_draw, T, F_, dtype=torch.int64, device="cuda")
    for rep in range(4):
        k.sample_fields(e1, table, fields, [offs[f] for f in fields], [sizes[f] for f in fields], [kk] * 4, tok, pos, temperature=temp, seed=1000 + rep)
        for f in fields:
            val, ind = logits[f][0].topk(kk)
            drawn = tok[:, 3, f]
            assert bool(torch.isin(drawn, ind).all()), f
            want = torch.softmax(val / temp, -1)
            got = torch.stack([(drawn == i).float().mean() for i in ind])
            assert float((got - want).abs().max()) < 0.04, (f, got.tolist(), want.tolist())


# ------------------------------------------------------------------ multi-buffer helpers
def test_multi_add_copy_gather(k):
    """spb_multi_add_f32 / spb_multi_copy / spb_gather_at_pos: many small adds / copies / position gathers in one launch each."""
    torch.manual_seed(1)
    sizes = [5, 512 * 64, 512, 7 * 13, 100003] + [33] * 60           # more pairs than one launch holds (48)
    dst = [randn(n) for n in sizes]
    src = [randn(n) for n in sizes]
    want = [d + s_ for d, s_ in zip(dst, src)]
    k.multi_add(dst, src)
    assert all(torch.equal(a, b) for a, b in zip(dst, want))
    # copies: mixed dtypes, odd byte counts, an unaligned view
    base = torch.arange(1000, device="cuda", dtype=torch.uint8)
    srcs = [torch.randint(0, 1000, (64, 512, 12), device="cuda"), torch.rand(7, device="cuda") > 0.5, randn(33, 3, dtype=BF16), base[3:990]]
    dsts = [torch.zeros_like(t) for t in srcs[:3]] + [torch.zeros(987, device="cuda", dtype=torch.uint8)]
    k.multi_copy(dsts, srcs)
    assert all(torch.equal(a, b) for a, b in zip(dsts, srcs))
    # gather at a device-side position, with shifts and clamping at the sequence end
    B, T = 5, 9
    a, b_, c = torch.randint(0, 99, (B, T, 12), device="cuda"), randn(B, T, 256), randn(B, T, 64)
    oa, ob, oc = torch.empty((B, 12), dtype=a.dtype, device="cuda"), torch.empty((B, 256), device="cuda"), torch.empty((B, 64), device="cuda")
    for pos in (0, 3, T - 1):
        pos_t = torch.tensor([pos], device="cuda")
        k.gather_at_pos([a, b_, c], [oa, ob, oc], [0, 1, 1], pos_t)
        nxt = min(pos + 1, T - 1)
        assert torch.equal(oa, a[:, pos]) and torch.equal(ob, b_[:, nxt]) and torch.equal(oc, c[:, nxt])

