"""Thin tensor-level wrappers over the C ABI (include/spb200.h).  No math happens in Python here.

Every wrapper launches on torch's current CUDA stream and bumps `LAUNCHES` by the number of kernels the
entry point launches, so bench.py can report `gpu_launches`.
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import ctypes
import torch
from torch import Tensor

from . import lib as _lib

BF16, F32 = torch.bfloat16, torch.float32
LAUNCHES = 0
# Optional device-side uint64 counter mixed into every dropout seed (set by train_step.TrainStep): kernels captured in a CUDA
# graph read it at run time, so replays draw fresh masks although the host-side seeds were baked in at capture.
RNG_OFFSET: Optional[Tensor] = None
# "tcgen05" (TMEM/TMA forward + backward kernels, need 4 heads) or "mma" (legacy mma.sync kernels); SPB_ATTN overrides.
import os as _os
ATTENTION_IMPL = _os.environ.get("SPB_ATTN", "tcgen05")


def _count(n: int = 1) -> None:
    global LAUNCHES
    LAUNCHES += n


def _p(t: Optional[Tensor]):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _require_cuda(*ts: Optional[Tensor]) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("scoreperformer_b200 kernels need CUDA tensors: there is no CPU fallback")


def _call(name: str, *args) -> None:
    fn = getattr(_lib.lib(), name)
    _lib.check(fn(*args), name)


def seed_from_torch() -> int:
    """Draw a 63-bit dropout seed from torch's CPU generator (so torch.manual_seed governs the masks)."""
    return int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())


# ----------------------------------------------------------------------------- elementwise helpers
def cast_bf16(x: Tensor, rowmask: Optional[Tensor] = None, out: Optional[Tensor] = None) -> Tensor:
    """fp32 -> bf16 copy; rows (last dim) where rowmask is False are zeroed."""
    _require_cuda(x)
    if x.dtype == BF16 and rowmask is None:
        return x
    assert x.dtype == F32 and x.is_contiguous(), (x.dtype, x.is_contiguous())
    if out is None:
        out = torch.empty(x.shape, dtype=BF16, device=x.device)
    row_len = x.shape[-1] if rowmask is not None else 0
    _call("spb_cast_f32_bf16", _p(x), _p(out), x.numel(), _p(rowmask), row_len, _stream())
    _count()
    return out


def colsum(x: Tensor, out: Optional[Tensor] = None) -> Tensor:
    """out[c] += sum_r x[r, c] (fp32 accumulate)."""
    _require_cuda(x)
    assert x.dim() == 2 and x.stride(1) == 1
    if out is None:
        out = torch.zeros(x.shape[1], dtype=F32, device=x.device)
    _call("spb_colsum", _p(x), int(x.dtype == F32), x.stride(0), _p(out), x.shape[0], x.shape[1], _stream())
    _count()
    return out


# ----------------------------------------------------------------------------- GEMM
def gemm(a: Tensor, b: Tensor, *, trans_a: bool = False, trans_b: bool = False, bias: Optional[Tensor] = None,
         residual: Optional[Tensor] = None, rowmask: Optional[Tensor] = None, out: Optional[Tensor] = None,
         out_dtype: torch.dtype = BF16, split_k: int = 1, accumulate: bool = False, alpha: Optional[Tensor] = None) -> Tensor:
    """C = op(A) op(B)^T with the fused epilogue of spb_gemm_bf16.

    a: [M,K] (or [K,M] when trans_a), b: [N,K] (or [K,N] when trans_b); both bf16 with unit inner stride.
    """
    _require_cuda(a, b)
    assert a.dtype == BF16 and b.dtype == BF16 and a.dim() == 2 and b.dim() == 2
    assert a.stride(1) == 1 and b.stride(1) == 1
    if trans_a:
        K, M = a.shape
    else:
        M, K = a.shape
    if trans_b:
        Kb, N = b.shape
    else:
        N, Kb = b.shape
    assert K == Kb, f"gemm: inner dims differ ({K} vs {Kb})"
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=a.device)
        if accumulate:
            out.zero_()
    assert out.shape == (M, N) and out.stride(1) == 1 and out.dtype in (BF16, F32)
    if residual is not None:
        assert residual.dtype == F32 and residual.shape == (M, N) and residual.stride(1) == 1
    if bias is not None:
        assert bias.dtype == F32 and bias.numel() == N
    _call("spb_gemm_bf16", _p(a), _p(b), _p(out), M, N, K, int(trans_a), int(trans_b), a.stride(0), b.stride(0), out.stride(0),
          _p(bias), _p(residual), residual.stride(0) if residual is not None else 0, _p(rowmask), int(out.dtype == F32),
          split_k, int(accumulate), _p(alpha), _stream())
    _count()
    return out


# ----------------------------------------------------------------------------- LayerNorm
def layer_norm_fwd(x: Tensor, w: Optional[Tensor], b: Optional[Tensor], gb: Optional[Tensor] = None,
                   out: Optional[Tensor] = None, out_dtype: torch.dtype = BF16, eps: float = 1e-5, need_stats: bool = True):
    """x [n, dim] (fp32 or bf16, unit inner stride) -> (y, mean, rstd)."""
    _require_cuda(x)
    assert x.dim() == 2 and x.stride(1) == 1
    n, dim = x.shape
    if out is None:
        out = torch.empty((n, dim), dtype=out_dtype, device=x.device)
    mean = torch.empty(n, dtype=F32, device=x.device) if need_stats else None
    rstd = torch.empty(n, dtype=F32, device=x.device) if need_stats else None
    _call("spb_layer_norm_fwd", _p(x), int(x.dtype == F32), x.stride(0), _p(w), _p(b), _p(gb), gb.stride(0) if gb is not None else 0,
          _p(out), int(out.dtype == F32), out.stride(0), _p(mean), _p(rstd), n, dim, float(eps), _stream())
    _count()
    return out, mean, rstd


def layer_norm_bwd(dy: Tensor, x: Tensor, mean: Tensor, rstd: Tensor, w: Optional[Tensor], gb: Optional[Tensor] = None,
                   dres: Optional[Tensor] = None, dx_dtype: torch.dtype = F32, dw: Optional[Tensor] = None,
                   db: Optional[Tensor] = None, dgb: Optional[Tensor] = None, want_dx16: bool = False,
                   dx16_rowmask: Optional[Tensor] = None):
    """Returns dx (or (dx, dx16) with want_dx16: a bf16, optionally row-masked copy); dw/db (fp32 [dim]) are accumulated into,
    dgb (bf16 view [n, 2*dim]) is written."""
    _require_cuda(dy, x)
    assert dy.dtype == BF16 and dy.stride(1) == 1 and x.stride(1) == 1
    n, dim = x.shape
    dx = torch.empty((n, dim), dtype=dx_dtype, device=x.device)
    dx16 = torch.empty((n, dim), dtype=BF16, device=x.device) if want_dx16 else None
    _call("spb_layer_norm_bwd", _p(dy), dy.stride(0), _p(x), int(x.dtype == F32), x.stride(0), _p(mean), _p(rstd), _p(w), _p(gb),
          gb.stride(0) if gb is not None else 0, _p(dres), dres.stride(0) if dres is not None else 0, _p(dx), int(dx.dtype == F32),
          dx.stride(0), _p(dw), _p(db), _p(dgb), dgb.stride(0) if dgb is not None else 0, _p(dx16), dim if want_dx16 else 0,
          _p(dx16_rowmask), n, dim, _stream())
    _count()
    return (dx, dx16) if want_dx16 else dx


# ----------------------------------------------------------------------------- persistent decode step
class DecodeStackPlan:
    """Pointer table + scratch of `spb_decode_stack_step` for one (stack, batch, cache) -- built once per decode session."""

    def __init__(self, layers, w_ada: Tensor, b_ada: Tensor, kv_caches, B: int, style_dim: int, keep_hiddens: bool = False,
                 advance: Optional[Tensor] = None):
        import ctypes
        dev = w_ada.device
        self.depth, self.B, self.S, self.cap = len(layers), B, style_dim, kv_caches[0].shape[1]
        self.w_ada, self.b_ada = w_ada, b_ada
        self._keep = [layers, kv_caches]                       # keep the tensors alive as long as the pointers are used
        ptrs = []
        self._transposed = []
        for w, kv in zip(layers, kv_caches):
            assert kv.dtype == BF16 and kv.is_contiguous() and kv.shape == (B, self.cap, 128)
            wqkv_t, wo_t = w["wqkv"].t().contiguous(), w["wo"].t().contiguous()      # input-major copies for the per-row products
            self._transposed += [wqkv_t, wo_t]
            for t in (w["wqkv"], w["wo"], w["ls"], w["w1"], w["b1"], w["w2"], kv, wqkv_t, wo_t):
                assert t.is_contiguous()
                ptrs.append(t.data_ptr())
        self.ptrs = (ctypes.c_void_p * len(ptrs))(*ptrs)
        n_norms = 2 * self.depth + 1
        self.gb = torch.empty((B, n_norms * 512), dtype=BF16, device=dev)
        self.qkv = torch.empty((B, 384), dtype=BF16, device=dev)
        self.o = torch.empty((B, 256), dtype=BF16, device=dev)
        self.hmid = torch.empty((B, 1024), dtype=BF16, device=dev)
        self.xres = torch.empty((B, 256), dtype=F32, device=dev)
        self.hid = torch.empty((self.depth, B, 256), dtype=F32, device=dev) if keep_hiddens else None
        self.out = torch.empty((B, 256), dtype=F32, device=dev)
        self.out16 = torch.empty((B, 256), dtype=BF16, device=dev)          # bf16 copy of `out`: the head projection's operand
        self._no_style = torch.zeros((B, style_dim), dtype=F32, device=dev)   # placeholder when the AdaLN terms are prepared ahead
        self._front = None
        # [CTA counter of sample_fields, grid-barrier word]; a render session passes its own, which session_begin clears every call
        if advance is None:
            advance = torch.zeros(2, dtype=torch.int32, device=dev)
        assert advance.dtype == torch.int32 and advance.shape == (2,) and advance.is_contiguous()
        self.advance = advance
        self.barrier = self.advance[1:]

    def set_kv(self, kv_caches) -> None:
        """Point the plan at another set of KV buffers of the same shape (the buffer sets of a render session)."""
        assert len(kv_caches) == self.depth
        for l, kv in enumerate(kv_caches):
            assert kv.dtype == BF16 and kv.is_contiguous() and kv.shape == (self.B, self.cap, 128)
            self.ptrs[9 * l + 6] = kv.data_ptr()
        self._keep[1] = kv_caches

    def prepare_adaln(self, style_all: Tensor) -> Tensor:
        """(gamma-1 | beta) rows of every AdaLN for ALL positions, style_all fp32 [B, T, S] -> bf16 [B, T, (2*depth+1)*512]: one
        large GEMM before a rendering loop instead of a tile phase in every note-step (pass the result as `gb_all` to step())."""
        B, T, S = style_all.shape
        assert B == self.B and S == self.S
        s16 = cast_bf16(style_all.reshape(B * T, S).contiguous())
        return gemm(s16, self.w_ada, bias=self.b_ada, out_dtype=BF16).view(B, T, -1)

    def set_front(self, x1: Tensor, w_front: Tensor, p2: Tensor, ln_w: Tensor, ln_b: Tensor, wc_t: Tensor, c2: Tensor) -> None:
        """Let step() evaluate the input front of the rendering loop itself: x = LN(x1 w_front^T + p2) wc_t + c2 (static buffers:
        x1 bf16 [B, 1536], p2 / c2 fp32 [B, 256] are refilled by the caller before every step)."""
        B = self.B
        assert x1.dtype == BF16 and x1.shape == (B, 1536) and x1.is_contiguous() and w_front.dtype == BF16 and w_front.shape == (256, 1536)
        assert w_front.is_contiguous() and wc_t.dtype == BF16 and wc_t.shape == (256, 256) and wc_t.is_contiguous()
        for t in (p2, c2):
            assert t.dtype == F32 and t.shape == (B, 256) and t.is_contiguous()
        for t in (ln_w, ln_b):
            assert t.dtype == F32 and t.numel() == 256 and t.is_contiguous()
        self._front_te = torch.empty((B, 256), dtype=F32, device=x1.device)
        self._front_keep = (x1, w_front, p2, self._front_te, ln_w, ln_b, wc_t, c2)
        self._front = _ptr_array(self._front_keep)

    def step(self, x: Optional[Tensor], style: Optional[Tensor], key_mask: Optional[Tensor], pos_dev: Tensor, eps: float = 1e-5,
             gb_all: Optional[Tensor] = None, use_front: bool = False, barrier_is_zero: bool = False) -> Tensor:
        front = self._front if use_front else None
        assert front is not None or (x is not None and x.dtype == F32 and x.is_contiguous() and x.shape == (self.B, 256))
        if gb_all is not None:
            assert gb_all.dtype == BF16 and gb_all.is_contiguous() and gb_all.shape[0] == self.B and gb_all.shape[2] == self.gb.shape[1]
            style = self._no_style if style is None else style
        assert style.dtype == F32 and style.is_contiguous() and style.shape == (self.B, self.S)
        assert pos_dev.dtype == torch.int64 and pos_dev.is_cuda
        assert key_mask is None or (key_mask.is_contiguous() and key_mask.shape == (self.B, self.cap))
        _call("spb_decode_stack_step", _p(x), _p(style), self.S, _p(self.w_ada), _p(self.b_ada), self.ptrs, self.depth, _p(key_mask),
              _p(pos_dev), self.B, self.cap, _p(self.gb), _p(self.qkv), _p(self.o), _p(self.hmid), _p(self.xres), _p(self.hid),
              _p(self.out), _p(self.out16), _p(self.barrier), float(eps), _p(gb_all), gb_all.shape[1] if gb_all is not None else 0,
              front, int(barrier_is_zero), _stream())
        _count()
        return self.out


def gather_at_pos(srcs: Sequence[Tensor], dsts: Sequence[Tensor], shifts: Sequence[int], pos_dev: Tensor) -> None:
    """dst_k[b] = src_k[b, pos + shift_k] for contiguous [B, T, ...] sources and [B, ...] destinations, ONE launch (the position is
    read on the device, so the launch can be replayed from a CUDA graph)."""
    _require_cuda(*srcs, *dsts)
    B, T = srcs[0].shape[0], srcs[0].shape[1]
    rows = []
    for s_, d in zip(srcs, dsts):
        assert s_.is_contiguous() and d.is_contiguous() and s_.shape[0] == B and s_.shape[1] == T and d.shape[0] == B
        assert s_.dtype == d.dtype and s_[0, 0].numel() == d[0].numel()
        rows.append(d[0].numel() * d.element_size())
    assert pos_dev.dtype == torch.int64 and pos_dev.is_cuda
    n = len(srcs)
    _call("spb_gather_at_pos", _ptr_array(srcs), _ptr_array(dsts), (ctypes.c_int * n)(*rows), (ctypes.c_int * n)(*[int(v) for v in shifts]),
          n, _p(pos_dev), B, T, _stream())
    _count()


def sample_fields(e: Tensor, table16: Tensor, fields: Sequence[int], offsets: Sequence[int], vocab: Sequence[int], topk: Sequence[int],
                  tokens: Tensor, pos_dev: Tensor, temperature: float = 1.0, seed: int = 0, n_banned: int = 2,
                  advance: Optional[Tensor] = None, top_p: Optional[Sequence[float]] = None,
                  top_a: Optional[Sequence[Optional[Tuple[float, float]]]] = None,
                  banned: Optional[Sequence[Sequence[int]]] = None) -> None:
    """Heads of `fields` + top-k sampling (k = 1: greedy) + write of tokens[:, pos + 1, field], one launch (csrc/decode_stack.cu).
    `advance` (int32 [2], [0] zero): the last CTA also does pos += 1 and clears both words (DecodeStackPlan.barrier is laid out so that
    advance[1] is the stack kernel's grid-barrier word).
    Per field (one entry per listed field; None = off for all): `top_p` thresholds (None or < 0: off), `top_a` (min_p_pow,
    min_p_ratio) pairs (None: off) and `banned` token ids never emitted besides [0, n_banned).  A field with a top-p / top-a filter
    ignores its k.  Without any of the three this is exactly the spb_sample_fields call."""
    import ctypes
    _require_cuda(e, table16, tokens)
    assert e.dtype == BF16 and e.stride(1) == 1 and table16.dtype == BF16 and table16.is_contiguous() and table16.shape[1] == 128
    assert tokens.dtype == torch.int64 and tokens.is_contiguous() and tokens.dim() == 3 and pos_dev.dtype == torch.int64
    n = len(fields)
    arr = lambda xs: (ctypes.c_int * n)(*[int(x) for x in xs])
    B, T, F = tokens.shape
    args = (_p(e), e.stride(0), _p(table16), arr(fields), arr(offsets), arr(vocab), arr(topk), n, int(n_banned), float(temperature),
            int(seed), _p(pos_dev), _p(tokens), B, T, F, _p(advance))
    if top_p is None and top_a is None and banned is None:
        _call("spb_sample_fields", *args, _stream())
    else:
        farr = lambda xs: None if xs is None else (ctypes.c_float * n)(*[float(x) for x in xs])
        assert all(len(x) == n for x in (top_p, top_a, banned) if x is not None)
        pp = None if top_p is None else [-1.0 if t is None else t for t in top_p]
        a_pow = None if top_a is None else [0.0 if a is None else a[0] for a in top_a]
        a_ratio = None if top_a is None else [0.0 if a is None else a[1] for a in top_a]
        bits = None
        if banned is not None:
            words = [0] * (8 * n)
            for i, ids in enumerate(banned):
                for v in ids:
                    v = int(v)
                    assert 0 <= v < 256, f"banned token {v} is outside 0..255"
                    words[8 * i + v // 32] |= 1 << (v % 32)
            bits = (ctypes.c_uint32 * (8 * n))(*words)
        _call("spb_sample_fields_filtered", *args, farr(pp), farr(a_pow), farr(a_ratio), bits, _stream())
    _count()


def fingerprint_table(tensors: Sequence[Tensor]) -> Tensor:
    """The [n, 3] int64 table session_begin hashes: (address, number of 32-bit words, index of the first word) per tensor, in order.
    Returned on the tensors' device.  Every tensor must be contiguous and a whole number of 4-byte-aligned words."""
    rows, first = [], 0
    for t in tensors:
        nbytes = t.numel() * t.element_size()
        if not t.is_contiguous() or nbytes % 4 or t.data_ptr() % 4:
            raise ValueError(f"fingerprint_table: needs contiguous tensors of whole 32-bit words, got {t.dtype} {tuple(t.shape)}")
        rows.append((t.data_ptr(), nbytes // 4, first))
        first += nbytes // 4
    return torch.tensor(rows, dtype=torch.int64).reshape(-1, 3).to(tensors[0].device if len(tensors) else "cpu")


def session_begin(table: Tensor, state: Tensor, advance: Tensor, pos_dev: Tensor, start: int) -> None:
    """One launch at the start of a render session's call (csrc/decode_stack.cu): fingerprint of the tensors in `table`
    (fingerprint_table) -> state[0], state[3] = 1 if it differs from the state[0] stored before, else 0; advance[:] = 0; pos_dev = start.
    state: int64 [4] (the kernel works on it as uint64), [1] and [2] zero between launches."""
    _require_cuda(table, state, advance, pos_dev)
    assert table.dtype == torch.int64 and table.dim() == 2 and table.shape[1] == 3 and table.is_contiguous()
    assert state.dtype == torch.int64 and state.shape == (4,) and state.is_contiguous()
    assert advance.dtype == torch.int32 and advance.shape == (2,) and pos_dev.dtype == torch.int64 and pos_dev.numel() == 1
    _call("spb_session_begin", _p(table), table.shape[0], _p(state), _p(advance), _p(pos_dev), int(start), _stream())
    _count()


def decode_stack_ok(depth: int, dim: int, heads: int, hidden: int, ada: bool, style_dim: int, cap: int) -> bool:
    return (ada and dim == 256 and heads == 4 and hidden == 1024 and 1 <= depth <= 8 and style_dim % 16 == 0 and 16 <= style_dim <= 256
            and cap <= 2048)


# ----------------------------------------------------------------------------- collator (device side)
def unpack_batch(perf, score, segs, dirs, perf_len, score_len, o_perf, o_masked, o_labels, o_score, o_segs, o_dirs, o_perf_mask,
                 o_score_mask, B: int, T: int, Fp: int, Fs: int, Fd: int, ignore_dims: int, ignore_ids: int, mask_token: int,
                 label_pad: int, label_pad_ignored_dims: bool) -> None:
    """Packed batch -> int64 model inputs + MixedLM masking, one launch (csrc/collate.cu; data/packed.py builds the arguments)."""
    _require_cuda(perf, o_perf)
    assert perf.dtype == torch.uint16 and perf_len.dtype == torch.int32 and o_perf.dtype == torch.int64
    assert score is None or score.dtype == torch.uint16
    assert segs is None or (segs.dtype == torch.int32 and segs.is_contiguous())
    assert dirs is None or dirs.dtype == torch.uint8
    _call("spb_unpack_batch", _p(perf), _p(score), _p(segs), _p(dirs), _p(perf_len), _p(score_len), _p(o_perf), _p(o_masked),
          _p(o_labels), _p(o_score), _p(o_segs), _p(o_dirs), _p(o_perf_mask), _p(o_score_mask), B, T, Fp, Fs, Fd, int(ignore_dims),
          int(ignore_ids), int(mask_token), int(label_pad), int(bool(label_pad_ignored_dims)), _stream())
    _count()


# ----------------------------------------------------------------------------- GLU
def glu_fwd(u: Tensor, dropout_p: float, seed: int) -> Tensor:
    _require_cuda(u)
    assert u.dtype == BF16 and u.is_contiguous()
    n, two_h = u.shape
    h = torch.empty((n, two_h // 2), dtype=BF16, device=u.device)
    _call("spb_glu_fwd", _p(u), _p(h), n, two_h // 2, float(dropout_p), seed, _p(RNG_OFFSET), _stream())
    _count()
    return h


def ffn_fwd(xn: Tensor, w1: Tensor, b1: Tensor, w2: Tensor, resid: Optional[Tensor], dropout_p: float, seed: int,
            save: bool = True):
    """Fused feed-forward sub-layer (one tcgen05 kernel): resid + W2 . dropout(GLU(xn W1^T + b1)).
    xn bf16 [n, 256]; w1 bf16 [2048, 256]; b1 fp32 [2048]; w2 bf16 [256, 1024]; resid fp32 [n, 256] or None.
    Returns (out fp32 [n, 256], u bf16 [n, 2048] or None, h bf16 [n, 1024] or None): u / h are what the backward consumes."""
    _require_cuda(xn, w1, w2)
    n, dim = xn.shape
    hidden = w2.shape[1]
    assert xn.dtype == BF16 and w1.dtype == BF16 and w2.dtype == BF16 and b1.dtype == F32 and xn.stride(1) == 1
    assert w1.is_contiguous() and w2.is_contiguous() and w1.shape == (2 * hidden, dim) and w2.shape == (dim, hidden)
    out = torch.empty((n, dim), dtype=F32, device=xn.device)
    u = torch.empty((n, 2 * hidden), dtype=BF16, device=xn.device) if save else None
    h = torch.empty((n, hidden), dtype=BF16, device=xn.device) if save else None
    if resid is not None:
        assert resid.dtype == F32 and resid.stride(1) == 1
    _call("spb_ffn_fwd", _p(xn), xn.stride(0), _p(w1), _p(b1), _p(w2), _p(resid), resid.stride(0) if resid is not None else 0, _p(out),
          out.stride(0), _p(u), _p(h), n, dim, hidden, float(dropout_p), seed, _p(RNG_OFFSET), _stream())
    _count()
    return out, u, h


def transpose_bf16(ws) -> Tensor:
    """w^T as a contiguous bf16 matrix -- or, for a list of up to 16 same-shaped matrices, [len, cols, rows] in one launch
    (the out-projection weights of a stack in the layout spb_ffn_bwd streams)."""
    single = isinstance(ws, Tensor)
    mats = [ws] if single else list(ws)
    _require_cuda(*mats)
    rows, cols = mats[0].shape
    assert all(w.dtype == BF16 and w.is_contiguous() and w.shape == (rows, cols) for w in mats)
    out = torch.empty((len(mats), cols, rows), dtype=BF16, device=mats[0].device)
    for i in range(0, len(mats), 16):
        part = mats[i:i + 16]
        _call("spb_transpose_bf16", _ptr_array(part), len(part), _p(out[i]), rows, cols, _stream())
        _count()
    return out[0] if single else out


def ffn_bwd(dy: Tensor, w2t: Tensor, w1: Tensor, u: Tensor, db1: Optional[Tensor], dropout_p: float, seed: int,
            in_place: bool = True):
    """Fused feed-forward backward, data path (one tcgen05 kernel): dy bf16 [n, 256], w2t bf16 [1024, 256] (W2 transposed),
    w1 bf16 [2048, 256], u bf16 [n, 2048] as saved by ffn_fwd.  Returns (dxn bf16 [n, 256], du bf16 [n, 2048]); with `in_place`
    du overwrites u.  db1 fp32 [2048] is accumulated into."""
    _require_cuda(dy, w2t, w1, u)
    n, dim = dy.shape
    hidden = w2t.shape[0]
    assert dy.dtype == BF16 and dy.stride(1) == 1 and u.dtype == BF16 and u.is_contiguous() and u.shape == (n, 2 * hidden)
    assert w1.dtype == BF16 and w2t.dtype == BF16 and w1.is_contiguous() and w2t.is_contiguous()
    assert w1.shape == (2 * hidden, dim) and w2t.shape == (hidden, dim)
    if db1 is not None:
        assert db1.dtype == F32 and db1.is_contiguous() and db1.numel() == 2 * hidden
    du = u if in_place else torch.empty_like(u)
    dxn = torch.empty((n, dim), dtype=BF16, device=dy.device)
    _call("spb_ffn_bwd", _p(dy), dy.stride(0), _p(w2t), _p(w1), _p(u), _p(du), _p(db1), _p(dxn), dxn.stride(0), n, dim, hidden,
          float(dropout_p), seed, _p(RNG_OFFSET), _stream())
    _count()
    return dxn, du


def multi_copy(dsts: Sequence[Tensor], srcs: Sequence[Tensor]) -> None:
    """dst_i.copy_(src_i) for lists of same-shaped, same-dtype contiguous CUDA tensors in ONE launch."""
    if not dsts:
        return
    _require_cuda(*dsts, *srcs)
    for d, s_ in zip(dsts, srcs):
        assert d.dtype == s_.dtype and d.shape == s_.shape and d.is_contiguous() and s_.is_contiguous()
    sizes = (ctypes.c_longlong * len(dsts))(*[d.numel() * d.element_size() for d in dsts])
    _call("spb_multi_copy", _ptr_array(dsts), _ptr_array(srcs), sizes, len(dsts), _stream())
    _count()


def multi_add(dsts: Sequence[Tensor], srcs: Sequence[Tensor]) -> None:
    """dst_i += src_i for lists of fp32 tensors (contiguous, same numel pairwise) in ONE launch."""
    if not dsts:
        return
    _require_cuda(*dsts, *srcs)
    assert len(dsts) == len(srcs)
    for d, s_ in zip(dsts, srcs):
        assert d.dtype == F32 and s_.dtype == F32 and d.is_contiguous() and s_.is_contiguous() and d.numel() == s_.numel()
    sizes = (ctypes.c_int * len(dsts))(*[d.numel() for d in dsts])
    _call("spb_multi_add_f32", _ptr_array(dsts), _ptr_array(srcs), sizes, len(dsts), _stream())
    _count()


def ffn_fused_ok(dim: int, hidden: int) -> bool:
    return dim == 256 and hidden == 1024 and _os.environ.get("SPB_FFN", "fused") == "fused"


def ffn_bwd_fused_ok(dim: int, hidden: int) -> bool:
    return dim == 256 and hidden == 1024 and _os.environ.get("SPB_FFN_BWD", "fused") == "fused"


def glu_bwd(dh: Tensor, u: Tensor, dbias: Optional[Tensor], dropout_p: float, seed: int) -> Tensor:
    assert dh.dtype == BF16 and dh.is_contiguous() and u.is_contiguous()
    n, two_h = u.shape
    du = torch.empty_like(u)
    _call("spb_glu_bwd", _p(dh), _p(u), _p(du), _p(dbias), n, two_h // 2, float(dropout_p), seed, _p(RNG_OFFSET), _stream())
    _count()
    return du


# ----------------------------------------------------------------------------- computed tables
def _ptr_array(tensors: Sequence[Tensor]):
    return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


def table_build_fwd(sizes: Sequence[int], per_field: Sequence[Sequence[Tensor]]) -> Tensor:
    """per_field[f] = (index_weight, token_values, discrete_mask, W0, b0, W1, b1) -> table fp32 [sum V, 128]."""
    flat = [t for fld in per_field for t in fld]
    _require_cuda(*flat)
    assert all(t.dtype == F32 and t.is_contiguous() for t in flat)
    table = torch.empty((int(sum(sizes)), 128), dtype=F32, device=flat[0].device)
    _call("spb_table_build_fwd", _sizes_array(sizes), len(sizes), _ptr_array(flat), _p(table), _stream())
    _count()
    return table


def table_build_bwd(sizes: Sequence[int], per_field: Sequence[Sequence[Tensor]], dtable: Tensor) -> None:
    """per_field[f] = the 7 forward tensors + (d_index_weight, dW0, db0, dW1, db1), accumulated into."""
    flat = [t for fld in per_field for t in fld]
    assert all(t.dtype == F32 and t.is_contiguous() for t in flat) and dtable.dtype == F32 and dtable.is_contiguous()
    _call("spb_table_build_bwd", _sizes_array(sizes), len(sizes), _ptr_array(flat), _p(dtable), _stream())
    _count()


# ----------------------------------------------------------------------------- tuple embedding
def _sizes_array(sizes: Sequence[int]):
    return (ctypes.c_int * len(sizes))(*[int(s) for s in sizes])


def embed_ln_fwd(tokens: Tensor, table: Tensor, sizes: Sequence[int], w: Tensor, b: Tensor, out: Optional[Tensor] = None,
                 eps: float = 1e-5):
    """tokens int64 [n, F] (any row stride), table fp32 [sum V, 128] -> (bf16 [n, F*128], mean, rstd)."""
    _require_cuda(tokens, table)
    assert tokens.dtype == torch.int64 and tokens.dim() == 2 and tokens.stride(1) == 1
    assert table.dtype == F32 and table.is_contiguous() and table.shape[1] == 128
    n, F = tokens.shape[0], len(sizes)
    if out is None:
        out = torch.empty((n, F * 128), dtype=BF16, device=tokens.device)
    mean = torch.empty(n, dtype=F32, device=tokens.device)
    rstd = torch.empty(n, dtype=F32, device=tokens.device)
    _call("spb_embed_ln_fwd", _p(tokens), tokens.stride(0), _p(table), _sizes_array(sizes), F, _p(w), _p(b), _p(out), out.stride(0),
          _p(mean), _p(rstd), n, float(eps), _stream())
    _count()
    return out, mean, rstd


def embed_ln_bwd(dy: Tensor, tokens: Tensor, table: Tensor, sizes: Sequence[int], w: Tensor, mean: Tensor, rstd: Tensor,
                 dtable: Tensor, dw: Tensor, db: Tensor) -> None:
    assert dy.dtype == BF16 and dy.stride(1) == 1
    n = tokens.shape[0]
    scratch = torch.empty((2, n), dtype=F32, device=dy.device)
    _call("spb_embed_ln_bwd", _p(dy), dy.stride(0), _p(tokens), tokens.stride(0), _p(table), _sizes_array(sizes), len(sizes), _p(w),
          _p(mean), _p(rstd), _p(scratch[0]), _p(scratch[1]), _p(dtable), _p(dw), _p(db), n, _stream())
    _count(2)


# ----------------------------------------------------------------------------- attention
class AttnAux:
    """Side outputs of the tcgen05 forward that its backward consumes: key-validity bit words and E_i[|i-j|]."""
    __slots__ = ("impl", "mask_bits", "edist")

    def __init__(self, impl: str, mask_bits: Optional[Tensor] = None, edist: Optional[Tensor] = None):
        self.impl, self.mask_bits, self.edist = impl, mask_bits, edist


def attention_impl(H: int) -> str:
    """"tcgen05" (TMEM/TMA kernels, need 4 heads) unless SPB_ATTN=mma selects the legacy mma.sync kernels."""
    return "tcgen05" if (H == 4 and ATTENTION_IMPL == "tcgen05") else "mma"


def attention_fwd(qkv: Tensor, key_mask: Optional[Tensor], logslopes: Tensor, B: int, T: int, H: int, causal: bool,
                  dropout_p: float, seed: int, impl: Optional[str] = None, need_aux: bool = True):
    """qkv bf16 [B*T, H*64+128] -> (out bf16 [B*T, H*64], lse fp32 [B,H,T], aux).  `aux` goes to attention_bwd unchanged."""
    _require_cuda(qkv)
    assert qkv.dtype == BF16 and qkv.stride(1) == 1 and logslopes.dtype == F32
    out = torch.empty((B * T, H * 64), dtype=BF16, device=qkv.device)
    lse = torch.empty((B, H, T), dtype=F32, device=qkv.device)
    impl = impl or attention_impl(H)
    if impl == "tcgen05":
        bits = torch.empty((B, (T + 31) // 32), dtype=torch.int32, device=qkv.device) if key_mask is not None else None
        edist = torch.empty((B, H, T), dtype=F32, device=qkv.device) if need_aux else None
        _call("spb_attention_fwd_tc", _p(qkv), qkv.stride(0), _p(key_mask), _p(bits), _p(logslopes), _p(out), out.stride(0), _p(lse),
              _p(edist), B, T, H, 64, int(causal), float(dropout_p), seed, _p(RNG_OFFSET), _stream())
        _count(2 if key_mask is not None else 1)
        return out, lse, AttnAux("tcgen05", bits, edist)
    _call("spb_attention_fwd", _p(qkv), qkv.stride(0), _p(key_mask), _p(logslopes), _p(out), out.stride(0), _p(lse), B, T, H, 64,
          int(causal), float(dropout_p), seed, _p(RNG_OFFSET), _stream())
    _count()
    return out, lse, AttnAux("mma")


_DQ_ACC = {}


def _dq_accumulator(n: int, cols: int, device) -> Tensor:
    """fp32 [n, cols] scratch of the tcgen05 backward: zero between calls (the kernel's last pass re-zeroes it), one per
    (stream, shape), so backward branches running on different streams never share one."""
    key = (torch.cuda.current_stream().cuda_stream, n, cols, str(device))
    buf = _DQ_ACC.get(key)
    if buf is None:
        buf = _DQ_ACC[key] = torch.zeros((n, cols), dtype=F32, device=device)
    return buf


def attention_bwd(qkv: Tensor, key_mask: Optional[Tensor], logslopes: Tensor, out: Tensor, dout: Tensor, lse: Tensor,
                  dlogslopes: Tensor, B: int, T: int, H: int, causal: bool, dropout_p: float, seed: int,
                  delta: Optional[Tensor] = None, aux: Optional[AttnAux] = None) -> Tensor:
    """`delta` fp32 [B, H, T] = rowsum(dO * O) may be supplied (gemm_rowdot produces it with dO); otherwise it is computed here.
    `aux` is what attention_fwd returned: it selects the matching backward implementation."""
    assert dout.dtype == BF16 and dout.stride(1) == 1 and dout.stride(0) == out.stride(0)
    dqkv = torch.empty_like(qkv)
    if aux is not None and aux.impl == "tcgen05":
        assert aux.edist is not None, "the tcgen05 backward needs the forward's edist (attention_fwd(need_aux=True))"
        if delta is None:
            delta = (dout.float().view(B, T, H, 64) * out.float().view(B, T, H, 64)).sum(-1).permute(0, 2, 1).contiguous()
        acc = _dq_accumulator(B * T, H * 64, qkv.device)
        _call("spb_attention_bwd_tc", _p(qkv), qkv.stride(0), _p(aux.mask_bits), _p(logslopes), _p(dout), dout.stride(0), _p(lse),
              _p(delta), _p(aux.edist), _p(acc), _p(dqkv), dqkv.stride(0), _p(dlogslopes), B, T, H, 64, int(causal), float(dropout_p),
              seed, _p(RNG_OFFSET), _stream())
        _count(2)
        return dqkv
    ready = delta is not None
    if delta is None:
        delta = torch.empty((B, H, T), dtype=F32, device=qkv.device)
    assert delta.dtype == F32 and delta.numel() == B * H * T and delta.is_contiguous()
    _call("spb_attention_bwd", _p(qkv), qkv.stride(0), _p(key_mask), _p(logslopes), _p(out), _p(dout), out.stride(0), _p(lse), _p(delta),
          _p(dqkv), dqkv.stride(0), _p(dlogslopes), B, T, H, 64, int(causal), float(dropout_p), seed, _p(RNG_OFFSET), int(ready),
          _stream())
    _count(2 if ready else 3)
    return dqkv


def gemm_rowdot(a: Tensor, b: Tensor, x: Tensor, T: int, H: int, *, trans_b: bool = False, bias: Optional[Tensor] = None,
                rowmask: Optional[Tensor] = None, alpha: Optional[Tensor] = None):
    """C = A op(B)^T as bf16 [M, H*64] plus delta[b, h, t] = sum over head h's 64 columns of C[b*T+t, :] * x[b*T+t, :].
    Returns (C, delta fp32 [M/T, H, T])."""
    _require_cuda(a, b, x)
    assert a.dtype == BF16 and b.dtype == BF16 and x.dtype == BF16 and a.stride(1) == 1 and b.stride(1) == 1 and x.stride(1) == 1
    M, Kd = a.shape
    N = b.shape[1] if trans_b else b.shape[0]
    assert N == H * 64 and M % T == 0 and x.shape == (M, N)
    out = torch.empty((M, N), dtype=BF16, device=a.device)
    delta = torch.empty((M // T, H, T), dtype=F32, device=a.device)
    _call("spb_gemm_bf16_rowdot", _p(a), _p(b), _p(out), M, N, Kd, 0, int(trans_b), a.stride(0), b.stride(0), out.stride(0), _p(bias),
          _p(rowmask), _p(alpha), _p(x), x.stride(0), _p(delta), T, H, _stream())
    _count()
    return out, delta


def attention_decode(q: Tensor, kv: Tensor, key_mask: Optional[Tensor], logslopes: Tensor, H: int, n_keys: int, q_pos: int,
                     pos_dev: Optional[Tensor] = None, append_kv: bool = False) -> Tensor:
    """q bf16 [B, >=H*64]; kv bf16 [B, cap, 128] (k | v); returns bf16 [B, H*64].

    With `pos_dev` (device int64 [1]) the position is read on the device and `n_keys` is the cache capacity, so the launch can
    be replayed from a CUDA graph; `append_kv` first stores q[:, H*64:H*64+128] as cache row q_pos."""
    _require_cuda(q, kv)
    assert q.dtype == BF16 and kv.dtype == BF16 and q.stride(1) == 1 and kv.stride(2) == 1
    assert pos_dev is None or (pos_dev.dtype == torch.int64 and pos_dev.is_cuda)
    assert not append_kv or q.shape[1] >= H * 64 + 128
    B = q.shape[0]
    out = torch.empty((B, H * 64), dtype=BF16, device=q.device)
    _call("spb_attention_decode", _p(q), q.stride(0), _p(kv), kv.stride(1), kv.stride(0), _p(key_mask),
          key_mask.stride(0) if key_mask is not None else 0, _p(logslopes), _p(out), out.stride(0), B, H, 64, n_keys, q_pos,
          _p(pos_dev), int(append_kv), _stream())
    _count()
    return out


# ----------------------------------------------------------------------------- latent levels / MMD
def latent_level_fwd(hidden: Tensor, style: Tensor, mask: Tensor, segments: Optional[Tensor], W: Tensor, bias: Tensor, col0: int,
                     S: int, z: int):
    """One VAE level.  Returns (latents [B,S,z], lmask [B,S] bool, pooled [B*S,320], counts [B*S])."""
    _require_cuda(hidden, style)
    B, T, D = hidden.shape
    assert hidden.dtype == F32 and hidden.is_contiguous() and style.dtype == F32 and style.is_contiguous()
    pooled = torch.zeros((B * S, 320), dtype=F32, device=hidden.device)
    counts = torch.zeros((B * S,), dtype=torch.int32, device=hidden.device)
    latents = torch.empty((B, S, z), dtype=F32, device=hidden.device)
    lmask = torch.empty((B, S), dtype=torch.bool, device=hidden.device)
    _call("spb_latent_level_fwd", _p(hidden), _p(style), style.shape[-1], _p(mask), _p(segments), _p(W), _p(bias), _p(pooled), _p(counts),
          _p(latents), _p(lmask), _p(style), col0, B, T, S, D, col0, z, _stream())
    _count(3)
    return latents, lmask, pooled, counts


def latent_level_bwd(d_style: Tensor, col0: int, dlat_direct: Optional[Tensor], mask: Tensor, segments: Optional[Tensor], W: Tensor,
                     pooled: Tensor, counts: Tensor, lmask: Tensor, d_hidden: Tensor, dW: Tensor, dbias: Tensor, S: int, z: int) -> None:
    B, T, D = d_hidden.shape
    dlat = torch.zeros((B * S, z), dtype=F32, device=d_hidden.device)
    dpooled = torch.empty((B * S, 320), dtype=F32, device=d_hidden.device)
    _call("spb_latent_level_bwd", _p(d_style), d_style.shape[-1], col0, _p(dlat_direct), _p(mask), _p(segments), _p(W), _p(pooled),
          _p(counts), _p(lmask), _p(dlat), _p(dpooled), _p(d_hidden), _p(dW), _p(dbias), B, T, S, D, col0, z, _stream())
    _count(5)


def mmd_fwd_bwd(z_prior: Tensor, y: Tensor, w: Tensor):
    """Returns (loss [1] fp32, grad_y [n_y, d] fp32)."""
    _require_cuda(z_prior, y)
    assert z_prior.dtype == F32 and y.dtype == F32 and z_prior.is_contiguous() and y.is_contiguous() and w.dtype == torch.bool
    n_z, d = z_prior.shape
    n_y = y.shape[0]
    coef = torch.empty(n_z + n_y, dtype=F32, device=y.device)
    loss = torch.zeros(1, dtype=F32, device=y.device)
    grad = torch.zeros_like(y)
    _call("spb_mmd_fwd_bwd", _p(z_prior), _p(y), _p(w), n_z, n_y, d, _p(coef), _p(loss), _p(grad), _stream())
    _count(2)
    return loss, grad


# ----------------------------------------------------------------------------- heads
def ce_rows(logits: Tensor, labels: Tensor, V: int, loss_sum: Tensor, count: Tensor, dlogits: Optional[Tensor] = None,
            argmax: Optional[Tensor] = None, ignore_index: int = -100) -> None:
    """logits fp32 [n, >=V]; labels int64 [n] (strided view allowed)."""
    assert logits.dtype == F32 and logits.stride(1) == 1 and labels.dtype == torch.int64 and labels.dim() == 1
    _call("spb_ce_rows", _p(logits), logits.stride(0), _p(labels), labels.stride(0), V, ignore_index, _p(loss_sum), _p(count),
          _p(dlogits), dlogits.stride(0) if dlogits is not None else 0, _p(argmax), logits.shape[0], _stream())
    _count()


def head_ce(e_f: Tensor, table_f: Tensor, labels: Tensor, loss_sum: Tensor, count: Tensor, dlogits: Optional[Tensor] = None,
            argmax: Optional[Tensor] = None, ignore_index: int = -100, token_values: Optional[Tensor] = None,
            stats: Optional[Tensor] = None) -> None:
    """Fused tied head + cross-entropy of one field: e_f bf16 [n, 128] (strided view allowed), table_f bf16 [V, 128],
    labels int64 [n] (strided view allowed).  loss_sum / count fp32 scalars are accumulated into; `stats` (fp32 [3], accumulated)
    receives the evaluator sums (hits, |tv[argmax]-tv[label]|, expected |tv[label]-tv[v]|) with tv = `token_values` fp32 [V]."""
    _require_cuda(e_f, table_f)
    assert e_f.dtype == BF16 and table_f.dtype == BF16 and e_f.shape[1] == 128 and table_f.shape[1] == 128
    assert e_f.stride(1) == 1 and table_f.stride(1) == 1 and labels.dtype == torch.int64 and labels.dim() == 1
    n, V = e_f.shape[0], table_f.shape[0]
    if dlogits is not None:
        assert dlogits.dtype == BF16 and dlogits.shape[0] == n and dlogits.stride(1) == 1
    if token_values is not None:
        assert stats is not None and token_values.dtype == F32 and token_values.numel() >= V and token_values.is_contiguous()
    if stats is not None:
        assert stats.dtype == F32 and stats.numel() >= 3 and stats.is_contiguous()
    _call("spb_head_ce", _p(e_f), e_f.stride(0), _p(table_f), table_f.stride(0), V, _p(labels), labels.stride(0), ignore_index,
          _p(loss_sum), _p(count), _p(dlogits), dlogits.stride(0) if dlogits is not None else 0, _p(argmax), _p(token_values),
          _p(stats), n, _stream())
    _count()


def adamw_step(p: Tensor, g: Tensor, m: Tensor, v: Tensor, shadow: Optional[Tensor], grad_norm: Optional[Tensor], step: Tensor, *,
               lr: float, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0, max_norm: float = 0.0,
               grad_scale: float = 1.0, lr_dev: Optional[Tensor] = None) -> None:
    """Clip-by-global-norm + AdamW + bf16 shadow refresh over flat fp32 buffers (one launch for the whole model)."""
    _require_cuda(p, g, m, v)
    assert p.dtype == F32 and g.dtype == F32 and m.dtype == F32 and v.dtype == F32 and step.dtype == torch.int64
    assert p.is_contiguous() and g.is_contiguous() and m.is_contiguous() and v.is_contiguous()
    n = p.numel()
    assert g.numel() == n and m.numel() == n and v.numel() == n and (shadow is None or (shadow.dtype == BF16 and shadow.numel() == n))
    _call("spb_adamw_step", _p(p), _p(g), _p(m), _p(v), _p(shadow), n, _p(grad_norm), float(grad_scale), float(max_norm), float(lr),
          float(betas[0]), float(betas[1]), float(eps), float(weight_decay), _p(step), _p(lr_dev), _stream())
    _count()


def clf_heads(x: Tensor, rowmask: Tensor, labels: Tensor, W: Tensor, bias: Tensor, class_w: Tensor, n_classes: Sequence[int],
              dropout_p: float, seed: int, num: Optional[Tensor] = None, den: Optional[Tensor] = None,
              dlogit_scale: Optional[Tensor] = None, dW: Optional[Tensor] = None, db: Optional[Tensor] = None) -> None:
    """x fp32 [n, in_dim]; labels int64 [n, n_heads]; forward when dlogit_scale is None, else backward."""
    assert x.dtype == F32 and x.stride(1) == 1 and labels.dtype == torch.int64 and labels.stride(1) == 1
    n, in_dim = x.shape
    backward = dlogit_scale is not None
    scratch = torch.empty((n, int(sum(n_classes))), dtype=F32, device=x.device) if backward else None
    _call("spb_clf_heads", _p(x), x.stride(0), _p(rowmask), _p(labels), labels.stride(0), _p(W), _p(bias), _p(class_w),
          _sizes_array(n_classes), len(n_classes), _p(num), _p(den), _p(dlogit_scale), _p(dW), _p(db), _p(scratch), n, in_dim,
          float(dropout_p), seed, _p(RNG_OFFSET), int(backward), _stream())
    _count(2 if backward else 1)


def clf_logits(x: Tensor, W: Tensor, bias: Tensor) -> Tensor:
    n, in_dim = x.shape
    out = torch.empty((n, W.shape[0]), dtype=F32, device=x.device)
    _call("spb_clf_logits", _p(x), x.stride(0), _p(W), _p(bias), _p(out), n, in_dim, W.shape[0], _stream())
    _count()
    return out
