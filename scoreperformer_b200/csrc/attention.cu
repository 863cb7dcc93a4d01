// Fused multi-query attention (1 KV head shared by H query heads) with in-kernel learned-slope ALiBi,
// key-padding + causal masking and dropout: forward and backward, flash style (no [T,T] tensor in HBM).
//
// Reference semantics: modules/transformer/attention.py:107-222 (MQA projections, masks, ALiBi) and
// modules/transformer/attend.py:58-126 (additive bias with masked fill, softmax, dropout, P@V).
//   S_ij = scale * q_i.k_j - slope_h * |i - j|     (modules/transformer/embeddings.py:294-325, symmetric)
//   masked (padded key, or j > i when causal) entries are excluded from the softmax
// Round-1 implementation: bf16 mma.sync.m16n8k16 with ldmatrix from XOR-swizzled shared memory tiles and
// cp.async double buffering; the tcgen05/TMEM version is the next step (DESIGN.md).
//
// Layout: qkv bf16 [B*T, ld] with q at columns [0, H*64), k at [H*64, H*64+64), v at [H*64+64, H*64+128).
#include "common.cuh"

namespace {

constexpr int DH = 64;
constexpr int TQ = 64;   // queries per CTA
constexpr int TK = 64;   // keys per tile
constexpr float LOG2E = 1.4426950408889634f;
constexpr int ATT_MAX_T = 8192;   // key-validity bits of one sequence live in shared memory (32 keys per word)

struct AttnParams {
    const __nv_bfloat16* qkv;
    int ld;                      // row stride of qkv (elements)
    const uint8_t* key_mask;     // [B, T] or null
    const float* logslopes;      // [H]
    int B, T, H;
    float scale;
    int causal;
    float dropout_p;
    uint64_t seed;
    const uint64_t* rng_offset;   // optional device counter mixed into the seed (CUDA-graph replays get fresh masks)
    uint32_t drop_thresh24;
    float keep_scale;
};

__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float* d, const uint32_t* a, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// Dropout: one 32-bit counter hash per PAIR of adjacent key columns (j, j^1) of a (batch, head, query) row gives two 16-bit
// uniform numbers; forward and both backward kernels evaluate the same function, so no mask is stored.
struct DropCtx {
    uint32_t seed32, thr16, half_t;
    float keep_scale;
    bool on;
};
__device__ __forceinline__ DropCtx make_drop(const AttnParams& p) {
    DropCtx d;
    d.seed32 = (uint32_t)(p.seed ^ (p.seed >> 32));
    d.thr16 = p.drop_thresh24 >> 8;
    d.half_t = (uint32_t)((p.T + 1) >> 1);
    d.keep_scale = p.keep_scale;
    d.on = p.drop_thresh24 != 0;
    return d;
}
__device__ __forceinline__ uint32_t hash32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
// row_lin = (b*H + h)*T + i
__device__ __forceinline__ uint32_t pair_hash(const DropCtx& d, uint32_t row_lin, uint32_t j) {
    return hash32((row_lin * d.half_t + (j >> 1)) * 0x9E3779B9u + d.seed32);
}

// A 64x64 bf16 tile: row r at r*128 B, 16-byte chunk c stored at chunk (c ^ (r & 7)).
__device__ __forceinline__ uint32_t tile_addr(uint32_t base, int row, int chunk) {
    return base + row * 128 + ((chunk ^ (row & 7)) << 4);
}

// Load a [64 rows x 64 cols] bf16 tile from global (row stride ld) starting at (row0, col0); rows >= n_valid zero-filled.
__device__ __forceinline__ void load_tile_async(void* smem, const __nv_bfloat16* g, int ld, int row0, int col0, int row_limit) {
    const uint32_t base = smem_u32(smem);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int idx = threadIdx.x + i * 128;
        const int r = idx >> 3, c = idx & 7;
        const bool ok = (row0 + r) < row_limit;
        const __nv_bfloat16* src = g + (size_t)(ok ? row0 + r : 0) * ld + col0 + c * 8;
        const uint32_t dst = tile_addr(base, r, c);
        const int bytes = ok ? 16 : 0;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(bytes) : "memory");
    }
}

// A fragments (16 rows x 64 k) of a row-major tile: frag[ks][0..3] for the 4 k-steps.
__device__ __forceinline__ void load_a_frags(uint32_t base, int row0, int lane, uint32_t frag[4][4]) {
    const int r = row0 + (lane & 7) + ((lane >> 3) & 1) * 8;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) ldsm_x4(tile_addr(base, r, ks * 2 + (lane >> 4)), frag[ks][0], frag[ks][1], frag[ks][2], frag[ks][3]);
}

// acc[nt][4] (16 x 64) = A(16 x 64k) * Tile^T where Tile is [n=64][k=64] row-major ("K-like": rows are n).
__device__ __forceinline__ void mma_a_tile_nt(float acc[8][4], const uint32_t a[4][4], uint32_t tile, int lane) {
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int kp = 0; kp < 2; ++kp) {   // two k-steps per ldmatrix.x4
            uint32_t b0, b1, b2, b3;
            ldsm_x4(tile_addr(tile, nt * 8 + (lane & 7), kp * 4 + (lane >> 3)), b0, b1, b2, b3);
            mma16816(acc[nt], a[kp * 2], b0, b1);
            mma16816(acc[nt], a[kp * 2 + 1], b2, b3);
        }
    }
}
// acc[nt][4] (16 x 64n) += P(16 x 64k, as A fragments pf[ks]) * Tile where Tile is [k=64][n=64] row-major ("V-like").
__device__ __forceinline__ void mma_p_tile_nn(float acc[8][4], const uint32_t pf[4][4], uint32_t tile, int lane) {
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
        for (int np = 0; np < 4; ++np) {   // two n-blocks per ldmatrix.x4.trans
            uint32_t b0, b1, b2, b3;
            ldsm_x4_t(tile_addr(tile, ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, np * 2 + (lane >> 4)), b0, b1, b2, b3);
            mma16816(acc[np * 2], pf[ks], b0, b1);
            mma16816(acc[np * 2 + 1], pf[ks], b2, b3);
        }
    }
}
// pack a 16x64 fp32 accumulator into A fragments for the next MMA
__device__ __forceinline__ void acc_to_frags(const float acc[8][4], uint32_t pf[4][4]) {
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        pf[ks][0] = pack_bf16x2(acc[2 * ks][0], acc[2 * ks][1]);
        pf[ks][1] = pack_bf16x2(acc[2 * ks][2], acc[2 * ks][3]);
        pf[ks][2] = pack_bf16x2(acc[2 * ks + 1][0], acc[2 * ks + 1][1]);
        pf[ks][3] = pack_bf16x2(acc[2 * ks + 1][2], acc[2 * ks + 1][3]);
    }
}

// ------------------------------------------------------------------------------------------- forward
// grid (ceil(T/64), H, B), 128 threads; warp w owns query rows [16w, 16w+16) of the tile.
__global__ void __launch_bounds__(128, 3)
attn_fwd_kernel(AttnParams p, __nv_bfloat16* __restrict__ out, int ld_out, float* __restrict__ lse_out) {
    if (p.rng_offset != nullptr) p.seed += *p.rng_offset * 0x9E3779B97F4A7C15ull;
    __shared__ __align__(128) uint8_t sQ[TQ * 128];
    __shared__ __align__(128) uint8_t sK[2][TK * 128];
    __shared__ __align__(128) uint8_t sV[2][TK * 128];
    __shared__ uint32_t sMaskAll[ATT_MAX_T / 32];    // key validity of the whole sequence, built once

    const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int T = p.T;
    const int q0 = qt * TQ;
    const DropCtx drop = make_drop(p);
    const int kcol = p.H * DH, vcol = kcol + DH;
    const __nv_bfloat16* base = p.qkv + (size_t)b * T * p.ld;
    const float slope = __expf(p.logslopes[h]) * LOG2E;
    const float scale2 = p.scale * LOG2E;

    const int n_kt = p.causal ? min(qt + 1, ceil_div(T, TK)) : ceil_div(T, TK);

    auto load_kv = [&](int kt, int buf) {
        load_tile_async(sK[buf], base, p.ld, kt * TK, kcol, T);
        load_tile_async(sV[buf], base, p.ld, kt * TK, vcol, T);
    };

    load_tile_async(sQ, base, p.ld, q0, h * DH, T);
    load_kv(0, 0);
    cp_async_commit();
    // key-validity words for every key tile, once per CTA (a per-tile global load would sit on the critical path)
    for (int w = warp; w * 32 < n_kt * TK; w += 4) {
        const int j = w * 32 + lane;
        const bool ok = (j < T) && (p.key_mask == nullptr || p.key_mask[(size_t)b * T + j]);
        const uint32_t bits = __ballot_sync(0xffffffffu, ok);
        if (lane == 0) sMaskAll[w] = bits;
    }

    float o_acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) o_acc[i][j] = 0.f;
    float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
    uint32_t qf[4][4];
    const int r_lo = q0 + warp * 16 + (lane >> 2);   // this thread's rows: r_lo and r_lo + 8

    for (int kt = 0; kt < n_kt; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < n_kt) load_kv(kt + 1, buf ^ 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        if (kt == 0) load_a_frags(smem_u32(sQ), warp * 16, lane, qf);

        float s[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
        mma_a_tile_nt(s, qf, smem_u32(sK[buf]), lane);

        // scores in base-2 units: s*scale2 - slope*|i-j|; the mask / causal tests only run on tiles that need them
        const uint32_t w0 = sMaskAll[kt * 2], w1 = sMaskAll[kt * 2 + 1];
        const bool diag = p.causal && (kt == qt);
        const float dbase0 = (float)(r_lo - (kt * TK + (lane & 3) * 2));     // i - j for e = 0, nt = 0
        if (diag || (w0 & w1) != 0xffffffffu) {
            // only tiles with padded keys or on the causal diagonal pay for masking: masked scores become -inf up front
            const uint32_t mlo = w0 >> ((lane & 3) * 2), mhi = w1 >> ((lane & 3) * 2);
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float d = dbase0 + (float)((e >> 1) * 8 - nt * 8 - (e & 1));
                    const uint32_t word = nt < 4 ? mlo : mhi;
                    const bool ok = ((word >> ((nt & 3) * 8 + (e & 1))) & 1u) && (!diag || d >= 0.f);
                    if (!ok) s[nt][e] = -INFINITY;
                }
            }
        }
        float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float d = dbase0 + (float)((e >> 1) * 8 - nt * 8 - (e & 1));
                const float v = fmaf(-slope, fabsf(d), s[nt][e] * scale2);      // -inf stays -inf
                s[nt][e] = v;
                mx[e >> 1] = fmaxf(mx[e >> 1], v);
            }
        }
        float corr[2], m_use[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
            const float m_new = fmaxf(m_run[r], mx[r]);
            m_use[r] = (m_new == -INFINITY) ? 0.f : m_new;
            corr[r] = exp2f(m_run[r] - m_use[r]);      // m_run = -inf -> 0
            m_run[r] = m_new;
        }
        float rs[2] = {0.f, 0.f};
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float pv = exp2f(s[nt][e] - m_use[e >> 1]);
                rs[e >> 1] += pv;
                s[nt][e] = pv;
            }
        }
        if (drop.on) {
#pragma unroll
            for (int rr = 0; rr < 2; ++rr) {
                const uint32_t row_lin = (uint32_t)((b * p.H + h) * T + r_lo + rr * 8);
#pragma unroll
                for (int nt = 0; nt < 8; ++nt) {
                    const uint32_t hsh = pair_hash(drop, row_lin, (uint32_t)(kt * TK + nt * 8 + (lane & 3) * 2));
                    s[nt][rr * 2] = (hsh & 0xffffu) >= drop.thr16 ? s[nt][rr * 2] * drop.keep_scale : 0.f;
                    s[nt][rr * 2 + 1] = (hsh >> 16) >= drop.thr16 ? s[nt][rr * 2 + 1] * drop.keep_scale : 0.f;
                }
            }
        }
#pragma unroll
        for (int r = 0; r < 2; ++r) l_run[r] = l_run[r] * corr[r] + rs[r];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            o_acc[nt][0] *= corr[0]; o_acc[nt][1] *= corr[0];
            o_acc[nt][2] *= corr[1]; o_acc[nt][3] *= corr[1];
        }
        uint32_t pf[4][4];
        acc_to_frags(s, pf);
        mma_p_tile_nn(o_acc, pf, smem_u32(sV[buf]), lane);
        __syncthreads();
    }

#pragma unroll
    for (int r = 0; r < 2; ++r) {
        l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
        l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int i = r_lo + r * 8;
        if (i < T) {
            const float inv = l_run[r] > 0.f ? 1.f / l_run[r] : 0.f;
            __nv_bfloat16* dst = out + ((size_t)b * T + i) * ld_out + h * DH + (lane & 3) * 2;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt)
                *reinterpret_cast<uint32_t*>(dst + nt * 8) = pack_bf16x2(o_acc[nt][r * 2] * inv, o_acc[nt][r * 2 + 1] * inv);
            if ((lane & 3) == 0 && lse_out != nullptr)
                lse_out[((size_t)b * p.H + h) * T + i] = l_run[r] > 0.f ? (m_run[r] + log2f(l_run[r])) : INFINITY;  // base-2 units; +inf => P = 0 in backward
        }
    }
}

// ------------------------------------------------------------------------------------------- backward
// delta[b,h,i] = sum_d dO[b,i,h,d] * O[b,i,h,d]
__global__ void attn_delta_kernel(const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ dout, int ld,
                                  float* __restrict__ delta, int B, int T, int H) {
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (gw >= B * T * H) return;
    const int h = gw % H;
    const int bt = gw / H;
    const float2 a = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(o + (size_t)bt * ld + h * DH + lane * 2));
    const float2 d = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(dout + (size_t)bt * ld + h * DH + lane * 2));
    const float s = warp_sum(a.x * d.x + a.y * d.y);
    if (lane == 0) delta[((size_t)(bt / T) * H + h) * T + (bt % T)] = s;
}

// dK, dV: grid (ceil(T/64) key tiles, B); warp w owns keys [16w, 16w+16); loops over heads and query tiles.
__global__ void __launch_bounds__(128)
attn_bwd_dkv_kernel(AttnParams p, const __nv_bfloat16* __restrict__ dout, int ld_do, const float* __restrict__ lse,
                    const float* __restrict__ delta, __nv_bfloat16* __restrict__ dqkv, int ld_dqkv) {
    if (p.rng_offset != nullptr) p.seed += *p.rng_offset * 0x9E3779B97F4A7C15ull;
    extern __shared__ __align__(128) uint8_t dyn_smem[];
    uint8_t* sK = dyn_smem;
    uint8_t* sV = sK + TK * 128;
    uint8_t (*sQ)[TQ * 128] = reinterpret_cast<uint8_t (*)[TQ * 128]>(sV + TK * 128);
    uint8_t (*sDO)[TQ * 128] = reinterpret_cast<uint8_t (*)[TQ * 128]>(sV + TK * 128 + 2 * TQ * 128);
    __shared__ __align__(16) float sLse[2][TQ];
    __shared__ __align__(16) float sDelta[2][TQ];

    const int kt = blockIdx.x, b = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int T = p.T, H = p.H;
    const int k0 = kt * TK;
    const DropCtx drop = make_drop(p);
    const int kcol = H * DH, vcol = kcol + DH;
    const __nv_bfloat16* base = p.qkv + (size_t)b * T * p.ld;
    const __nv_bfloat16* dbase = dout + (size_t)b * T * ld_do;
    const float scale2 = p.scale * LOG2E;

    const int n_qt = ceil_div(T, TQ);
    const int qt_begin = p.causal ? kt : 0;
    const int iters = H * (n_qt - qt_begin);

    // (head, query tile) of an iteration advance as counters: an integer division per use costs ~40 instructions here
    auto load_q = [&](int h, int qt, int buf) {
        load_tile_async(sQ[buf], base, p.ld, qt * TQ, h * DH, T);
        load_tile_async(sDO[buf], dbase, ld_do, qt * TQ, h * DH, T);
        if (threadIdx.x < TQ) {
            // asynchronous like the tiles (a plain load here parks the warp on the long scoreboard every iteration).  Rows
            // beyond T are zero-filled: their Q and dO rows are zero too, so P stays finite and dS = dV-contribution = 0.
            const int i = qt * TQ + threadIdx.x;
            const bool ok = i < T;
            const size_t src = ((size_t)b * H + h) * T + (ok ? i : 0);
            const int bytes = ok ? 4 : 0;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_u32(&sLse[buf][threadIdx.x])), "l"(lse + src), "r"(bytes) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_u32(&sDelta[buf][threadIdx.x])), "l"(delta + src), "r"(bytes) : "memory");
        }
    };

    load_tile_async(sK, base, p.ld, k0, kcol, T);
    load_tile_async(sV, base, p.ld, k0, vcol, T);
    if (iters > 0) load_q(0, qt_begin, 0);
    cp_async_commit();

    float dk[8][4], dv[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { dk[i][j] = 0.f; dv[i][j] = 0.f; }
    uint32_t kf[4][4], vf[4][4];
    const int j_lo = k0 + warp * 16 + (lane >> 2);   // this thread's keys: j_lo, j_lo + 8
    bool key_ok[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int j = j_lo + r * 8;
        key_ok[r] = (j < T) && (p.key_mask == nullptr || p.key_mask[(size_t)b * T + j]);
    }
    const bool keys_plain = __all_sync(0xffffffffu, key_ok[0] && key_ok[1]);     // no padded key among this warp's 16

    int h = 0, qt = qt_begin;
    for (int it = 0; it < iters; ++it) {
        const int buf = it & 1;
        int h_next = h, qt_next = qt + 1;
        if (qt_next == n_qt) { qt_next = qt_begin; ++h_next; }
        if (it + 1 < iters) load_q(h_next, qt_next, buf ^ 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        if (it == 0) {
            load_a_frags(smem_u32(sK), warp * 16, lane, kf);
            load_a_frags(smem_u32(sV), warp * 16, lane, vf);
        }
        const float slope = __expf(p.logslopes[h]) * LOG2E;

        // S^T[keys x queries] = K Q^T
        float st[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) st[i][j] = 0.f;
        mma_a_tile_nt(st, kf, smem_u32(sQ[buf]), lane);
        // dP^T[keys x queries] = V dO^T
        float dpt[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) dpt[i][j] = 0.f;
        mma_a_tile_nt(dpt, vf, smem_u32(sDO[buf]), lane);

        uint32_t pf[4][4];
        const bool diag = p.causal && (qt == kt);
        const float dbase0 = (float)(qt * TQ + (lane & 3) * 2 - j_lo);       // i - j for e = 0, nt = 0
        if (diag || !keys_plain) {
            // masked scores become -inf up front (P = exp2(-inf) = 0), so the main loop carries no mask logic
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float d = dbase0 + (float)(nt * 8 + (e & 1) - (e >> 1) * 8);
                    if (!(key_ok[e >> 1] && (!diag || d >= 0.f))) st[nt][e] = -INFINITY;
                }
            }
        }
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            float pd[4];
            const float2 lse2 = *reinterpret_cast<const float2*>(&sLse[buf][nt * 8 + (lane & 3) * 2]);
            const float2 del2 = *reinterpret_cast<const float2*>(&sDelta[buf][nt * 8 + (lane & 3) * 2]);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float d = dbase0 + (float)(nt * 8 + (e & 1) - (e >> 1) * 8);
                const float lse_i = (e & 1) ? lse2.y : lse2.x;
                const float pv = exp2f(fmaf(-slope, fabsf(d), st[nt][e] * scale2) - lse_i);
                float keep = 1.f;
                if (drop.on) {
                    const int i = qt * TQ + nt * 8 + (lane & 3) * 2 + (e & 1);
                    const int j = j_lo + (e >> 1) * 8;
                    const uint32_t hsh = pair_hash(drop, (uint32_t)((b * H + h) * T + i), (uint32_t)j);
                    const uint32_t u16 = (j & 1) ? (hsh >> 16) : (hsh & 0xffffu);
                    keep = u16 >= drop.thr16 ? drop.keep_scale : 0.f;
                }
                pd[e] = pv * keep;                                                        // dropped P^T (for dV)
                st[nt][e] = pv * (dpt[nt][e] * keep - ((e & 1) ? del2.y : del2.x));       // dS^T
            }
            // pack P^T_drop into A fragments as we go (two n-tiles form one k-step)
            const int ks = nt >> 1;
            if ((nt & 1) == 0) { pf[ks][0] = pack_bf16x2(pd[0], pd[1]); pf[ks][1] = pack_bf16x2(pd[2], pd[3]); }
            else { pf[ks][2] = pack_bf16x2(pd[0], pd[1]); pf[ks][3] = pack_bf16x2(pd[2], pd[3]); }
        }
        mma_p_tile_nn(dv, pf, smem_u32(sDO[buf]), lane);   // dV += P^T_drop dO
        acc_to_frags(st, pf);
        mma_p_tile_nn(dk, pf, smem_u32(sQ[buf]), lane);    // dK += dS^T Q
        __syncthreads();
        h = h_next;
        qt = qt_next;
    }

#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int j = j_lo + r * 8;
        if (j < T) {
            __nv_bfloat16* dst = dqkv + ((size_t)b * T + j) * ld_dqkv + (lane & 3) * 2;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                *reinterpret_cast<uint32_t*>(dst + kcol + nt * 8) = pack_bf16x2(dk[nt][r * 2] * p.scale, dk[nt][r * 2 + 1] * p.scale);
                *reinterpret_cast<uint32_t*>(dst + vcol + nt * 8) = pack_bf16x2(dv[nt][r * 2], dv[nt][r * 2 + 1]);
            }
        }
    }
}

// dQ and d(logslope): grid (ceil(T/64), H, B); same tiling as the forward.
__global__ void __launch_bounds__(128, 3)
attn_bwd_dq_kernel(AttnParams p, const __nv_bfloat16* __restrict__ dout, int ld_do, const float* __restrict__ lse,
                   const float* __restrict__ delta, __nv_bfloat16* __restrict__ dqkv, int ld_dqkv,
                   float* __restrict__ dlogslopes) {
    if (p.rng_offset != nullptr) p.seed += *p.rng_offset * 0x9E3779B97F4A7C15ull;
    extern __shared__ __align__(128) uint8_t dyn_smem[];
    uint8_t* sQ = dyn_smem;
    uint8_t* sDO = sQ + TQ * 128;
    uint8_t (*sK)[TK * 128] = reinterpret_cast<uint8_t (*)[TK * 128]>(sDO + TQ * 128);
    uint8_t (*sV)[TK * 128] = reinterpret_cast<uint8_t (*)[TK * 128]>(sDO + TQ * 128 + 2 * TK * 128);
    __shared__ uint32_t sMaskAll[ATT_MAX_T / 32];    // key validity of the whole sequence, built once

    const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int T = p.T, H = p.H;
    const DropCtx drop = make_drop(p);
    const int q0 = qt * TQ;
    const int kcol = H * DH, vcol = kcol + DH;
    const __nv_bfloat16* base = p.qkv + (size_t)b * T * p.ld;
    const __nv_bfloat16* dbase = dout + (size_t)b * T * ld_do;
    const float slope_nat = __expf(p.logslopes[h]);
    const float slope = slope_nat * LOG2E;
    const float scale2 = p.scale * LOG2E;
    const int n_kt = p.causal ? min(qt + 1, ceil_div(T, TK)) : ceil_div(T, TK);

    auto load_kv = [&](int kt, int buf) {
        load_tile_async(sK[buf], base, p.ld, kt * TK, kcol, T);
        load_tile_async(sV[buf], base, p.ld, kt * TK, vcol, T);
    };
    load_tile_async(sQ, base, p.ld, q0, h * DH, T);
    load_tile_async(sDO, dbase, ld_do, q0, h * DH, T);
    load_kv(0, 0);
    cp_async_commit();
    // key-validity words for every key tile, once per CTA (a per-tile global load would sit on the critical path)
    for (int w = warp; w * 32 < n_kt * TK; w += 4) {
        const int j = w * 32 + lane;
        const bool ok = (j < T) && (p.key_mask == nullptr || p.key_mask[(size_t)b * T + j]);
        const uint32_t bits = __ballot_sync(0xffffffffu, ok);
        if (lane == 0) sMaskAll[w] = bits;
    }

    const int r_lo = q0 + warp * 16 + (lane >> 2);
    float lse_r[2], delta_r[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int i = r_lo + r * 8;
        lse_r[r] = i < T ? lse[((size_t)b * H + h) * T + i] : INFINITY;
        delta_r[r] = i < T ? delta[((size_t)b * H + h) * T + i] : 0.f;
    }
    float dq[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dq[i][j] = 0.f;
    uint32_t qf[4][4], dof[4][4];
    // d slope needs sum_j dS_ij * |i-j|.  In exact arithmetic sum_j dS_ij = 0; the bf16 rounding of O makes delta_i
    // slightly off, which would leak eps_i * E_i[|i-j|] into the sum.  Track the row residual and remove that term.
    float ds_dist[2] = {0.f, 0.f}, ds_sum[2] = {0.f, 0.f}, p_dist[2] = {0.f, 0.f};

    for (int kt = 0; kt < n_kt; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < n_kt) load_kv(kt + 1, buf ^ 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        if (kt == 0) {
            load_a_frags(smem_u32(sQ), warp * 16, lane, qf);
            load_a_frags(smem_u32(sDO), warp * 16, lane, dof);
        }
        float s[8][4], dp[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) { s[i][j] = 0.f; dp[i][j] = 0.f; }
        mma_a_tile_nt(s, qf, smem_u32(sK[buf]), lane);     // S = Q K^T
        mma_a_tile_nt(dp, dof, smem_u32(sV[buf]), lane);   // dP = dO V^T
        const uint32_t w0 = sMaskAll[kt * 2], w1 = sMaskAll[kt * 2 + 1];
        const bool diag = p.causal && (kt == qt);
        const float dbase0 = (float)(r_lo - (kt * TK + (lane & 3) * 2));
        if (diag || (w0 & w1) != 0xffffffffu) {
            // masked scores become -inf up front (P = exp2(-inf) = 0), so the main loop carries no mask logic
            const uint32_t mlo = w0 >> ((lane & 3) * 2), mhi = w1 >> ((lane & 3) * 2);
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float d = dbase0 + (float)((e >> 1) * 8 - nt * 8 - (e & 1));
                    const uint32_t word = nt < 4 ? mlo : mhi;
                    const bool ok = ((word >> ((nt & 3) * 8 + (e & 1))) & 1u) && (!diag || d >= 0.f);
                    if (!ok) s[nt][e] = -INFINITY;
                }
            }
        }
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            uint32_t hsh[2] = {0, 0};
            if (drop.on) {
#pragma unroll
                for (int rr = 0; rr < 2; ++rr)
                    hsh[rr] = pair_hash(drop, (uint32_t)((b * H + h) * T + r_lo + rr * 8), (uint32_t)(kt * TK + nt * 8 + (lane & 3) * 2));
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float d = dbase0 + (float)((e >> 1) * 8 - nt * 8 - (e & 1));
                const float dist = fabsf(d);
                const float pv = exp2f(fmaf(-slope, dist, s[nt][e] * scale2) - lse_r[e >> 1]);
                float keep = 1.f;
                if (drop.on) {
                    const uint32_t u16 = (e & 1) ? (hsh[e >> 1] >> 16) : (hsh[e >> 1] & 0xffffu);
                    keep = u16 >= drop.thr16 ? drop.keep_scale : 0.f;
                }
                const float ds = pv * (dp[nt][e] * keep - delta_r[e >> 1]);
                ds_dist[e >> 1] += ds * dist;
                ds_sum[e >> 1] += ds;
                p_dist[e >> 1] += pv * dist;
                s[nt][e] = ds;
            }
        }
        uint32_t pf[4][4];
        acc_to_frags(s, pf);
        mma_p_tile_nn(dq, pf, smem_u32(sK[buf]), lane);    // dQ += dS K
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int i = r_lo + r * 8;
        if (i < T) {
            __nv_bfloat16* dst = dqkv + ((size_t)b * T + i) * ld_dqkv + h * DH + (lane & 3) * 2;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt)
                *reinterpret_cast<uint32_t*>(dst + nt * 8) = pack_bf16x2(dq[nt][r * 2] * p.scale, dq[nt][r * 2 + 1] * p.scale);
        }
    }
    // d logslope_h = slope_h * sum_ij dS_ij * (-|i-j|)
    float dslope = 0.f;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
#pragma unroll
        for (int o = 1; o <= 2; o <<= 1) {
            ds_dist[r] += __shfl_xor_sync(0xffffffffu, ds_dist[r], o);
            ds_sum[r] += __shfl_xor_sync(0xffffffffu, ds_sum[r], o);
            p_dist[r] += __shfl_xor_sync(0xffffffffu, p_dist[r], o);
        }
        if ((lane & 3) == 0) dslope -= ds_dist[r] - ds_sum[r] * p_dist[r];
    }
    dslope = warp_sum(dslope);
    if (lane == 0 && dlogslopes != nullptr) atomicAdd(dlogslopes + h, dslope * slope_nat);
}

int fill_params(AttnParams& p, const void* qkv, int ld, const uint8_t* key_mask, const float* logslopes, int B, int T, int H,
                int dim_head, int causal, float dropout_p, uint64_t seed, const uint64_t* rng_offset) {
    p.rng_offset = rng_offset;
    SPB_CHECK_ARG(qkv && logslopes, "attention: null pointer");
    SPB_CHECK_ARG(dim_head == DH, "attention: dim_head must be %d, got %d", DH, dim_head);
    SPB_CHECK_ARG(T <= ATT_MAX_T, "attention: at most %d positions per sequence, got %d", ATT_MAX_T, T);
    SPB_CHECK_ARG(ld % 8 == 0 && ld >= H * DH + 2 * DH, "attention: qkv row stride %d too small / unaligned", ld);
    SPB_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f, "attention: dropout_p must be in [0,1)");
    p.qkv = reinterpret_cast<const __nv_bfloat16*>(qkv);
    p.ld = ld; p.key_mask = key_mask; p.logslopes = logslopes;
    p.B = B; p.T = T; p.H = H;
    p.scale = 1.f / sqrtf((float)dim_head);
    p.causal = causal;
    p.dropout_p = dropout_p;
    p.seed = seed;
    double t = (double)dropout_p * 16777216.0;
    p.drop_thresh24 = dropout_p > 0.f ? (uint32_t)(t < 1 ? 1 : t) : 0;
    p.keep_scale = 1.f / (1.f - dropout_p);
    return SPB_OK;
}

}  // namespace

// out bf16 [B*T, ld_out] (H*64 columns written); lse fp32 [B, H, T] in base-2 units (consumed only by the backward).
extern "C" int spb_attention_fwd(const void* qkv, int ld, const uint8_t* key_mask, const float* logslopes, void* out, int ld_out,
                                 float* lse, int B, int T, int H, int dim_head, int causal, float dropout_p, uint64_t seed,
                                 const uint64_t* rng_offset, cudaStream_t stream) {
    if (B <= 0 || T <= 0) return SPB_OK;
    AttnParams p;
    int rc = fill_params(p, qkv, ld, key_mask, logslopes, B, T, H, dim_head, causal, dropout_p, seed, rng_offset);
    if (rc != SPB_OK) return rc;
    SPB_CHECK_ARG(out != nullptr && ld_out % 2 == 0, "spb_attention_fwd: bad output");
    attn_fwd_kernel<<<dim3(ceil_div(T, TQ), H, B), 128, 0, stream>>>(p, reinterpret_cast<__nv_bfloat16*>(out), ld_out, lse);
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}

// dqkv bf16 [B*T, ld_dqkv]: dq | dk | dv in the qkv column layout; delta fp32 [B,H,T] scratch;
// dlogslopes fp32 [H] is ACCUMULATED into.
extern "C" int spb_attention_bwd(const void* qkv, int ld, const uint8_t* key_mask, const float* logslopes, const void* out,
                                 const void* dout, int ld_out, const float* lse, float* delta, void* dqkv, int ld_dqkv,
                                 float* dlogslopes, int B, int T, int H, int dim_head, int causal, float dropout_p,
                                 uint64_t seed, const uint64_t* rng_offset, int delta_ready, cudaStream_t stream) {
    if (B <= 0 || T <= 0) return SPB_OK;
    AttnParams p;
    int rc = fill_params(p, qkv, ld, key_mask, logslopes, B, T, H, dim_head, causal, dropout_p, seed, rng_offset);
    if (rc != SPB_OK) return rc;
    SPB_CHECK_ARG(out && dout && lse && delta && dqkv, "spb_attention_bwd: null pointer");
    if (!delta_ready) {      // delta = rowsum(dO * O); the out-projection dgrad GEMM can emit it instead (spb_gemm_bf16_rowdot)
        const int n_warps = B * T * H;
        attn_delta_kernel<<<ceil_div((int64_t)n_warps * 32, 256), 256, 0, stream>>>(
            reinterpret_cast<const __nv_bfloat16*>(out), reinterpret_cast<const __nv_bfloat16*>(dout), ld_out, delta, B, T, H);
        SPB_CHECK_LAUNCH();
    }
    constexpr int BWD_SMEM = 6 * 64 * 128;
    static bool configured = false;
    if (!configured) {
        SPB_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_dkv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD_SMEM));
        SPB_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD_SMEM));
        configured = true;
    }
    attn_bwd_dkv_kernel<<<dim3(ceil_div(T, TK), B), 128, BWD_SMEM, stream>>>(p, reinterpret_cast<const __nv_bfloat16*>(dout), ld_out, lse,
                                                                     delta, reinterpret_cast<__nv_bfloat16*>(dqkv), ld_dqkv);
    SPB_CHECK_LAUNCH();
    attn_bwd_dq_kernel<<<dim3(ceil_div(T, TQ), H, B), 128, BWD_SMEM, stream>>>(p, reinterpret_cast<const __nv_bfloat16*>(dout), ld_out, lse,
                                                                       delta, reinterpret_cast<__nv_bfloat16*>(dqkv), ld_dqkv,
                                                                       dlogslopes);
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}

// ------------------------------------------------------------------------------------------- incremental decode
// One new query position per sequence against a KV cache (modules/transformer/attention.py:155-156 + transformer.py:161-186).
// grid (B), 32*H threads: warp h = head h.  Scores: lane <-> key (16-byte loads of the key row); PV: lane <-> 2 value dims.
namespace {
constexpr int DEC_MAX_T = 4096;

__global__ void attn_decode_kernel(const __nv_bfloat16* __restrict__ q, int ld_q, const __nv_bfloat16* __restrict__ kv, int ld_kv,
                                   long long kv_batch_stride, const uint8_t* __restrict__ key_mask, int mask_stride,
                                   const float* __restrict__ logslopes, __nv_bfloat16* __restrict__ out, int ld_out, int n_keys,
                                   int q_pos, float scale, const long long* __restrict__ pos_dev, int append_kv, int n_heads) {
    extern __shared__ float sp[];                  // [H][capacity]
    const int b = blockIdx.x, h = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cap = n_keys;
    if (pos_dev != nullptr) {                      // position lives on the device: the launch is replayable from a CUDA graph
        q_pos = (int)*pos_dev;
        n_keys = min(cap, q_pos + 1);
    }
    float* p = sp + (size_t)h * cap;
    __nv_bfloat16* kvb = const_cast<__nv_bfloat16*>(kv) + (size_t)b * kv_batch_stride;
    if (append_kv) {
        // the new position's (k | v) sit right after the H query heads of this row: append them to the cache first.  A device
        // position is caller data that the host never sees: a row outside the cache is not written
        if (threadIdx.x < 16 && q_pos >= 0 && q_pos < cap)
            reinterpret_cast<uint4*>(kvb + (size_t)q_pos * ld_kv)[threadIdx.x] =
                reinterpret_cast<const uint4*>(q + (size_t)b * ld_q + n_heads * DH)[threadIdx.x];
        __syncthreads();
    }
    const float slope = __expf(logslopes[h]);
    float qv[DH];
    {
        const __nv_bfloat16* qr = q + (size_t)b * ld_q + h * DH;
#pragma unroll
        for (int c = 0; c < DH / 8; ++c) {
            const uint4 u = *reinterpret_cast<const uint4*>(qr + c * 8);
            const float2 a = unpack_bf16x2(u.x), b2 = unpack_bf16x2(u.y), c2 = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
            qv[c * 8 + 0] = a.x; qv[c * 8 + 1] = a.y; qv[c * 8 + 2] = b2.x; qv[c * 8 + 3] = b2.y;
            qv[c * 8 + 4] = c2.x; qv[c * 8 + 5] = c2.y; qv[c * 8 + 6] = d.x; qv[c * 8 + 7] = d.y;
        }
    }
    float mx = -INFINITY;
    for (int j = lane; j < n_keys; j += 32) {
        const bool ok = (key_mask == nullptr || key_mask[(size_t)b * mask_stride + j]) && j <= q_pos;
        float s = -INFINITY;
        if (ok) {
            const __nv_bfloat16* kr = kvb + (size_t)j * ld_kv;
            float acc = 0.f;
#pragma unroll
            for (int c = 0; c < DH / 8; ++c) {
                const uint4 u = *reinterpret_cast<const uint4*>(kr + c * 8);
                const float2 a = unpack_bf16x2(u.x), b2 = unpack_bf16x2(u.y), c2 = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
                acc += qv[c * 8] * a.x + qv[c * 8 + 1] * a.y + qv[c * 8 + 2] * b2.x + qv[c * 8 + 3] * b2.y + qv[c * 8 + 4] * c2.x +
                       qv[c * 8 + 5] * c2.y + qv[c * 8 + 6] * d.x + qv[c * 8 + 7] * d.y;
            }
            s = acc * scale - slope * fabsf((float)(q_pos - j));
        }
        p[j] = s;
        mx = fmaxf(mx, s);
    }
    mx = warp_max(mx);
    const float m_use = mx == -INFINITY ? 0.f : mx;
    float sum = 0.f;
    for (int j = lane; j < n_keys; j += 32) {
        const float e = __expf(p[j] - m_use);
        p[j] = e;
        sum += e;
    }
    sum = warp_sum(sum);
    __syncwarp();
    const float inv = sum > 0.f ? 1.f / sum : 0.f;
    // P.V: 8 lanes cover the 64 value dims with 16-byte loads, the 4 lane groups walk 4 different keys, two keys per group in
    // flight; the groups' partial sums meet through shuffles at the end.
    const int grp = lane >> 3, sub = lane & 7;
    float o[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) o[e] = 0.f;
    const __nv_bfloat16* vbase = kvb + DH + sub * 8;
    int j = grp;
    for (; j + 4 < n_keys; j += 8) {
        const float p0 = p[j], p1 = p[j + 4];
        const uint4 u0 = *reinterpret_cast<const uint4*>(vbase + (size_t)j * ld_kv);
        const uint4 u1 = *reinterpret_cast<const uint4*>(vbase + (size_t)(j + 4) * ld_kv);
        const float2 a0 = unpack_bf16x2(u0.x), a1 = unpack_bf16x2(u0.y), a2 = unpack_bf16x2(u0.z), a3 = unpack_bf16x2(u0.w);
        const float2 b0 = unpack_bf16x2(u1.x), b1 = unpack_bf16x2(u1.y), b2 = unpack_bf16x2(u1.z), b3 = unpack_bf16x2(u1.w);
        o[0] += p0 * a0.x + p1 * b0.x; o[1] += p0 * a0.y + p1 * b0.y; o[2] += p0 * a1.x + p1 * b1.x; o[3] += p0 * a1.y + p1 * b1.y;
        o[4] += p0 * a2.x + p1 * b2.x; o[5] += p0 * a2.y + p1 * b2.y; o[6] += p0 * a3.x + p1 * b3.x; o[7] += p0 * a3.y + p1 * b3.y;
    }
    for (; j < n_keys; j += 4) {
        const float p0 = p[j];
        const uint4 u0 = *reinterpret_cast<const uint4*>(vbase + (size_t)j * ld_kv);
        const float2 a0 = unpack_bf16x2(u0.x), a1 = unpack_bf16x2(u0.y), a2 = unpack_bf16x2(u0.z), a3 = unpack_bf16x2(u0.w);
        o[0] += p0 * a0.x; o[1] += p0 * a0.y; o[2] += p0 * a1.x; o[3] += p0 * a1.y;
        o[4] += p0 * a2.x; o[5] += p0 * a2.y; o[6] += p0 * a3.x; o[7] += p0 * a3.y;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        o[e] += __shfl_xor_sync(0xffffffffu, o[e], 8);
        o[e] += __shfl_xor_sync(0xffffffffu, o[e], 16);
    }
    if (grp == 0) {
        const uint4 r = make_uint4(pack_bf16x2(o[0] * inv, o[1] * inv), pack_bf16x2(o[2] * inv, o[3] * inv),
                                   pack_bf16x2(o[4] * inv, o[5] * inv), pack_bf16x2(o[6] * inv, o[7] * inv));
        *reinterpret_cast<uint4*>(out + (size_t)b * ld_out + h * DH + sub * 8) = r;
    }
}
}  // namespace

// q bf16 [B, >= H*64] (row stride ld_q); kv bf16 cache [B][n_keys rows of (k | v) = 128 columns] (row stride ld_kv, batch stride in
// elements); key_mask [B, mask_stride] or NULL; out bf16 [B, H*64].  The query sits at position q_pos (keys j <= q_pos attend).
// pos_dev (optional): device int64 holding q_pos; n_keys is then the cache CAPACITY and keys j <= *pos_dev are used.
// append_kv: copy columns [H*64, H*64+128) of each q row into cache row q_pos before attending (saves a separate copy); a device
// position outside [0, capacity) appends nothing.  H * n_keys fp32 scores must fit the device's shared memory per block.
extern "C" int spb_attention_decode(const void* q, int ld_q, void* kv, int ld_kv, long long kv_batch_stride, const uint8_t* key_mask,
                                    int mask_stride, const float* logslopes, void* out, int ld_out, int B, int H, int dim_head,
                                    int n_keys, int q_pos, const int64_t* pos_dev, int append_kv, cudaStream_t stream) {
    if (B <= 0 || n_keys <= 0) return SPB_OK;
    SPB_CHECK_ARG(q && kv && logslopes && out, "spb_attention_decode: null pointer");
    SPB_CHECK_ARG(dim_head == DH && H >= 1 && H <= 32, "spb_attention_decode: dim_head must be %d, 1..32 heads", DH);
    SPB_CHECK_ARG(n_keys <= DEC_MAX_T, "spb_attention_decode: at most %d cached keys", DEC_MAX_T);
    SPB_CHECK_ARG(ld_q % 8 == 0 && ld_kv % 8 == 0 && ld_out % 8 == 0, "spb_attention_decode: leading dims must be multiples of 8");
    SPB_CHECK_ARG(pos_dev != nullptr || !append_kv || (q_pos >= 0 && q_pos < n_keys),
                  "spb_attention_decode: append_kv needs 0 <= q_pos < n_keys, got q_pos %d, n_keys %d", q_pos, n_keys);
    const size_t smem = (size_t)H * n_keys * sizeof(float);
    static int smem_max = 0;
    if (smem_max == 0) {
        int dev = 0;
        SPB_CHECK_CUDA(cudaGetDevice(&dev));
        SPB_CHECK_CUDA(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    }
    SPB_CHECK_ARG(smem <= (size_t)smem_max, "spb_attention_decode: %d heads x %d keys need %zu bytes of shared memory, the device has %d per block",
                  H, n_keys, smem, smem_max);
    static size_t configured = 48 * 1024;
    if (smem > configured) {
        SPB_CHECK_CUDA(cudaFuncSetAttribute(attn_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    attn_decode_kernel<<<B, 32 * H, smem, stream>>>(reinterpret_cast<const __nv_bfloat16*>(q), ld_q, reinterpret_cast<const __nv_bfloat16*>(kv),
                                                   ld_kv, kv_batch_stride, key_mask, mask_stride, logslopes,
                                                   reinterpret_cast<__nv_bfloat16*>(out), ld_out, n_keys, q_pos, 1.f / sqrtf((float)dim_head),
                                                   reinterpret_cast<const long long*>(pos_dev), append_kv, H);
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}
