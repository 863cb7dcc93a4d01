// Row-wise (HBM-bound) kernels of the ScorePerformer step: LayerNorm / AdaptiveLayerNorm forward+backward,
// GLU(SiLU) forward+backward with in-kernel dropout, and the fused SPMuple tuple-token embedding
// (per-field table gather -> concat -> LayerNorm) forward+backward.
//
// Reference semantics:
//   LayerNorm / AdaLN      modules/layers.py:31-47, nn.LayerNorm (eps 1e-5)
//   GLU + dropout          modules/transformer/feedforward.py:13-22,56-61
//   tuple embedding        models/scoreperformer/embeddings.py:121-143 (gather, cat, LayerNorm(E*F))
// One warp owns one row; 128-bit loads; per-row statistics by warp shuffles; parameter gradients are
// accumulated in registers across the rows a warp visits, reduced through shared memory and flushed with
// one fp32 atomic per column per CTA.
#include "common.cuh"

namespace {

constexpr int ROW_WARPS = 8;

template <typename T>
struct Ld8;  // load / store 8 contiguous elements as floats
template <>
struct Ld8<float> {
    static __device__ __forceinline__ void load(const float* p, float* v) {
        float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
    static __device__ __forceinline__ void store(float* p, const float* v) {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
    }
};
template <>
struct Ld8<__nv_bfloat16> {
    static __device__ __forceinline__ void load(const __nv_bfloat16* p, float* v) {
        uint4 u = *reinterpret_cast<const uint4*>(p);
        float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
    }
    static __device__ __forceinline__ void store(__nv_bfloat16* p, const float* v) {
        uint4 u;
        u.x = pack_bf16x2(v[0], v[1]); u.y = pack_bf16x2(v[2], v[3]);
        u.z = pack_bf16x2(v[4], v[5]); u.w = pack_bf16x2(v[6], v[7]);
        *reinterpret_cast<uint4*>(p) = u;
    }
};

// ------------------------------------------------------------------------------------------- LayerNorm
// D = 256 * G.  Lane l owns elements g*256 + l*8 + j (g < G, j < 8).
template <int G, typename Tin, typename Tout, bool ADA>
__global__ void __launch_bounds__(ROW_WARPS * 32, G >= 5 ? 2 : 1)
ln_fwd_kernel(const Tin* __restrict__ x, int ldx, const float* __restrict__ w, const float* __restrict__ b,
              const __nv_bfloat16* __restrict__ gb, int ldgb, Tout* __restrict__ y, int ldy, float* __restrict__ mean_out,
              float* __restrict__ rstd_out, int n_rows, float eps) {
    constexpr int D = 256 * G;
    const int lane = threadIdx.x & 31;
    const int warp_global = blockIdx.x * ROW_WARPS + (threadIdx.x >> 5);
    const int warp_stride = gridDim.x * ROW_WARPS;
    for (int row = warp_global; row < n_rows; row += warp_stride) {
        float v[G][8];
        float s = 0.f;
#pragma unroll
        for (int g = 0; g < G; ++g) {
            Ld8<Tin>::load(x + (size_t)row * ldx + g * 256 + lane * 8, v[g]);
#pragma unroll
            for (int j = 0; j < 8; ++j) s += v[g][j];
        }
        const float mean = warp_sum(s) * (1.f / D);
        float sq = 0.f;
#pragma unroll
        for (int g = 0; g < G; ++g)
#pragma unroll
            for (int j = 0; j < 8; ++j) { const float d = v[g][j] - mean; sq += d * d; }
        const float rstd = rsqrtf(warp_sum(sq) * (1.f / D) + eps);
        if (lane == 0) {
            if (mean_out) mean_out[row] = mean;
            if (rstd_out) rstd_out[row] = rstd;
        }
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const int c = g * 256 + lane * 8;
            float gam[8], bet[8], o[8];
            if (ADA) {
                // gb holds (gamma - 1 | beta): gamma sits near its initial value 1 (layers.py:38-40), and bf16 keeps eight bits of
                // the small deviation instead of eight bits of 1.0x
                Ld8<__nv_bfloat16>::load(gb + (size_t)row * ldgb + c, gam);
                Ld8<__nv_bfloat16>::load(gb + (size_t)row * ldgb + D + c, bet);
#pragma unroll
                for (int j = 0; j < 8; ++j) gam[j] += 1.f;
            } else {
                Ld8<float>::load(w + c, gam);
                Ld8<float>::load(b + c, bet);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = (v[g][j] - mean) * rstd * gam[j] + bet[j];
            Ld8<Tout>::store(y + (size_t)row * ldy + c, o);
        }
    }
}

// dx = rstd * (dy*gamma - mean(dy*gamma) - xhat * mean(dy*gamma*xhat)) (+ dres);  dw += dy*xhat; db += dy
template <int G, typename Tin, typename Tdx, bool ADA>
__global__ void __launch_bounds__(ROW_WARPS * 32)
ln_bwd_kernel(const __nv_bfloat16* __restrict__ dy, int lddy, const Tin* __restrict__ x, int ldx,
              const float* __restrict__ mean_in, const float* __restrict__ rstd_in, const float* __restrict__ w,
              const __nv_bfloat16* __restrict__ gb, int ldgb, const float* __restrict__ dres, int lddres,
              Tdx* __restrict__ dx, int lddx, float* __restrict__ dw, float* __restrict__ db,
              __nv_bfloat16* __restrict__ dgb, int lddgb, __nv_bfloat16* __restrict__ dx16, int lddx16,
              const uint8_t* __restrict__ dx16_rowmask, int n_rows) {
    constexpr int D = 256 * G;
    __shared__ float red[ROW_WARPS][256];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int warp_global = blockIdx.x * ROW_WARPS + warp;
    const int warp_stride = gridDim.x * ROW_WARPS;
    float acc_w[G][8], acc_b[G][8];
#pragma unroll
    for (int g = 0; g < G; ++g)
#pragma unroll
        for (int j = 0; j < 8; ++j) { acc_w[g][j] = 0.f; acc_b[g][j] = 0.f; }

    for (int row = warp_global; row < n_rows; row += warp_stride) {
        const float mean = mean_in[row], rstd = rstd_in[row];
        float xh[G][8], dyw[G][8];
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const int c = g * 256 + lane * 8;
            float xv[8], dv[8], gam[8];
            Ld8<Tin>::load(x + (size_t)row * ldx + c, xv);
            Ld8<__nv_bfloat16>::load(dy + (size_t)row * lddy + c, dv);
            if (ADA) {
                Ld8<__nv_bfloat16>::load(gb + (size_t)row * ldgb + c, gam);
#pragma unroll
                for (int j = 0; j < 8; ++j) gam[j] += 1.f;       // gb = (gamma - 1 | beta), see ln_fwd_kernel
            } else {
                Ld8<float>::load(w + c, gam);
            }
            float dgam[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                xh[g][j] = (xv[j] - mean) * rstd;
                dyw[g][j] = dv[j] * gam[j];
                s1 += dyw[g][j];
                s2 += dyw[g][j] * xh[g][j];
                dgam[j] = dv[j] * xh[g][j];
                if (!ADA) { acc_w[g][j] += dgam[j]; acc_b[g][j] += dv[j]; }
            }
            if (ADA) {
                Ld8<__nv_bfloat16>::store(dgb + (size_t)row * lddgb + c, dgam);
                Ld8<__nv_bfloat16>::store(dgb + (size_t)row * lddgb + D + c, dv);
            }
        }
        const float c1 = warp_sum(s1) * (1.f / D), c2 = warp_sum(s2) * (1.f / D);
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const int c = g * 256 + lane * 8;
            float o[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = rstd * (dyw[g][j] - c1 - xh[g][j] * c2);
            if (dres != nullptr) {
                float r[8];
                Ld8<float>::load(dres + (size_t)row * lddres + c, r);
#pragma unroll
                for (int j = 0; j < 8; ++j) o[j] += r[j];
            }
            Ld8<Tdx>::store(dx + (size_t)row * lddx + c, o);
            if (dx16 != nullptr) {     // bf16 (optionally row-masked) copy for the next backward GEMM: saves a separate cast pass
                if (dx16_rowmask != nullptr && !dx16_rowmask[row]) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) o[j] = 0.f;
                }
                Ld8<__nv_bfloat16>::store(dx16 + (size_t)row * lddx16 + c, o);
            }
        }
    }
    if (!ADA && dw != nullptr) {
#pragma unroll
        for (int g = 0; g < G; ++g) {
            for (int pass = 0; pass < 2; ++pass) {
                __syncthreads();
#pragma unroll
                for (int j = 0; j < 8; ++j) red[warp][lane * 8 + j] = pass == 0 ? acc_w[g][j] : acc_b[g][j];
                __syncthreads();
                const int c = threadIdx.x;  // 256 threads == 256 columns of this group
                float s = 0.f;
#pragma unroll
                for (int k = 0; k < ROW_WARPS; ++k) s += red[k][c];
                atomicAdd((pass == 0 ? dw : db) + g * 256 + c, s);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------- GLU (SiLU)
// u: [n, 2H] (value | gate) -> h[n, H] = value * silu(gate) * dropout_keep / (1-p);  8 elements (16 bytes) per thread
__global__ void __launch_bounds__(256)
glu_fwd_kernel(const __nv_bfloat16* __restrict__ u, __nv_bfloat16* __restrict__ h, int n_rows, int H, uint64_t seed,
               const uint64_t* __restrict__ rng_offset, uint32_t thr32, float keep_scale) {
    if (rng_offset != nullptr) seed += *rng_offset * 0x9E3779B97F4A7C15ull;
    const uint32_t seed32 = spb_seed32(seed);
    const int per_row = H / 8;
    const int64_t total = (int64_t)n_rows * per_row;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int row = (int)(i / per_row);
        const int c = (int)(i % per_row) * 8;
        float xs[8], gs[8], o[8];
        Ld8<__nv_bfloat16>::load(u + (size_t)row * 2 * H + c, xs);
        Ld8<__nv_bfloat16>::load(u + (size_t)row * 2 * H + H + c, gs);
        const uint32_t quad0 = (uint32_t)row * (uint32_t)(H >> 2) + (uint32_t)(c >> 2);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float sig = 1.f / (1.f + __expf(-gs[j]));
            o[j] = xs[j] * gs[j] * sig;
        }
        if (thr32 != 0) {         // the mask function of the fused feed-forward kernel (ffn.cu) and of glu_bwd_kernel
#pragma unroll
            for (int j = 0; j < 8; j += 4) {
                const uint32_t qh = spb_quad_hash(seed32, quad0 + (uint32_t)(j >> 2));
#pragma unroll
                for (int e = 0; e < 4; ++e) o[j + e] = spb_quad_keep(qh, e, thr32) ? o[j + e] * keep_scale : 0.f;
            }
        }
        Ld8<__nv_bfloat16>::store(h + (size_t)row * H + c, o);
    }
}

// du[n, 2H] from dh[n, H]; dbias[2H] += column sums of du.  Block b walks rows b, b+grid, ...; thread t owns
// the 4-column groups t, t+256, ... so column sums accumulate in registers (H <= 4096).
// (8-byte accesses on purpose: the 16-byte / 8-column form needs ~90 registers, drops to 2 blocks per SM and measured
//  15-40% slower on B200 in two separate attempts -- bytes in flight per SM matter more than bytes per instruction here.)
template <int MAXG>
__global__ void __launch_bounds__(256)
glu_bwd_kernel(const __nv_bfloat16* __restrict__ dh, const __nv_bfloat16* __restrict__ u, __nv_bfloat16* __restrict__ du,
               float* __restrict__ dbias, int n_rows, int H, uint64_t seed, const uint64_t* __restrict__ rng_offset,
               uint32_t thr32, float keep_scale) {
    if (rng_offset != nullptr) seed += *rng_offset * 0x9E3779B97F4A7C15ull;
    const uint32_t seed32 = spb_seed32(seed);
    float sx[MAXG][4], sg[MAXG][4];
#pragma unroll
    for (int k = 0; k < MAXG; ++k)
#pragma unroll
        for (int j = 0; j < 4; ++j) { sx[k][j] = 0.f; sg[k][j] = 0.f; }
    for (int row = blockIdx.x; row < n_rows; row += gridDim.x) {
#pragma unroll
        for (int k = 0; k < MAXG; ++k) {
            const int c = (k * 256 + threadIdx.x) * 4;
            if (c < H) {
                const uint2 dv = *reinterpret_cast<const uint2*>(dh + (size_t)row * H + c);
                const uint2 xv = *reinterpret_cast<const uint2*>(u + (size_t)row * 2 * H + c);
                const uint2 gv = *reinterpret_cast<const uint2*>(u + (size_t)row * 2 * H + H + c);
                const float2 d0 = unpack_bf16x2(dv.x), d1 = unpack_bf16x2(dv.y);
                const float2 x0 = unpack_bf16x2(xv.x), x1 = unpack_bf16x2(xv.y);
                const float2 g0 = unpack_bf16x2(gv.x), g1 = unpack_bf16x2(gv.y);
                float ds[4] = {d0.x, d0.y, d1.x, d1.y}, xs[4] = {x0.x, x0.y, x1.x, x1.y}, gs[4] = {g0.x, g0.y, g1.x, g1.y};
                float ox[4], og[4];
                if (thr32 != 0) {      // same (seed, quad) hashes as the forward kernels
                    const uint32_t qh = spb_quad_hash(seed32, (uint32_t)row * (uint32_t)(H >> 2) + (uint32_t)(c >> 2));
#pragma unroll
                    for (int j = 0; j < 4; ++j) ds[j] = spb_quad_keep(qh, j, thr32) ? ds[j] * keep_scale : 0.f;
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float d = ds[j];
                    const float sig = 1.f / (1.f + __expf(-gs[j]));
                    const float silu = gs[j] * sig;
                    ox[j] = d * silu;
                    og[j] = d * xs[j] * sig * (1.f + gs[j] * (1.f - sig));
                    // accumulate the bias gradient from the *rounded* values that flow on, like autograd would
                    sx[k][j] += ox[j];
                    sg[k][j] += og[j];
                }
                uint2 o1, o2;
                o1.x = pack_bf16x2(ox[0], ox[1]); o1.y = pack_bf16x2(ox[2], ox[3]);
                o2.x = pack_bf16x2(og[0], og[1]); o2.y = pack_bf16x2(og[2], og[3]);
                *reinterpret_cast<uint2*>(du + (size_t)row * 2 * H + c) = o1;
                *reinterpret_cast<uint2*>(du + (size_t)row * 2 * H + H + c) = o2;
            }
        }
    }
    if (dbias != nullptr) {
#pragma unroll
        for (int k = 0; k < MAXG; ++k) {
            const int c = (k * 256 + threadIdx.x) * 4;
            if (c < H) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    atomicAdd(dbias + c + j, sx[k][j]);
                    atomicAdd(dbias + H + c + j, sg[k][j]);
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------- tuple embedding

// out[n, F*128] = LayerNorm_{F*128}( cat_f table[offset_f + tokens[n, f]] ); one warp per tuple.
template <int F>
__global__ void __launch_bounds__(ROW_WARPS * 32)
embed_ln_fwd_kernel(const int64_t* __restrict__ tokens, int ld_tok, const float* __restrict__ table, FieldTable ft,
                    const float* __restrict__ w, const float* __restrict__ b, __nv_bfloat16* __restrict__ out, int ld_out,
                    float* __restrict__ mean_out, float* __restrict__ rstd_out, int n_rows, float eps) {
    constexpr int D = F * 128;
    const int lane = threadIdx.x & 31;
    const int warp_global = blockIdx.x * ROW_WARPS + (threadIdx.x >> 5);
    for (int row = warp_global; row < n_rows; row += gridDim.x * ROW_WARPS) {
        long long tok = 0;
        if (lane < F) {
            tok = tokens[(size_t)row * ld_tok + lane];
            tok = tok < 0 ? 0 : (tok >= ft.size[lane] ? ft.size[lane] - 1 : tok);
            tok += ft.offset[lane];
        }
        float4 v[F];
        float s = 0.f;
#pragma unroll
        for (int f = 0; f < F; ++f) {
            const int r = (int)__shfl_sync(0xffffffffu, (int)tok, f);
            v[f] = *reinterpret_cast<const float4*>(table + (size_t)r * 128 + lane * 4);
            s += v[f].x + v[f].y + v[f].z + v[f].w;
        }
        const float mean = warp_sum(s) * (1.f / D);
        float sq = 0.f;
#pragma unroll
        for (int f = 0; f < F; ++f) {
            const float a = v[f].x - mean, bb = v[f].y - mean, c = v[f].z - mean, d = v[f].w - mean;
            sq += a * a + bb * bb + c * c + d * d;
        }
        const float rstd = rsqrtf(warp_sum(sq) * (1.f / D) + eps);
        if (lane == 0) { mean_out[row] = mean; rstd_out[row] = rstd; }
#pragma unroll
        for (int f = 0; f < F; ++f) {
            const int c = f * 128 + lane * 4;
            const float4 g = *reinterpret_cast<const float4*>(w + c), be = *reinterpret_cast<const float4*>(b + c);
            uint2 o;
            o.x = pack_bf16x2((v[f].x - mean) * rstd * g.x + be.x, (v[f].y - mean) * rstd * g.y + be.y);
            o.y = pack_bf16x2((v[f].z - mean) * rstd * g.z + be.z, (v[f].w - mean) * rstd * g.w + be.w);
            *reinterpret_cast<uint2*>(out + (size_t)row * ld_out + c) = o;
        }
    }
}

// Backward pass 1: per-tuple c1 = mean(dy*w), c2 = mean(dy*w*xhat); dw += dy*xhat, db += dy.
template <int F>
__global__ void __launch_bounds__(ROW_WARPS * 32, 2)
embed_ln_bwd_stats_kernel(const __nv_bfloat16* __restrict__ dy, int ld_dy, const int64_t* __restrict__ tokens, int ld_tok,
                          const float* __restrict__ table, FieldTable ft, const float* __restrict__ w,
                          const float* __restrict__ mean_in, const float* __restrict__ rstd_in, float* __restrict__ c1_out,
                          float* __restrict__ c2_out, float* __restrict__ dw, float* __restrict__ db, int n_rows) {
    constexpr int D = F * 128;
    __shared__ float red[ROW_WARPS][128];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    float aw[F][4], ab[F][4];
#pragma unroll
    for (int f = 0; f < F; ++f)
#pragma unroll
        for (int j = 0; j < 4; ++j) { aw[f][j] = 0.f; ab[f][j] = 0.f; }
    for (int row = blockIdx.x * ROW_WARPS + warp; row < n_rows; row += gridDim.x * ROW_WARPS) {
        long long tok = 0;
        if (lane < F) {
            tok = tokens[(size_t)row * ld_tok + lane];
            tok = tok < 0 ? 0 : (tok >= ft.size[lane] ? ft.size[lane] - 1 : tok);
            tok += ft.offset[lane];
        }
        const float mean = mean_in[row], rstd = rstd_in[row];
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int f = 0; f < F; ++f) {
            const int r = (int)__shfl_sync(0xffffffffu, (int)tok, f);
            const int c = f * 128 + lane * 4;
            const float4 xv = *reinterpret_cast<const float4*>(table + (size_t)r * 128 + lane * 4);
            const uint2 dv = *reinterpret_cast<const uint2*>(dy + (size_t)row * ld_dy + c);
            const float4 g = *reinterpret_cast<const float4*>(w + c);
            const float2 d0 = unpack_bf16x2(dv.x), d1 = unpack_bf16x2(dv.y);
            const float ds[4] = {d0.x, d0.y, d1.x, d1.y}, xs[4] = {xv.x, xv.y, xv.z, xv.w}, gs[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float xh = (xs[j] - mean) * rstd;
                s1 += ds[j] * gs[j];
                s2 += ds[j] * gs[j] * xh;
                aw[f][j] += ds[j] * xh;
                ab[f][j] += ds[j];
            }
        }
        s1 = warp_sum(s1) * (1.f / D);
        s2 = warp_sum(s2) * (1.f / D);
        if (lane == 0) { c1_out[row] = s1; c2_out[row] = s2; }
    }
#pragma unroll
    for (int f = 0; f < F; ++f) {
        for (int pass = 0; pass < 2; ++pass) {
            __syncthreads();
#pragma unroll
            for (int j = 0; j < 4; ++j) red[warp][lane * 4 + j] = pass == 0 ? aw[f][j] : ab[f][j];
            __syncthreads();
            if (threadIdx.x < 128) {
                float s = 0.f;
#pragma unroll
                for (int k = 0; k < ROW_WARPS; ++k) s += red[k][threadIdx.x];
                atomicAdd((pass == 0 ? dw : db) + f * 128 + threadIdx.x, s);
            }
        }
    }
}

int row_grid(int n_rows) {
    int blocks = ceil_div(n_rows, ROW_WARPS);
    int cap = spb_num_sms() * 8;
    return blocks < cap ? (blocks < 1 ? 1 : blocks) : cap;
}

}  // namespace

// ------------------------------------------------------------------------------------------- C-ABI
// dtype codes: 0 = bf16, 1 = fp32
extern "C" int spb_layer_norm_fwd(const void* x, int x_fp32, int ldx, const float* w, const float* b, const void* gb, int ldgb,
                                  void* y, int y_fp32, int ldy, float* mean, float* rstd, int n_rows, int dim, float eps,
                                  cudaStream_t stream) {
    if (n_rows <= 0) return SPB_OK;
    SPB_CHECK_ARG(x && y, "spb_layer_norm_fwd: null pointer");
    SPB_CHECK_ARG((gb != nullptr) != (w != nullptr && b != nullptr), "spb_layer_norm_fwd: pass either (w,b) or gb");
    SPB_CHECK_ARG(ldx % 8 == 0 && ldy % 8 == 0 && (gb == nullptr || ldgb % 8 == 0), "spb_layer_norm_fwd: leading dims must be multiples of 8");
    const bool ada = gb != nullptr;
    const int grid = row_grid(n_rows), thr = ROW_WARPS * 32;
    const __nv_bfloat16* gbp = reinterpret_cast<const __nv_bfloat16*>(gb);
#define LN_FWD(G, TI, TO, A)                                                                                              \
    ln_fwd_kernel<G, TI, TO, A><<<grid, thr, 0, stream>>>(reinterpret_cast<const TI*>(x), ldx, w, b, gbp, ldgb,          \
                                                          reinterpret_cast<TO*>(y), ldy, mean, rstd, n_rows, eps)
    if (dim == 256 && x_fp32 && !y_fp32 && !ada) LN_FWD(1, float, __nv_bfloat16, false);
    else if (dim == 256 && x_fp32 && !y_fp32 && ada) LN_FWD(1, float, __nv_bfloat16, true);
    else if (dim == 256 && x_fp32 && y_fp32 && !ada) LN_FWD(1, float, float, false);
    else if (dim == 256 && x_fp32 && y_fp32 && ada) LN_FWD(1, float, float, true);
    else if (dim == 256 && !x_fp32 && !y_fp32 && !ada) LN_FWD(1, __nv_bfloat16, __nv_bfloat16, false);
    else if (dim == 256 && !x_fp32 && y_fp32 && !ada) LN_FWD(1, __nv_bfloat16, float, false);
    else if (dim == 1536 && !x_fp32 && !y_fp32 && !ada) LN_FWD(6, __nv_bfloat16, __nv_bfloat16, false);
    else if (dim == 1536 && x_fp32 && !y_fp32 && !ada) LN_FWD(6, float, __nv_bfloat16, false);
    else if (dim == 1280 && !x_fp32 && !y_fp32 && !ada) LN_FWD(5, __nv_bfloat16, __nv_bfloat16, false);
    else if (dim == 512 && x_fp32 && !y_fp32 && !ada) LN_FWD(2, float, __nv_bfloat16, false);
    else if (dim == 512 && x_fp32 && !y_fp32 && ada) LN_FWD(2, float, __nv_bfloat16, true);
    else {
        spb_set_error("spb_layer_norm_fwd: unsupported combination dim=%d x_fp32=%d y_fp32=%d ada=%d", dim, x_fp32, y_fp32, (int)ada);
        return SPB_ERR_ARG;
    }
#undef LN_FWD
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}

extern "C" int spb_layer_norm_bwd(const void* dy, int lddy, const void* x, int x_fp32, int ldx, const float* mean,
                                  const float* rstd, const float* w, const void* gb, int ldgb, const float* dres, int lddres,
                                  void* dx, int dx_fp32, int lddx, float* dw, float* db, void* dgb, int lddgb, void* dx16,
                                  int lddx16, const uint8_t* dx16_rowmask, int n_rows, int dim, cudaStream_t stream) {
    if (n_rows <= 0) return SPB_OK;
    SPB_CHECK_ARG(dy && x && dx && mean && rstd, "spb_layer_norm_bwd: null pointer");
    const bool ada = gb != nullptr;
    SPB_CHECK_ARG(ada ? dgb != nullptr : w != nullptr, "spb_layer_norm_bwd: missing weight / dgb");
    int grid = row_grid(n_rows);
    if (grid > 2 * spb_num_sms()) grid = 2 * spb_num_sms();
    const int thr = ROW_WARPS * 32;
    const __nv_bfloat16* dyp = reinterpret_cast<const __nv_bfloat16*>(dy);
    const __nv_bfloat16* gbp = reinterpret_cast<const __nv_bfloat16*>(gb);
    __nv_bfloat16* dgbp = reinterpret_cast<__nv_bfloat16*>(dgb);
#define LN_BWD(G, TI, TD, A)                                                                                              \
    ln_bwd_kernel<G, TI, TD, A><<<grid, thr, 0, stream>>>(dyp, lddy, reinterpret_cast<const TI*>(x), ldx, mean, rstd, w, \
                                                          gbp, ldgb, dres, lddres, reinterpret_cast<TD*>(dx), lddx, dw,  \
                                                          db, dgbp, lddgb, reinterpret_cast<__nv_bfloat16*>(dx16), lddx16,  \
                                                          dx16_rowmask, n_rows)
    if (dim == 256 && x_fp32 && dx_fp32 && !ada) LN_BWD(1, float, float, false);
    else if (dim == 256 && x_fp32 && dx_fp32 && ada) LN_BWD(1, float, float, true);
    else if (dim == 256 && x_fp32 && !dx_fp32 && !ada) LN_BWD(1, float, __nv_bfloat16, false);
    else if (dim == 256 && !x_fp32 && !dx_fp32 && !ada) LN_BWD(1, __nv_bfloat16, __nv_bfloat16, false);
    else if (dim == 1536 && !x_fp32 && !dx_fp32 && !ada) LN_BWD(6, __nv_bfloat16, __nv_bfloat16, false);
    else if (dim == 1536 && x_fp32 && !dx_fp32 && !ada) LN_BWD(6, float, __nv_bfloat16, false);
    else if (dim == 1280 && !x_fp32 && !dx_fp32 && !ada) LN_BWD(5, __nv_bfloat16, __nv_bfloat16, false);
    else {
        spb_set_error("spb_layer_norm_bwd: unsupported combination dim=%d x_fp32=%d dx_fp32=%d ada=%d", dim, x_fp32, dx_fp32, (int)ada);
        return SPB_ERR_ARG;
    }
#undef LN_BWD
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}

static inline uint32_t drop_thresh(float p) {
    if (p <= 0.f) return 0;
    double t = (double)p * 16777216.0;
    return (uint32_t)(t < 1 ? 1 : (t > 16777215.0 ? 16777215.0 : t));
}

extern "C" int spb_glu_fwd(const void* u, void* h, int n_rows, int hidden, float dropout_p, uint64_t seed, const uint64_t* rng_offset,
                           cudaStream_t stream) {
    if (n_rows <= 0) return SPB_OK;
    SPB_CHECK_ARG(u && h && hidden % 8 == 0, "spb_glu_fwd: hidden must be a multiple of 8");
    const int64_t total = (int64_t)n_rows * hidden / 8;
    int64_t blocks = (total + 255) / 256;
    if (blocks > spb_num_sms() * 16) blocks = spb_num_sms() * 16;
    glu_fwd_kernel<<<(int)blocks, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(u), reinterpret_cast<__nv_bfloat16*>(h),
                                                    n_rows, hidden, seed, rng_offset, spb_drop_thr32(dropout_p), 1.f / (1.f - dropout_p));
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}

extern "C" int spb_glu_bwd(const void* dh, const void* u, void* du, float* dbias, int n_rows, int hidden, float dropout_p,
                           uint64_t seed, const uint64_t* rng_offset, cudaStream_t stream) {
    if (n_rows <= 0) return SPB_OK;
    SPB_CHECK_ARG(dh && u && du && hidden % 4 == 0 && hidden <= 4096, "spb_glu_bwd: bad arguments (hidden <= 4096, multiple of 4)");
    int grid = spb_num_sms() * 4;
    if (grid > n_rows) grid = n_rows;
    const uint32_t th = spb_drop_thr32(dropout_p);
    const float ks = 1.f / (1.f - dropout_p);
    if (hidden <= 1024)
        glu_bwd_kernel<1><<<grid, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(dh), reinterpret_cast<const __nv_bfloat16*>(u),
                                                    reinterpret_cast<__nv_bfloat16*>(du), dbias, n_rows, hidden, seed, rng_offset, th, ks);
    else
        glu_bwd_kernel<4><<<grid, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(dh), reinterpret_cast<const __nv_bfloat16*>(u),
                                                    reinterpret_cast<__nv_bfloat16*>(du), dbias, n_rows, hidden, seed, rng_offset, th, ks);
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}

static int fill_field_table(FieldTable& ft, const int* sizes, int n_fields) {
    SPB_CHECK_ARG(n_fields > 0 && n_fields <= MAX_FIELDS, "tuple embedding: 1..%d fields supported, got %d", MAX_FIELDS, n_fields);
    ft.n_fields = n_fields;
    int off = 0;
    for (int f = 0; f < n_fields; ++f) {
        ft.offset[f] = off;
        ft.size[f] = sizes[f];
        off += sizes[f];
    }
    return SPB_OK;
}

// tokens int64 [n, ld_tok]; table fp32 [sum V_f, 128]; out bf16 [n, ld_out] (F*128 columns written)
extern "C" int spb_embed_ln_fwd(const int64_t* tokens, int ld_tok, const float* table, const int* field_sizes, int n_fields,
                                const float* w, const float* b, void* out, int ld_out, float* mean, float* rstd, int n_rows,
                                float eps, cudaStream_t stream) {
    if (n_rows <= 0) return SPB_OK;
    SPB_CHECK_ARG(tokens && table && w && b && out && mean && rstd, "spb_embed_ln_fwd: null pointer");
    FieldTable ft;
    int rc = fill_field_table(ft, field_sizes, n_fields);
    if (rc != SPB_OK) return rc;
    const int grid = row_grid(n_rows), thr = ROW_WARPS * 32;
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
    if (n_fields == 12) embed_ln_fwd_kernel<12><<<grid, thr, 0, stream>>>(tokens, ld_tok, table, ft, w, b, o, ld_out, mean, rstd, n_rows, eps);
    else if (n_fields == 10) embed_ln_fwd_kernel<10><<<grid, thr, 0, stream>>>(tokens, ld_tok, table, ft, w, b, o, ld_out, mean, rstd, n_rows, eps);
    else {
        spb_set_error("spb_embed_ln_fwd: compiled for 10 (score) or 12 (performance) fields, got %d", n_fields);
        return SPB_ERR_ARG;
    }
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}

// dtable / dw / db are ACCUMULATED into (caller zero-initialises); c1/c2 are fp32 [n] scratch.
extern "C" int spb_embed_ln_bwd(const void* dy, int ld_dy, const int64_t* tokens, int ld_tok, const float* table,
                                const int* field_sizes, int n_fields, const float* w, const float* mean, const float* rstd,
                                float* c1, float* c2, float* dtable, float* dw, float* db, int n_rows, cudaStream_t stream) {
    if (n_rows <= 0) return SPB_OK;
    SPB_CHECK_ARG(dy && tokens && table && w && mean && rstd && c1 && c2 && dtable && dw && db, "spb_embed_ln_bwd: null pointer");
    FieldTable ft;
    int rc = fill_field_table(ft, field_sizes, n_fields);
    if (rc != SPB_OK) return rc;
    const __nv_bfloat16* d = reinterpret_cast<const __nv_bfloat16*>(dy);
    int grid = row_grid(n_rows);
    if (grid > 2 * spb_num_sms()) grid = 2 * spb_num_sms();
    const int thr = ROW_WARPS * 32;
    if (n_fields == 12) embed_ln_bwd_stats_kernel<12><<<grid, thr, 0, stream>>>(d, ld_dy, tokens, ld_tok, table, ft, w, mean, rstd, c1, c2, dw, db, n_rows);
    else if (n_fields == 10) embed_ln_bwd_stats_kernel<10><<<grid, thr, 0, stream>>>(d, ld_dy, tokens, ld_tok, table, ft, w, mean, rstd, c1, c2, dw, db, n_rows);
    else {
        spb_set_error("spb_embed_ln_bwd: compiled for 10 or 12 fields, got %d", n_fields);
        return SPB_ERR_ARG;
    }
    SPB_CHECK_LAUNCH();
    return spb_embed_scatter_mma(d, ld_dy, tokens, ld_tok, table, ft, w, mean, rstd, c1, c2, dtable, n_rows, stream);
}
