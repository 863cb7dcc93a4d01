// One new position through the whole decoder stack in ONE persistent kernel (SURVEY.md section 8 row a13, north_star item 6).
//
// Reference semantics: the cache path of Transformer.forward (modules/transformer/transformer.py:161-186,219-221) for B scores
// that advance in lockstep -- per layer AdaLN -> q|k|v -> append k|v to the cache -> MQA attention of the new query over the
// cache with the ALiBi bias (attend.py:58-126, attention.py:139-197) -> out-projection + residual -> AdaLN -> GLU feed-forward
// + residual (feedforward.py:13-64), then the final AdaLN (layers.py:31-47).
//
// A note-step is ~2 GFLOP on [B <= 256, 256] activations against 7.6 MB of bf16 weights: as ~45 separate launches it is pure
// launch / dependency latency (8 us per kernel, 0.5 ms per note).  Here every SM takes a slice of every phase -- weights stream
// from L2 once per step over the whole chip, the KV cache is read once -- and the phases are separated by a grid barrier
// (one atomic counter; all CTAs are co-resident: grid <= #SMs, one CTA per SM):
//   phase 0        gb = style W_ada^T + b          (gamma-1 | beta) of all 2*depth+1 AdaLNs, bf16 scratch -- skipped when the caller
//                                                 prepared the terms of all positions with one GEMM (gb_all);
//                  with `front`: te = x1 Wf^T + p2  first half of the input front of the rendering loop, 32x16 tiles over K = 1536
//   per layer  ABC per score (two per CTA, warps 0-3 / 4-7), no barrier in between:
//                  [layer 0 with `front`: x = LN(te) Wc^T + c2 as a per-row product]
//                  qkv = AdaLN(x) Wqkv^T as a per-row product over the transposed weights (16-byte loads, k split over thread
//                  groups, fixed summation order); cache[pos] = k|v;
//                  o = softmax(q K^T s - slope|i-j|) V on tensor cores: mma.sync m16n8k16 with the 4 heads as rows 0-3, online
//                  softmax per warp over its quarter of the keys, K fragments straight from the cache rows (dims permuted so a
//                  thread owns 16 contiguous dims), V tiles through a cp.async ring + ldmatrix.trans;
//                  x += mask * (o Wo^T) as a per-row product
//              D   h    = GLU(AdaLN(x) W1^T + b1)     32x32 tiles, mma.sync m16n8k16 (M is tiny: tcgen05's 128-row tiles would idle
//                                                     3/4 of the tensor core); value and gate chains in the same warp
//              E   x   += h W2^T                       32x16 tiles over K = 1024, K split inside the CTA, fixed summation order
//   final          out  = AdaLN(x)  (+ a bf16 copy for the head projection)
// Tile phases issue all of their staging loads before the first shared-memory store.  Nothing in the kernel uses atomics on data:
// a rendering is bit-reproducible.
// Algorithmic HBM/L2 bytes per note-step: B * pos * 4 layers * 256 B of KV cache (the roofline term, SURVEY 8(d)) + 7.6 MB of
// weights out of L2.
#include <cmath>

#include "common.cuh"

namespace {

constexpr int DS_D = 256, DS_H = 4, DS_DH = 64, DS_HID = 1024, DS_QKV = DS_H * DS_DH + 2 * DS_DH;      // 384
constexpr int DS_MAX_DEPTH = 8;
constexpr int DS_THREADS = 256;
constexpr int DS_TM = 32, DS_TN = 32;            // CTA tile
constexpr int DS_LDA = DS_D + 8;                 // padded smem row (bf16 elements): conflict-free fragment loads
constexpr int DS_MAX_KEYS = 2048;

struct DecodeStackParams {
    int B, depth, S, cap;                        // scores, layers, style width, cache capacity (rows per score)
    const float* x_in;                           // [B, 256] stream input of the new position
    const float* style;                          // [B, S]
    const __nv_bfloat16* w_ada;                  // [(2*depth+1) * 512, S]
    const float* b_ada;                          // [(2*depth+1) * 512]  (gamma - 1 | beta)
    const __nv_bfloat16* wqkv[DS_MAX_DEPTH];     // [384, 256]
    const __nv_bfloat16* wo[DS_MAX_DEPTH];
    const __nv_bfloat16* wqkv_t[DS_MAX_DEPTH];   // [256, 384]: Wqkv transposed (input-major), for the per-row matrix-vector products
    const __nv_bfloat16* wo_t[DS_MAX_DEPTH];     // [256, 256]: Wo transposed       // [256, 256]
    const float* logslopes[DS_MAX_DEPTH];        // [4]
    const __nv_bfloat16* w1[DS_MAX_DEPTH];       // [2048, 256] value rows | gate rows
    const float* b1[DS_MAX_DEPTH];               // [2048]
    const __nv_bfloat16* w2[DS_MAX_DEPTH];       // [256, 1024]
    __nv_bfloat16* kv[DS_MAX_DEPTH];             // [B, cap, 128] k | v
    const uint8_t* key_mask;                     // [B, cap] or null
    const long long* pos_dev;                    // device scalar: index of the new position
    // scratch
    __nv_bfloat16* gb;                           // [B, (2*depth+1) * 512]
    __nv_bfloat16* qkv;                          // [B, 384]
    __nv_bfloat16* o;                            // [B, 256]
    __nv_bfloat16* hmid;                         // [B, 1024]
    float* xres;                                 // [B, 256] residual stream
    float* hid_out;                              // [depth, B, 256] inputs of the attention layers (cache contract), or null
    float* out;                                  // [B, 256]
    __nv_bfloat16* out16;                        // optional bf16 copy of `out` (operand of the head projection), or null
    unsigned* barrier;                           // zeroed by the host before the launch
    float eps;
    const __nv_bfloat16* gb_all;                 // optional [B, T_all, (2*depth+1)*512]: the AdaLN terms of every position, prepared ahead
    int T_all;
    // optional input front of the rendering loop (decode.py): x = LN(x1 Wf^T + p2) Wc^T + c2 replaces x_in
    const __nv_bfloat16* f_x1;                   // [B, 1536] tuple embedding of the previous note (bf16), or null: no front
    const __nv_bfloat16* f_w;                    // [256, 1536] composed projection (project_multiemb left half . project_emb)
    const float* f_p2;                           // [B, 256] prepared term of the masked tuple (+ biases)
    float* f_te;                                 // [B, 256] scratch
    const float* f_lnw;                          // emb_norm weight / bias [256]
    const float* f_lnb;
    const __nv_bfloat16* f_wct;                  // [256, 256] left half of the decoder's project_emb, transposed (input-major)
    const float* f_c2;                           // [B, 256] prepared context term (+ bias)
};
constexpr int DS_FK = 1536, DS_FKQ = DS_FK / 4, DS_FLDA = DS_FKQ + 8;      // front GEMM: K, K per warp-pair quarter, padded smem row

__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned& epoch) {
    __syncthreads();
    if (threadIdx.x == 0) {
        ++epoch;
        __threadfence();
        atomicAdd(counter, 1u);
        const unsigned target = epoch * gridDim.x;
        unsigned seen;
        long long t0 = clock64();
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counter) : "memory");
            if (seen < target && clock64() - t0 > 4000000000ll) {
                printf("spb200: decode_stack grid barrier timed out (block %d, epoch %u, seen %u)\n", blockIdx.x, epoch, seen);
                __trap();
            }
        } while (seen < target);
        __threadfence();
    }
    __syncthreads();
}

__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void cp_async16_zfill(uint32_t dst_smem, const void* src, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void ldsm_x4_trans(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}

// acc[4] of this warp's m16n8 piece of a 32 x 32 CTA tile: rows r0 + 16*(warp&1).., columns of W  n0 + 8*(warp>>1)..
// A: smem bf16 [32][lda] (k contiguous);  W: global bf16 [N][ldw] (k contiguous), rows n_row0.. are this tile's columns
__device__ __forceinline__ void tile_mma(float (&acc)[4], const __nv_bfloat16* sA, int lda, const __nv_bfloat16* __restrict__ W, int ldw,
                                         int n_row0, int K, int warp, int lane) {
    const int g = lane >> 2, tig = lane & 3;
    const __nv_bfloat16* a_lo = sA + (size_t)((warp & 1) * 16 + g) * lda + tig * 2;
    const __nv_bfloat16* a_hi = a_lo + 8 * lda;
    const __nv_bfloat16* wr = W + (size_t)(n_row0 + (warp >> 1) * 8 + g) * ldw + tig * 2;
#pragma unroll 4
    for (int k = 0; k < K; k += 16) {
        const uint32_t a0 = *reinterpret_cast<const uint32_t*>(a_lo + k), a1 = *reinterpret_cast<const uint32_t*>(a_hi + k);
        const uint32_t a2 = *reinterpret_cast<const uint32_t*>(a_lo + k + 8), a3 = *reinterpret_cast<const uint32_t*>(a_hi + k + 8);
        const uint32_t b0 = __ldg(reinterpret_cast<const uint32_t*>(wr + k)), b1 = __ldg(reinterpret_cast<const uint32_t*>(wr + k + 8));
        mma_bf16_16816(acc, a0, a1, a2, a3, b0, b1);
    }
}

// The same product with the weight fragments fetched up front: a tile's 2 * KSTEPS 32-bit loads leave together BEFORE the
// activation tile is staged, so one L2 round trip (not KSTEPS / 4 of them) sits on the tile's critical path.
template <int KSTEPS>
__device__ __forceinline__ void load_w(uint32_t (&bf)[2 * KSTEPS], const __nv_bfloat16* __restrict__ W, int ldw, int n_row, int lane) {
    const __nv_bfloat16* wr = W + (size_t)(n_row + (lane >> 2)) * ldw + (lane & 3) * 2;
#pragma unroll
    for (int k = 0; k < KSTEPS; ++k) {
        bf[2 * k] = __ldg(reinterpret_cast<const uint32_t*>(wr + 16 * k));
        bf[2 * k + 1] = __ldg(reinterpret_cast<const uint32_t*>(wr + 16 * k + 8));
    }
}
template <int KSTEPS>
__device__ __forceinline__ void mma_pre(float (&acc)[4], const __nv_bfloat16* sA, int lda, const uint32_t (&bf)[2 * KSTEPS], int warp, int lane) {
    const int g = lane >> 2, tig = lane & 3;
    const __nv_bfloat16* a_lo = sA + (size_t)((warp & 1) * 16 + g) * lda + tig * 2;
    const __nv_bfloat16* a_hi = a_lo + 8 * lda;
#pragma unroll
    for (int k = 0; k < KSTEPS; ++k) {
        const uint32_t a0 = *reinterpret_cast<const uint32_t*>(a_lo + 16 * k), a1 = *reinterpret_cast<const uint32_t*>(a_hi + 16 * k);
        const uint32_t a2 = *reinterpret_cast<const uint32_t*>(a_lo + 16 * k + 8), a3 = *reinterpret_cast<const uint32_t*>(a_hi + 16 * k + 8);
        mma_bf16_16816(acc, a0, a1, a2, a3, bf[2 * k], bf[2 * k + 1]);
    }
}

// AdaLN of 32 rows of the fp32 residual stream -> bf16 smem tile [32][DS_LDA]; one warp per 4 rows (rows beyond B are zeroed).
// The loads of all four rows (residual and gamma / beta) are issued before the first reduction.
__device__ __forceinline__ void stage_adaln(__nv_bfloat16* sA, const float* xres, const __nv_bfloat16* gb, size_t ld_gb, int norm_idx, int row0,
                                            int B, float eps, int warp, int lane) {
    constexpr int RPW = DS_TM / (DS_THREADS / 32);          // 4 rows per warp
    float4 x0[RPW], x1[RPW];
    uint4 gu[RPW], bu[RPW];
#pragma unroll
    for (int i = 0; i < RPW; ++i) {
        const int row = row0 + warp + i * (DS_THREADS / 32);
        const bool ok = row < B;
        const float* xr = xres + (size_t)(ok ? row : 0) * DS_D + lane * 8;
        const __nv_bfloat16* gr = gb + (size_t)(ok ? row : 0) * ld_gb + norm_idx * 2 * DS_D + lane * 8;
        x0[i] = *reinterpret_cast<const float4*>(xr);
        x1[i] = *reinterpret_cast<const float4*>(xr + 4);
        gu[i] = *reinterpret_cast<const uint4*>(gr);
        bu[i] = *reinterpret_cast<const uint4*>(gr + DS_D);
    }
#pragma unroll
    for (int i = 0; i < RPW; ++i) {
        const int rr = warp + i * (DS_THREADS / 32);
        __nv_bfloat16* dst = sA + (size_t)rr * DS_LDA + lane * 8;
        if (row0 + rr >= B) {
            *reinterpret_cast<uint4*>(dst) = make_uint4(0u, 0u, 0u, 0u);
            continue;
        }
        float v[8] = {x0[i].x, x0[i].y, x0[i].z, x0[i].w, x1[i].x, x1[i].y, x1[i].z, x1[i].w};
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) s += v[j];
        const float mean = warp_sum(s) * (1.f / DS_D);
        float q = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) { v[j] -= mean; q += v[j] * v[j]; }
        const float rstd = rsqrtf(warp_sum(q) * (1.f / DS_D) + eps);
        const float2 g0 = unpack_bf16x2(gu[i].x), g1 = unpack_bf16x2(gu[i].y), g2 = unpack_bf16x2(gu[i].z), g3 = unpack_bf16x2(gu[i].w);
        const float2 b0 = unpack_bf16x2(bu[i].x), b1 = unpack_bf16x2(bu[i].y), b2 = unpack_bf16x2(bu[i].z), b3 = unpack_bf16x2(bu[i].w);
        const float gm[8] = {g0.x, g0.y, g1.x, g1.y, g2.x, g2.y, g3.x, g3.y}, bt[8] = {b0.x, b0.y, b1.x, b1.y, b2.x, b2.y, b3.x, b3.y};
        float y[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = v[j] * rstd * (1.f + gm[j]) + bt[j];        // gb holds gamma - 1 (rowops.cu)
        *reinterpret_cast<uint4*>(dst) = make_uint4(pack_bf16x2(y[0], y[1]), pack_bf16x2(y[2], y[3]), pack_bf16x2(y[4], y[5]), pack_bf16x2(y[6], y[7]));
    }
}

// The four K quarters (KQ columns each, KQ = PT * 64) of 32 rows of a bf16 [B, ld] matrix -> four smem tiles [32][lda], with ALL of a
// thread's 16-byte loads issued before the first store: a loop of load -> store pairs walks the L2 latency once per iteration.
template <int PT>
__device__ __forceinline__ void stage_quarters(__nv_bfloat16* sA, int lda, const __nv_bfloat16* src, int ld, int row0, int B) {
    constexpr int KQ = PT * 64, PER_ROW = KQ / 8;
    uint4 v[4][PT];
#pragma unroll
    for (int q4 = 0; q4 < 4; ++q4)
#pragma unroll
        for (int j = 0; j < PT; ++j) {
            const int i = threadIdx.x + j * DS_THREADS;
            const int rr = i / PER_ROW, c = (i - rr * PER_ROW) * 8;
            const int row = row0 + rr;
            v[q4][j] = row < B ? __ldg(reinterpret_cast<const uint4*>(src + (size_t)row * ld + q4 * KQ + c)) : make_uint4(0u, 0u, 0u, 0u);
        }
#pragma unroll
    for (int q4 = 0; q4 < 4; ++q4)
#pragma unroll
        for (int j = 0; j < PT; ++j) {
            const int i = threadIdx.x + j * DS_THREADS;
            const int rr = i / PER_ROW, c = (i - rr * PER_ROW) * 8;
            *reinterpret_cast<uint4*>(sA + (size_t)q4 * DS_TM * lda + (size_t)rr * lda + c) = v[q4][j];
        }
}

__global__ void __launch_bounds__(DS_THREADS, 1)
decode_stack_kernel(DecodeStackParams p) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    __nv_bfloat16* sA = reinterpret_cast<__nv_bfloat16*>(smem_raw);                          // [32][DS_LDA]
    float* sP = reinterpret_cast<float*>(smem_raw + DS_TM * DS_LDA * 2);                      // [8 warps][cap] attention scores
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, tig = lane & 3;
    const int B = p.B, n_norms = 2 * p.depth + 1, ld_gb = n_norms * 2 * DS_D;
    const int row_blocks = (B + DS_TM - 1) / DS_TM;
    const int pos = (int)*p.pos_dev;
    unsigned epoch = 0;
    // the AdaLN terms of this step: computed here (phase 0) from the style rows, or -- when the caller prepared them for all positions
    // in one large GEMM -- read in place at position pos + 1 (the style a note-step uses is that of the note it predicts)
    const __nv_bfloat16* gbp = p.gb;
    size_t gb_stride = (size_t)ld_gb;
    if (p.gb_all != nullptr) {
        const int t_style = min(pos + 1, p.T_all - 1);
        gbp = p.gb_all + (size_t)t_style * ld_gb;
        gb_stride = (size_t)p.T_all * ld_gb;
    }

    // ---- phase 0: gb = style W_ada^T + b_ada for every norm; the residual stream starts as the input
    {
        const int col_blocks = ld_gb / DS_TN;
        for (int t = blockIdx.x; t < row_blocks * col_blocks && p.gb_all == nullptr; t += gridDim.x) {
            const int rb = t / col_blocks, cb = t - rb * col_blocks;
            __syncthreads();
            for (int i = threadIdx.x; i < DS_TM * p.S; i += DS_THREADS) {        // style rows -> bf16 tile (S <= 256)
                const int rr = i / p.S, c = i - rr * p.S;
                const int row = rb * DS_TM + rr;
                sA[(size_t)rr * DS_LDA + c] = __float2bfloat16_rn(row < B ? p.style[(size_t)row * p.S + c] : 0.f);
            }
            __syncthreads();
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            tile_mma(acc, sA, DS_LDA, p.w_ada, p.S, cb * DS_TN, p.S, warp, lane);
            const int col = cb * DS_TN + (warp >> 1) * 8 + tig * 2;
            const float bb0 = p.b_ada[col], bb1 = p.b_ada[col + 1];
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
                const int row = rb * DS_TM + (warp & 1) * 16 + g + hf * 8;
                if (row < B)
                    *reinterpret_cast<uint32_t*>(p.gb + (size_t)row * ld_gb + col) = pack_bf16x2(acc[2 * hf] + bb0, acc[2 * hf + 1] + bb1);
            }
        }
        if (p.f_x1 == nullptr) {
            for (int i = blockIdx.x * DS_THREADS + threadIdx.x; i < B * DS_D / 4; i += gridDim.x * DS_THREADS)
                reinterpret_cast<float4*>(p.xres)[i] = reinterpret_cast<const float4*>(p.x_in)[i];
        } else {
            // front, first half: te = x1 Wf^T + p2.  32 x 16 tiles over the whole K = 1536: the four warp pairs take a quarter of K
            // each and the quarters are summed through shared memory in a fixed order (same scheme as phase E)
            constexpr int TN_F = 16;
            const int col_blocks = DS_D / TN_F;
            const int mh = warp & 1, kq = warp >> 1;
            __nv_bfloat16* sAk = sA + (size_t)kq * DS_TM * DS_FLDA;
            float* red = reinterpret_cast<float*>(smem_raw + 4 * DS_TM * DS_FLDA * 2);
            for (int t = blockIdx.x; t < row_blocks * col_blocks; t += gridDim.x) {
                const int rb = t / col_blocks, cb = t - rb * col_blocks;
                uint32_t bf0[2 * (DS_FKQ / 16)], bf1[2 * (DS_FKQ / 16)];
                load_w<DS_FKQ / 16>(bf0, p.f_w + kq * DS_FKQ, DS_FK, cb * TN_F, lane);
                load_w<DS_FKQ / 16>(bf1, p.f_w + kq * DS_FKQ, DS_FK, cb * TN_F + 8, lane);
                __syncthreads();
                stage_quarters<DS_FKQ / 64>(sA, DS_FLDA, p.f_x1, DS_FK, rb * DS_TM, B);
                __syncthreads();
                float acc0[4] = {0.f, 0.f, 0.f, 0.f}, acc1[4] = {0.f, 0.f, 0.f, 0.f};
                mma_pre<DS_FKQ / 16>(acc0, sAk, DS_FLDA, bf0, warp, lane);
                mma_pre<DS_FKQ / 16>(acc1, sAk, DS_FLDA, bf1, warp, lane);
                float4* my = reinterpret_cast<float4*>(red) + ((kq * 2 + mh) * 2) * 32 + lane;
                my[0] = make_float4(acc0[0], acc0[1], acc0[2], acc0[3]);
                my[32] = make_float4(acc1[0], acc1[1], acc1[2], acc1[3]);
                __syncthreads();
                if (kq == 0) {
#pragma unroll
                    for (int piece = 0; piece < 2; ++piece) {
                        float4 sum = reinterpret_cast<const float4*>(red)[((0 * 2 + mh) * 2 + piece) * 32 + lane];
#pragma unroll
                        for (int q4 = 1; q4 < 4; ++q4) {
                            const float4 v = reinterpret_cast<const float4*>(red)[((q4 * 2 + mh) * 2 + piece) * 32 + lane];
                            sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
                        }
                        const int col = cb * TN_F + piece * 8 + tig * 2;
                        const float part[4] = {sum.x, sum.y, sum.z, sum.w};
#pragma unroll
                        for (int hf = 0; hf < 2; ++hf) {
                            const int row = rb * DS_TM + mh * 16 + g + hf * 8;
                            if (row < B) {
                                const float2 r2 = *reinterpret_cast<const float2*>(p.f_p2 + (size_t)row * DS_D + col);
                                *reinterpret_cast<float2*>(p.f_te + (size_t)row * DS_D + col) = make_float2(part[2 * hf] + r2.x, part[2 * hf + 1] + r2.y);
                            }
                        }
                    }
                }
            }
        }
    }
    grid_barrier(p.barrier, epoch);

    for (int l = 0; l < p.depth; ++l) {
        // ---- A + B + C for two scores per CTA at a time (warps 0-3 / 4-7), no grid barrier in between: everything here is local to
        // a score's row.  A: AdaLN of the residual row and qkv = xn Wqkv^T as a matrix-vector product per row (thread = two output
        // columns, transposed weights streamed from L2, coalesced); B: append k|v, attention of the new query over the cache;
        // C: x += mask * (o Wo^T), again per row.  (A 32-row tensor-core tile would share the weights between rows, but costs two
        // more grid barriers and two more latency-bound tile phases per layer: 5 -> 3 phases.)  MQA: the
        // four heads share K and V, so the four warps of a score split the KEYS and each evaluates all four heads on its quarter
        // -- every cache row is fetched once, and a warp walks a quarter of the sequential load -> use -> load chain.
        {
            const int n_keys = min(p.cap, pos + 1);
            const float scale = rsqrtf((float)DS_DH);
            // (the first 8 * cap floats of sP held the scores of the scalar attention; the tensor-core path keeps them in registers)
            float* sRed = sP + (size_t)(DS_THREADS / 32) * p.cap;             // [2][4 warps][4 heads] maxima, then [2][4][4] sums
            float* sO = sRed + 64;                                            // [2][4 warps][4 heads][64] partial outputs
            float* sXn = sO + 2 * 4 * 4 * 64;                                 // [2][256] AdaLN'd rows (bf16-rounded)
            float* sOrow = sXn + 2 * DS_D;                                    // [2][256] attention outputs (bf16-rounded)
            uint32_t* sQKV = reinterpret_cast<uint32_t*>(sOrow + 2 * DS_D);   // [2][192] qkv rows, bf16 pairs
            float* sPart = reinterpret_cast<float*>(sQKV + 2 * (DS_QKV / 2));   // [8][2][256] (or [5][2][384]) k-split partial sums
            constexpr int VST_ROW = 144, VST_STAGE = 16 * VST_ROW;            // V tile of 16 keys x 64 dims, rows padded to 144 B
            const uint32_t vst = smem_u32(sPart + 8 * 2 * DS_D) + (uint32_t)(warp * 3 * VST_STAGE);     // three stages per warp
            const int bl = warp >> 2, wq = warp & 3;
            const int per_warp = ((n_keys + 3) / 4 + 15) & ~15;               // keys per warp, a multiple of 16 (one PV k-step)
            const int k_lo = wq * per_warp, k_hi = min(n_keys, k_lo + per_warp);
            for (int pair = blockIdx.x; pair * 2 < B; pair += gridDim.x) {
                const int b = pair * 2 + bl;
                const bool live = b < B;
                __syncthreads();                                      // the previous pair's rows in shared memory are done with
                if (l == 0 && p.f_x1 != nullptr) {
                    // front, second half: x = LN(te) Wc^T + c2 for the two rows of this pair (per-row product like the out-projection)
                    if (wq == 0) {
                        float y[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                        if (live) {
                            const float4 v0 = *reinterpret_cast<const float4*>(p.f_te + (size_t)b * DS_D + lane * 8);
                            const float4 v1 = *reinterpret_cast<const float4*>(p.f_te + (size_t)b * DS_D + lane * 8 + 4);
                            float v[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
                            float s_ = 0.f;
#pragma unroll
                            for (int j = 0; j < 8; ++j) s_ += v[j];
                            const float mean = warp_sum(s_) * (1.f / DS_D);
                            float q_ = 0.f;
#pragma unroll
                            for (int j = 0; j < 8; ++j) { v[j] -= mean; q_ += v[j] * v[j]; }
                            const float rstd = rsqrtf(warp_sum(q_) * (1.f / DS_D) + p.eps);
#pragma unroll
                            for (int j = 0; j < 8; ++j)
                                y[j] = __bfloat162float(__float2bfloat16_rn(v[j] * rstd * p.f_lnw[lane * 8 + j] + p.f_lnb[lane * 8 + j]));
                        }
                        float* xo = sOrow + bl * DS_D + lane * 8;
                        *reinterpret_cast<float4*>(xo) = make_float4(y[0], y[1], y[2], y[3]);
                        *reinterpret_cast<float4*>(xo + 4) = make_float4(y[4], y[5], y[6], y[7]);
                    }
                    __syncthreads();
                    {
                        const int kg = threadIdx.x >> 5, cg = threadIdx.x & 31;
                        const __nv_bfloat16* wt = p.f_wct + cg * 8;
                        float a0[8], a1[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) { a0[j] = 0.f; a1[j] = 0.f; }
#pragma unroll 16
                        for (int k = kg * 32; k < kg * 32 + 32; ++k) {
                            const uint4 w = __ldg(reinterpret_cast<const uint4*>(wt + (size_t)k * DS_D));
                            const float2 w0 = unpack_bf16x2(w.x), w1 = unpack_bf16x2(w.y), w2 = unpack_bf16x2(w.z), w3 = unpack_bf16x2(w.w);
                            const float wv[8] = {w0.x, w0.y, w1.x, w1.y, w2.x, w2.y, w3.x, w3.y};
                            const float x0 = sOrow[k], x1 = sOrow[DS_D + k];
#pragma unroll
                            for (int j = 0; j < 8; ++j) { a0[j] = fmaf(x0, wv[j], a0[j]); a1[j] = fmaf(x1, wv[j], a1[j]); }
                        }
                        float* pp = sPart + (size_t)kg * 2 * DS_D + cg * 8;
                        *reinterpret_cast<float4*>(pp) = make_float4(a0[0], a0[1], a0[2], a0[3]);
                        *reinterpret_cast<float4*>(pp + 4) = make_float4(a0[4], a0[5], a0[6], a0[7]);
                        *reinterpret_cast<float4*>(pp + DS_D) = make_float4(a1[0], a1[1], a1[2], a1[3]);
                        *reinterpret_cast<float4*>(pp + DS_D + 4) = make_float4(a1[4], a1[5], a1[6], a1[7]);
                        __syncthreads();
                        const int c = threadIdx.x;
#pragma unroll
                        for (int r = 0; r < 2; ++r) {
                            const int row = pair * 2 + r;
                            if (row < B) {
                                float sum = p.f_c2[(size_t)row * DS_D + c];
#pragma unroll
                                for (int k8 = 0; k8 < 8; ++k8) sum += sPart[(size_t)(k8 * 2 + r) * DS_D + c];
                                p.xres[(size_t)row * DS_D + c] = sum;
                            }
                        }
                    }
                    __syncthreads();
                }
                if (wq == 0) {                                        // warps 0 and 4: AdaLN of one residual row each
                    float* xn = sXn + bl * DS_D + lane * 8;
                    float y[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                    if (live) {
                        const float4 v0 = *reinterpret_cast<const float4*>(p.xres + (size_t)b * DS_D + lane * 8);
                        const float4 v1 = *reinterpret_cast<const float4*>(p.xres + (size_t)b * DS_D + lane * 8 + 4);
                        if (p.hid_out != nullptr) {                   // the cache contract's copy of the layer input
                            float* ho = p.hid_out + ((size_t)l * B + b) * DS_D + lane * 8;
                            *reinterpret_cast<float4*>(ho) = v0;
                            *reinterpret_cast<float4*>(ho + 4) = v1;
                        }
                        float v[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
                        float s_ = 0.f;
#pragma unroll
                        for (int j = 0; j < 8; ++j) s_ += v[j];
                        const float mean = warp_sum(s_) * (1.f / DS_D);
                        float q_ = 0.f;
#pragma unroll
                        for (int j = 0; j < 8; ++j) { v[j] -= mean; q_ += v[j] * v[j]; }
                        const float rstd = rsqrtf(warp_sum(q_) * (1.f / DS_D) + p.eps);
                        const __nv_bfloat16* gr = gbp + (size_t)b * gb_stride + (2 * l) * 2 * DS_D + lane * 8;
                        const uint4 gu = *reinterpret_cast<const uint4*>(gr), bu = *reinterpret_cast<const uint4*>(gr + DS_D);
                        const float2 g0 = unpack_bf16x2(gu.x), g1 = unpack_bf16x2(gu.y), g2 = unpack_bf16x2(gu.z), g3 = unpack_bf16x2(gu.w);
                        const float2 b0 = unpack_bf16x2(bu.x), b1 = unpack_bf16x2(bu.y), b2 = unpack_bf16x2(bu.z), b3 = unpack_bf16x2(bu.w);
                        const float gm[8] = {g0.x, g0.y, g1.x, g1.y, g2.x, g2.y, g3.x, g3.y}, bt[8] = {b0.x, b0.y, b1.x, b1.y, b2.x, b2.y, b3.x, b3.y};
#pragma unroll
                        for (int j = 0; j < 8; ++j) y[j] = __bfloat162float(__float2bfloat16_rn(v[j] * rstd * (1.f + gm[j]) + bt[j]));
                    }
                    *reinterpret_cast<float4*>(xn) = make_float4(y[0], y[1], y[2], y[3]);
                    *reinterpret_cast<float4*>(xn + 4) = make_float4(y[4], y[5], y[6], y[7]);
                }
                __syncthreads();
                // qkv of both rows: thread = 8 adjacent output columns x one fifth of k (16-byte weight loads, all of a thread's
                // loads in flight together); the five partial sums meet in shared memory and are added in a fixed order
                if (threadIdx.x < 5 * (DS_QKV / 8)) {
                    const int kg = threadIdx.x / (DS_QKV / 8), cg = threadIdx.x - kg * (DS_QKV / 8);
                    const int k_lo2 = kg * 52, k_hi2 = min(DS_D, k_lo2 + 52);
                    const __nv_bfloat16* wt = p.wqkv_t[l] + cg * 8;
                    float a0[8], a1[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) { a0[j] = 0.f; a1[j] = 0.f; }
#pragma unroll 13
                    for (int k = k_lo2; k < k_hi2; ++k) {
                        const uint4 w = __ldg(reinterpret_cast<const uint4*>(wt + (size_t)k * DS_QKV));
                        const float2 w0 = unpack_bf16x2(w.x), w1 = unpack_bf16x2(w.y), w2 = unpack_bf16x2(w.z), w3 = unpack_bf16x2(w.w);
                        const float wv[8] = {w0.x, w0.y, w1.x, w1.y, w2.x, w2.y, w3.x, w3.y};
                        const float x0 = sXn[k], x1 = sXn[DS_D + k];
#pragma unroll
                        for (int j = 0; j < 8; ++j) { a0[j] = fmaf(x0, wv[j], a0[j]); a1[j] = fmaf(x1, wv[j], a1[j]); }
                    }
                    float* pp = sPart + (size_t)kg * 2 * DS_QKV + cg * 8;
                    *reinterpret_cast<float4*>(pp) = make_float4(a0[0], a0[1], a0[2], a0[3]);
                    *reinterpret_cast<float4*>(pp + 4) = make_float4(a0[4], a0[5], a0[6], a0[7]);
                    *reinterpret_cast<float4*>(pp + DS_QKV) = make_float4(a1[0], a1[1], a1[2], a1[3]);
                    *reinterpret_cast<float4*>(pp + DS_QKV + 4) = make_float4(a1[4], a1[5], a1[6], a1[7]);
                }
                __syncthreads();
                if (threadIdx.x < DS_QKV / 2) {
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        float s0 = 0.f, s1 = 0.f;
#pragma unroll
                        for (int kg = 0; kg < 5; ++kg) {
                            const float2 v = *reinterpret_cast<const float2*>(sPart + (size_t)(kg * 2 + r) * DS_QKV + threadIdx.x * 2);
                            s0 += v.x; s1 += v.y;
                        }
                        sQKV[r * (DS_QKV / 2) + threadIdx.x] = pack_bf16x2(s0, s1);
                    }
                }
                __syncthreads();
                const __nv_bfloat16* qrow = reinterpret_cast<const __nv_bfloat16*>(sQKV + bl * (DS_QKV / 2));
                if (live) {
                    __nv_bfloat16* kvw = p.kv[l] + (size_t)b * p.cap * 128;
                    const int lw = threadIdx.x & 127;
                    if (lw < 16 && pos < p.cap)
                        reinterpret_cast<uint4*>(kvw + (size_t)pos * 128)[lw] = reinterpret_cast<const uint4*>(qrow + DS_H * DS_DH)[lw];
                }
                __syncthreads();
                const __nv_bfloat16* kvb = p.kv[l] + (size_t)(live ? b : 0) * p.cap * 128;
                // ---- attention on tensor cores (mma.sync m16n8k16, fp32 accumulate), online softmax per warp over its quarter of the
                // keys.  S = q K^T: the 4 heads are rows 0-3 of the A tile (rows 4-15 zero); the 64 dims are permuted so that thread
                // (g, tig) owns dims [16 tig, 16 tig + 16) of key row g -- its B fragments of all four k-steps are two 16-byte loads
                // straight from the cache row, whole 128-byte lines per key.  O = P V: P is the S accumulator fragment re-packed as A,
                // V tiles of 16 keys are staged by cp.async (three stages per warp) and read with ldmatrix.trans.
                uint32_t qa0[4], qa2[4];
#pragma unroll
                for (int s_ = 0; s_ < 4; ++s_) {
                    const bool has = live && g < 4;
                    qa0[s_] = has ? *reinterpret_cast<const uint32_t*>(qrow + g * DS_DH + tig * 16 + 4 * s_) : 0u;
                    qa2[s_] = has ? *reinterpret_cast<const uint32_t*>(qrow + g * DS_DH + tig * 16 + 4 * s_ + 2) : 0u;
                }
                const float slope_h = g < 4 ? __expf(p.logslopes[l][g]) : 0.f;
                const int nblk = live ? (max(0, k_hi - k_lo) + 15) / 16 : 0;
                auto issue_v = [&](int blk, int st) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int c = lane + 32 * i, row = c >> 3, col = c & 7;
                        const int j = k_lo + blk * 16 + row;
                        const bool ok = j < k_hi;
                        cp_async16_zfill(vst + (uint32_t)(st * VST_STAGE + row * VST_ROW + col * 16),
                                         kvb + (size_t)(ok ? j : 0) * 128 + DS_DH + col * 8, ok ? 16 : 0);
                    }
                    cp_async_commit();
                };
                auto load_k = [&](int blk, uint4 (&kr)[4]) {
#pragma unroll
                    for (int tile = 0; tile < 2; ++tile) {
                        const int j = k_lo + blk * 16 + tile * 8 + g;
                        const bool ok = j < k_hi;
                        const uint4* src = reinterpret_cast<const uint4*>(kvb + (size_t)(ok ? j : 0) * 128 + tig * 16);
                        kr[2 * tile] = ok ? __ldg(src) : make_uint4(0u, 0u, 0u, 0u);
                        kr[2 * tile + 1] = ok ? __ldg(src + 1) : make_uint4(0u, 0u, 0u, 0u);
                    }
                };
                float m_run = -INFINITY, l_run = 0.f;
                float oacc[8][4];
#pragma unroll
                for (int n = 0; n < 8; ++n) { oacc[n][0] = 0.f; oacc[n][1] = 0.f; oacc[n][2] = 0.f; oacc[n][3] = 0.f; }
                // two blocks of 16 keys are in flight behind the one being evaluated (K in registers, V in the shared-memory ring)
                uint4 kr[4], kn[4], kn2[4];
                if (nblk > 0) {
                    issue_v(0, 0);
                    load_k(0, kn);
                }
                if (nblk > 1) {
                    issue_v(1, 1);
                    load_k(1, kn2);
                }
                for (int blk = 0; blk < nblk; ++blk) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) { kr[i] = kn[i]; kn[i] = kn2[i]; }
                    if (blk + 2 < nblk) {
                        issue_v(blk + 2, (blk + 2) % 3);
                        load_k(blk + 2, kn2);
                        cp_async_wait<2>();
                    } else if (blk + 1 < nblk) {
                        cp_async_wait<1>();
                    } else {
                        cp_async_wait<0>();
                    }
                    __syncwarp();
                    float s0[4] = {0.f, 0.f, 0.f, 0.f}, s1[4] = {0.f, 0.f, 0.f, 0.f};
                    mma_bf16_16816(s0, qa0[0], 0u, qa2[0], 0u, kr[0].x, kr[0].y);
                    mma_bf16_16816(s0, qa0[1], 0u, qa2[1], 0u, kr[0].z, kr[0].w);
                    mma_bf16_16816(s0, qa0[2], 0u, qa2[2], 0u, kr[1].x, kr[1].y);
                    mma_bf16_16816(s0, qa0[3], 0u, qa2[3], 0u, kr[1].z, kr[1].w);
                    mma_bf16_16816(s1, qa0[0], 0u, qa2[0], 0u, kr[2].x, kr[2].y);
                    mma_bf16_16816(s1, qa0[1], 0u, qa2[1], 0u, kr[2].z, kr[2].w);
                    mma_bf16_16816(s1, qa0[2], 0u, qa2[2], 0u, kr[3].x, kr[3].y);
                    mma_bf16_16816(s1, qa0[3], 0u, qa2[3], 0u, kr[3].z, kr[3].w);
                    // this lane (g < 4): head g, keys jb + 2 tig + {0,1} (tile 0) and jb + 8 + 2 tig + {0,1} (tile 1)
                    const int jb = k_lo + blk * 16;
                    float pv[4] = {s0[0], s0[1], s1[0], s1[1]};
                    float mblk = -INFINITY;
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        const int j = jb + (t >> 1) * 8 + tig * 2 + (t & 1);
                        const bool ok = g < 4 && j < k_hi && (p.key_mask == nullptr || p.key_mask[(size_t)b * p.cap + j]);
                        pv[t] = ok ? pv[t] * scale - slope_h * (float)(pos - j) : -INFINITY;
                        mblk = fmaxf(mblk, pv[t]);
                    }
                    mblk = fmaxf(mblk, __shfl_xor_sync(0xffffffffu, mblk, 1));
                    mblk = fmaxf(mblk, __shfl_xor_sync(0xffffffffu, mblk, 2));
                    const float m_new = fmaxf(m_run, mblk);
                    const float m_use = m_new == -INFINITY ? 0.f : m_new;
                    const float alpha = m_run == -INFINITY ? 0.f : __expf(m_run - m_use);
                    float psum = 0.f;
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        pv[t] = pv[t] == -INFINITY ? 0.f : __expf(pv[t] - m_use);
                        psum += pv[t];
                    }
                    l_run = l_run * alpha + psum;
                    m_run = m_new;
#pragma unroll
                    for (int n = 0; n < 8; ++n) { oacc[n][0] *= alpha; oacc[n][1] *= alpha; }
                    const uint32_t pa0 = pack_bf16x2(pv[0], pv[1]), pa2 = pack_bf16x2(pv[2], pv[3]);
                    const uint32_t stage = vst + (uint32_t)((blk % 3) * VST_STAGE);
                    // ldmatrix.x4.trans: matrices (keys 0-7 | 8-15) x (dim block 2 np | 2 np + 1); lane L supplies row L & 7 of matrix L >> 3
                    const uint32_t lrow = stage + (uint32_t)((((lane >> 3) & 1) * 8 + (lane & 7)) * VST_ROW + (lane >> 4) * 16);
#pragma unroll
                    for (int np = 0; np < 4; ++np) {
                        uint32_t r0, r1, r2, r3;
                        ldsm_x4_trans(lrow + (uint32_t)(np * 32), r0, r1, r2, r3);
                        mma_bf16_16816(oacc[2 * np], pa0, 0u, pa2, 0u, r0, r1);
                        mma_bf16_16816(oacc[2 * np + 1], pa0, 0u, pa2, 0u, r2, r3);
                    }
                }
                // the four lanes of a head hold partial sums of its keys; the four warps of the score meet through shared memory
                l_run += __shfl_xor_sync(0xffffffffu, l_run, 1);
                l_run += __shfl_xor_sync(0xffffffffu, l_run, 2);
                if (g < 4 && tig == 0) sRed[(bl * 4 + wq) * 4 + g] = m_run;
                __syncthreads();
                {
                    float fac = 0.f;
                    if (g < 4) {
                        const float mg = fmaxf(fmaxf(sRed[(bl * 4 + 0) * 4 + g], sRed[(bl * 4 + 1) * 4 + g]),
                                               fmaxf(sRed[(bl * 4 + 2) * 4 + g], sRed[(bl * 4 + 3) * 4 + g]));
                        fac = m_run == -INFINITY ? 0.f : __expf(m_run - mg);
                        if (tig == 0) sRed[32 + (bl * 4 + wq) * 4 + g] = l_run * fac;
#pragma unroll
                        for (int n = 0; n < 8; ++n)
                            *reinterpret_cast<float2*>(sO + ((size_t)(bl * 4 + wq) * 4 + g) * 64 + n * 8 + tig * 2) =
                                make_float2(oacc[n][0] * fac, oacc[n][1] * fac);
                    }
                }
                __syncthreads();
                if (live) {
                    // warp wq finishes head wq: 64 dims, two per lane
                    const int h = wq;
                    const float tot = sRed[32 + (bl * 4 + 0) * 4 + h] + sRed[32 + (bl * 4 + 1) * 4 + h] + sRed[32 + (bl * 4 + 2) * 4 + h] +
                                      sRed[32 + (bl * 4 + 3) * 4 + h];
                    const float inv = tot > 0.f ? 1.f / tot : 0.f;
                    float r0 = 0.f, r1 = 0.f;
#pragma unroll
                    for (int w2 = 0; w2 < 4; ++w2) {
                        r0 += sO[((size_t)(bl * 4 + w2) * 4 + h) * 64 + lane * 2];
                        r1 += sO[((size_t)(bl * 4 + w2) * 4 + h) * 64 + lane * 2 + 1];
                    }
                    sOrow[bl * DS_D + h * DS_DH + lane * 2] = __bfloat162float(__float2bfloat16_rn(r0 * inv));
                    sOrow[bl * DS_D + h * DS_DH + lane * 2 + 1] = __bfloat162float(__float2bfloat16_rn(r1 * inv));
                } else {
                    sOrow[bl * DS_D + wq * DS_DH + lane * 2] = 0.f;
                    sOrow[bl * DS_D + wq * DS_DH + lane * 2 + 1] = 0.f;
                }
                __syncthreads();
                {                                                     // C: x += mask * (o Wo^T): thread = 8 columns x one eighth of k
                    const int kg = threadIdx.x >> 5, cg = threadIdx.x & 31;
                    const __nv_bfloat16* wt = p.wo_t[l] + cg * 8;
                    float a0[8], a1[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) { a0[j] = 0.f; a1[j] = 0.f; }
#pragma unroll 16
                    for (int k = kg * 32; k < kg * 32 + 32; ++k) {
                        const uint4 w = __ldg(reinterpret_cast<const uint4*>(wt + (size_t)k * DS_D));
                        const float2 w0 = unpack_bf16x2(w.x), w1 = unpack_bf16x2(w.y), w2 = unpack_bf16x2(w.z), w3 = unpack_bf16x2(w.w);
                        const float wv[8] = {w0.x, w0.y, w1.x, w1.y, w2.x, w2.y, w3.x, w3.y};
                        const float x0 = sOrow[k], x1 = sOrow[DS_D + k];
#pragma unroll
                        for (int j = 0; j < 8; ++j) { a0[j] = fmaf(x0, wv[j], a0[j]); a1[j] = fmaf(x1, wv[j], a1[j]); }
                    }
                    float* pp = sPart + (size_t)kg * 2 * DS_D + cg * 8;
                    *reinterpret_cast<float4*>(pp) = make_float4(a0[0], a0[1], a0[2], a0[3]);
                    *reinterpret_cast<float4*>(pp + 4) = make_float4(a0[4], a0[5], a0[6], a0[7]);
                    *reinterpret_cast<float4*>(pp + DS_D) = make_float4(a1[0], a1[1], a1[2], a1[3]);
                    *reinterpret_cast<float4*>(pp + DS_D + 4) = make_float4(a1[4], a1[5], a1[6], a1[7]);
                    __syncthreads();
                    const int c = threadIdx.x;
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        float sum = 0.f;
#pragma unroll
                        for (int k8 = 0; k8 < 8; ++k8) sum += sPart[(size_t)(k8 * 2 + r) * DS_D + c];
                        const int row = pair * 2 + r;
                        if (row < B && (p.key_mask == nullptr || pos >= p.cap || p.key_mask[(size_t)row * p.cap + pos]))
                            p.xres[(size_t)row * DS_D + c] += sum;
                    }
                }
            }
        }
        grid_barrier(p.barrier, epoch);

        // ---- D: h = GLU(AdaLN(x) W1^T + b1): a tile is 32 rows x 32 hidden units; every warp computes the value AND the gate columns of
        // its 8 hidden units (two m16n8 chains), so the GLU needs no exchange between warps and a CTA walks two tiles, not four
        {
            // every CTA takes a contiguous run of tiles (column blocks fastest): the AdaLN'd rows are staged once per run
            constexpr int TH = 32;
            const int col_blocks = DS_HID / TH, total = row_blocks * col_blocks;
            const int per_cta = (total + gridDim.x - 1) / gridDim.x;
            const int t_lo = blockIdx.x * per_cta, t_hi = min(total, t_lo + per_cta);
            const int piece = warp >> 1;
            int staged_rb = -1;
            for (int t = t_lo; t < t_hi; ++t) {
                const int rb = t / col_blocks, cb = t - rb * col_blocks;
                const int hcol0 = cb * TH + piece * 8;
                uint32_t bfv[32], bfg[32];
                load_w<16>(bfv, p.w1[l], DS_D, hcol0, lane);
                load_w<16>(bfg, p.w1[l], DS_D, DS_HID + hcol0, lane);
                const float2 bias_v = *reinterpret_cast<const float2*>(p.b1[l] + hcol0 + tig * 2);
                const float2 bias_g = *reinterpret_cast<const float2*>(p.b1[l] + DS_HID + hcol0 + tig * 2);
                if (rb != staged_rb) {
                    __syncthreads();
                    stage_adaln(sA, p.xres, gbp, gb_stride, 2 * l + 1, rb * DS_TM, B, p.eps, warp, lane);
                    staged_rb = rb;
                    __syncthreads();
                }
                float av[4] = {0.f, 0.f, 0.f, 0.f}, ag[4] = {0.f, 0.f, 0.f, 0.f};
                mma_pre<16>(av, sA, DS_LDA, bfv, warp, lane);
                mma_pre<16>(ag, sA, DS_LDA, bfg, warp, lane);
                av[0] += bias_v.x; av[1] += bias_v.y; av[2] += bias_v.x; av[3] += bias_v.y;
                ag[0] += bias_g.x; ag[1] += bias_g.y; ag[2] += bias_g.x; ag[3] += bias_g.y;
                float hv[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) hv[e] = av[e] * ag[e] / (1.f + __expf(-ag[e]));
                const int hcol = hcol0 + tig * 2;
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    const int row = rb * DS_TM + (warp & 1) * 16 + g + hf * 8;
                    if (row < B) *reinterpret_cast<uint32_t*>(p.hmid + (size_t)row * DS_HID + hcol) = pack_bf16x2(hv[2 * hf], hv[2 * hf + 1]);
                }
            }
        }
        grid_barrier(p.barrier, epoch);

        // ---- E: x += h W2^T.  A tile is 32 rows x 16 columns over the WHOLE K = 1024: the four warp pairs of the CTA each take a
        // quarter of K (two m16n8 pieces per warp) and the quarters are summed through shared memory in a fixed order, so the
        // residual stream -- and with it every rendered token -- is bit-reproducible from run to run (no atomics)
        {
            constexpr int TN_E = 16;
            const int col_blocks = DS_D / TN_E;
            const int mh = warp & 1, kq = warp >> 1;
            __nv_bfloat16* sAk = sA + (size_t)kq * DS_TM * DS_LDA;                       // this warp's K quarter of the staged rows
            float* red = reinterpret_cast<float*>(smem_raw + 4 * DS_TM * DS_LDA * 2);     // [4 kq][2 mh][2 pieces][32 lanes][4]
            for (int t = blockIdx.x; t < row_blocks * col_blocks; t += gridDim.x) {
                const int rb = t / col_blocks, cb = t - rb * col_blocks;
                uint32_t bf0[32], bf1[32];
                load_w<16>(bf0, p.w2[l] + kq * DS_D, DS_HID, cb * TN_E, lane);
                load_w<16>(bf1, p.w2[l] + kq * DS_D, DS_HID, cb * TN_E + 8, lane);
                __syncthreads();
                stage_quarters<DS_D / 64>(sA, DS_LDA, p.hmid, DS_HID, rb * DS_TM, B);
                __syncthreads();
                float acc0[4] = {0.f, 0.f, 0.f, 0.f}, acc1[4] = {0.f, 0.f, 0.f, 0.f};
                mma_pre<16>(acc0, sAk, DS_LDA, bf0, warp, lane);
                mma_pre<16>(acc1, sAk, DS_LDA, bf1, warp, lane);
                float4* my = reinterpret_cast<float4*>(red) + ((kq * 2 + mh) * 2) * 32 + lane;
                my[0] = make_float4(acc0[0], acc0[1], acc0[2], acc0[3]);
                my[32] = make_float4(acc1[0], acc1[1], acc1[2], acc1[3]);
                __syncthreads();
                if (kq == 0) {
#pragma unroll
                    for (int piece = 0; piece < 2; ++piece) {
                        float4 sum = reinterpret_cast<const float4*>(red)[((0 * 2 + mh) * 2 + piece) * 32 + lane];
#pragma unroll
                        for (int q4 = 1; q4 < 4; ++q4) {
                            const float4 v = reinterpret_cast<const float4*>(red)[((q4 * 2 + mh) * 2 + piece) * 32 + lane];
                            sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
                        }
                        const int col = cb * TN_E + piece * 8 + tig * 2;
                        const float part[4] = {sum.x, sum.y, sum.z, sum.w};
#pragma unroll
                        for (int hf = 0; hf < 2; ++hf) {
                            const int row = rb * DS_TM + mh * 16 + g + hf * 8;
                            if (row < B) {
                                float2* xr = reinterpret_cast<float2*>(p.xres + (size_t)row * DS_D + col);
                                float2 v = *xr;
                                v.x += part[2 * hf];
                                v.y += part[2 * hf + 1];
                                *xr = v;
                            }
                        }
                    }
                }
            }
        }
        grid_barrier(p.barrier, epoch);
    }

    // ---- final AdaLN -> fp32 out, one warp per row
    for (int row = blockIdx.x * (DS_THREADS / 32) + warp; row < B; row += gridDim.x * (DS_THREADS / 32)) {
        const float4 v0 = *reinterpret_cast<const float4*>(p.xres + (size_t)row * DS_D + lane * 8);
        const float4 v1 = *reinterpret_cast<const float4*>(p.xres + (size_t)row * DS_D + lane * 8 + 4);
        float v[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) s += v[j];
        const float mean = warp_sum(s) * (1.f / DS_D);
        float q = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) { v[j] -= mean; q += v[j] * v[j]; }
        const float rstd = rsqrtf(warp_sum(q) * (1.f / DS_D) + p.eps);
        const __nv_bfloat16* gr = gbp + (size_t)row * gb_stride + (2 * p.depth) * 2 * DS_D + lane * 8;
        const uint4 gu = *reinterpret_cast<const uint4*>(gr), bu = *reinterpret_cast<const uint4*>(gr + DS_D);
        const float2 g0 = unpack_bf16x2(gu.x), g1 = unpack_bf16x2(gu.y), g2 = unpack_bf16x2(gu.z), g3 = unpack_bf16x2(gu.w);
        const float2 b0 = unpack_bf16x2(bu.x), b1 = unpack_bf16x2(bu.y), b2 = unpack_bf16x2(bu.z), b3 = unpack_bf16x2(bu.w);
        const float gm[8] = {g0.x, g0.y, g1.x, g1.y, g2.x, g2.y, g3.x, g3.y}, bt[8] = {b0.x, b0.y, b1.x, b1.y, b2.x, b2.y, b3.x, b3.y};
        float y[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = v[j] * rstd * (1.f + gm[j]) + bt[j];
        *reinterpret_cast<float4*>(p.out + (size_t)row * DS_D + lane * 8) = make_float4(y[0], y[1], y[2], y[3]);
        *reinterpret_cast<float4*>(p.out + (size_t)row * DS_D + lane * 8 + 4) = make_float4(y[4], y[5], y[6], y[7]);
        if (p.out16 != nullptr)
            *reinterpret_cast<uint4*>(p.out16 + (size_t)row * DS_D + lane * 8) =
                make_uint4(pack_bf16x2(y[0], y[1]), pack_bf16x2(y[2], y[3]), pack_bf16x2(y[4], y[5]), pack_bf16x2(y[6], y[7]));
    }
}

// dst_k[b, :] = src_k[b, pos + shift_k, :] for up to 8 row-major [B, T, row] arrays in one launch (blockIdx.y = array): what a
// note-step reads at its device-side position -- the previous tuple, and the per-position terms prepared before the loop
constexpr int GATHER_MAX = 8;
struct GatherParams {
    const uint8_t* src[GATHER_MAX];
    uint8_t* dst[GATHER_MAX];
    int row_bytes[GATHER_MAX];
    int shift[GATHER_MAX];
    const long long* pos_dev;
    int T;
};
__global__ void __launch_bounds__(128) gather_at_pos_kernel(GatherParams g) {
    const int k = blockIdx.y, b = blockIdx.x;
    long long t = *g.pos_dev + g.shift[k];
    if (t < 0) t = 0;
    if (t >= g.T) t = g.T - 1;
    const int rb = g.row_bytes[k];
    const uint8_t* __restrict__ src = g.src[k] + ((size_t)b * g.T + (size_t)t) * rb;
    uint8_t* __restrict__ dst = g.dst[k] + (size_t)b * rb;
    if ((rb & 15) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0) {
        for (int i = threadIdx.x; i < rb / 16; i += 128) reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(src)[i];
    } else {
        for (int i = threadIdx.x; i < rb; i += 128) dst[i] = src[i];
    }
}

}  // namespace

// One new position through an AdaLN decoder stack (see the header of this file).  `ptrs` is a HOST array of device pointers:
// per layer l (9 entries at 9*l): wqkv bf16 [384,256], wo bf16 [256,256], logslopes fp32 [4], w1 bf16 [2048,256], b1 fp32 [2048],
// w2 bf16 [256,1024], kv cache bf16 [B, cap, 128], wqkv^T bf16 [256,384], wo^T bf16 [256,256].  w_ada bf16 [(2*depth+1)*512, S] / b_ada fp32 hold (gamma-1 | beta) rows per
// norm.  scratch: bf16 gb [B,(2*depth+1)*512], qkv [B,384], o [B,256], hmid [B,1024]; fp32 xres [B,256]; `barrier` one uint32.
// hid_out (fp32 [depth, B, 256], may be NULL) receives the inputs of the attention layers (the reference's cache contract);
// out_bf16 (bf16 [B, 256], may be NULL) a bf16 copy of `out`.  gb_all (bf16 [B, T_all, (2*depth+1)*512], may be NULL): the
// (gamma-1 | beta) rows of every position, prepared by one GEMM before a rendering loop; the step then reads position *pos_dev + 1
// in place and `style` / phase 0 are not used.  front (HOST array of 8 device pointers, may be NULL) = the input front of the
// rendering loop evaluated inside this launch instead of x_in: x1 bf16 [B,1536], Wf bf16 [256,1536], p2 fp32 [B,256], scratch fp32
// [B,256], LayerNorm weight / bias fp32 [256], Wc^T bf16 [256,256], c2 fp32 [B,256]:  x = LN(x1 Wf^T + p2) Wc^T + c2.
extern "C" int spb_decode_stack_step(const float* x_in, const float* style, int S, const void* w_ada, const float* b_ada,
                                     const void* const* ptrs, int depth, const uint8_t* key_mask, const long long* pos_dev, int B, int cap,
                                     void* gb, void* qkv, void* o, void* hmid, float* xres, float* hid_out, float* out, void* out_bf16,
                                     unsigned* barrier, float eps, const void* gb_all, int T_all, const void* const* front,
                                     int barrier_is_zero, cudaStream_t stream) {
    if (B <= 0) return SPB_OK;
    SPB_CHECK_ARG((x_in || front) && style && w_ada && b_ada && ptrs && pos_dev && gb && qkv && o && hmid && xres && out && barrier,
                  "spb_decode_stack_step: null pointer");
    SPB_CHECK_ARG(depth >= 1 && depth <= DS_MAX_DEPTH, "spb_decode_stack_step: depth must be in 1..%d", DS_MAX_DEPTH);
    SPB_CHECK_ARG(S % 16 == 0 && S >= 16 && S <= DS_D, "spb_decode_stack_step: style width must be a multiple of 16 in [16, 256], got %d", S);
    SPB_CHECK_ARG(cap >= 1 && cap <= DS_MAX_KEYS, "spb_decode_stack_step: cache capacity must be in 1..%d", DS_MAX_KEYS);
    DecodeStackParams p;
    p.B = B; p.depth = depth; p.S = S; p.cap = cap;
    p.x_in = x_in; p.style = style;
    p.w_ada = reinterpret_cast<const __nv_bfloat16*>(w_ada); p.b_ada = b_ada;
    for (int l = 0; l < depth; ++l) {
        p.wqkv[l] = reinterpret_cast<const __nv_bfloat16*>(ptrs[9 * l]);
        p.wo[l] = reinterpret_cast<const __nv_bfloat16*>(ptrs[9 * l + 1]);
        p.logslopes[l] = reinterpret_cast<const float*>(ptrs[9 * l + 2]);
        p.w1[l] = reinterpret_cast<const __nv_bfloat16*>(ptrs[9 * l + 3]);
        p.b1[l] = reinterpret_cast<const float*>(ptrs[9 * l + 4]);
        p.w2[l] = reinterpret_cast<const __nv_bfloat16*>(ptrs[9 * l + 5]);
        p.kv[l] = reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(ptrs[9 * l + 6]));
        p.wqkv_t[l] = reinterpret_cast<const __nv_bfloat16*>(ptrs[9 * l + 7]);
        p.wo_t[l] = reinterpret_cast<const __nv_bfloat16*>(ptrs[9 * l + 8]);
        SPB_CHECK_ARG(p.wqkv[l] && p.wo[l] && p.logslopes[l] && p.w1[l] && p.b1[l] && p.w2[l] && p.kv[l] && p.wqkv_t[l] && p.wo_t[l],
                      "spb_decode_stack_step: null layer pointer");
    }
    p.key_mask = key_mask; p.pos_dev = pos_dev;
    p.gb = reinterpret_cast<__nv_bfloat16*>(gb); p.qkv = reinterpret_cast<__nv_bfloat16*>(qkv);
    p.o = reinterpret_cast<__nv_bfloat16*>(o); p.hmid = reinterpret_cast<__nv_bfloat16*>(hmid);
    p.xres = xres; p.hid_out = hid_out; p.out = out; p.out16 = reinterpret_cast<__nv_bfloat16*>(out_bf16); p.barrier = barrier; p.eps = eps;
    p.gb_all = reinterpret_cast<const __nv_bfloat16*>(gb_all); p.T_all = T_all;
    SPB_CHECK_ARG(gb_all == nullptr || T_all > 0, "spb_decode_stack_step: gb_all needs T_all > 0");
    p.f_x1 = nullptr;
    if (front != nullptr) {
        for (int i = 0; i < 8; ++i) SPB_CHECK_ARG(front[i] != nullptr, "spb_decode_stack_step: front[%d] is null", i);
        p.f_x1 = reinterpret_cast<const __nv_bfloat16*>(front[0]); p.f_w = reinterpret_cast<const __nv_bfloat16*>(front[1]);
        p.f_p2 = reinterpret_cast<const float*>(front[2]); p.f_te = reinterpret_cast<float*>(const_cast<void*>(front[3]));
        p.f_lnw = reinterpret_cast<const float*>(front[4]); p.f_lnb = reinterpret_cast<const float*>(front[5]);
        p.f_wct = reinterpret_cast<const __nv_bfloat16*>(front[6]); p.f_c2 = reinterpret_cast<const float*>(front[7]);
    }
    int smem = DS_TM * DS_LDA * 2 + (DS_THREADS / 32) * cap * 4 + 64 * 4 + 2 * 4 * 4 * 64 * 4 + (2 * DS_D + 2 * DS_D) * 4 + 2 * (DS_QKV / 2) * 4 + 8 * 2 * DS_D * 4 + (DS_THREADS / 32) * 3 * 16 * 144;
    const int smem_e = 4 * DS_TM * DS_LDA * 2 + 4 * 2 * 2 * 32 * 16;        // phase E: four K quarters of the rows + the reduction scratch
    if (smem < smem_e) smem = smem_e;
    const int smem_f = 4 * DS_TM * DS_FLDA * 2 + 4 * 2 * 2 * 32 * 16;       // front GEMM: four K quarters of the rows + the reduction scratch
    if (front != nullptr && smem < smem_f) smem = smem_f;
    SPB_CHECK_CUDA(cudaFuncSetAttribute(decode_stack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    if (!barrier_is_zero) SPB_CHECK_CUDA(cudaMemsetAsync(barrier, 0, sizeof(unsigned), stream));
    decode_stack_kernel<<<spb_num_sms(), DS_THREADS, smem, stream>>>(p);
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}

// dst_k[b, :] = src_k[b, *pos_dev + shift_k, :] (row_bytes_k bytes per row; src_k row-major [B, T, row]) for n <= 8 arrays in one
// launch; positions are clamped to [0, T).  srcs / dsts / row_bytes / shifts are HOST arrays.
extern "C" int spb_gather_at_pos(const void* const* srcs, void* const* dsts, const int* row_bytes, const int* shifts, int n,
                                 const long long* pos_dev, int B, int T, cudaStream_t stream) {
    if (n <= 0 || B <= 0) return SPB_OK;
    SPB_CHECK_ARG(srcs && dsts && row_bytes && shifts && pos_dev && n <= GATHER_MAX && T > 0, "spb_gather_at_pos: bad arguments (n <= %d)", GATHER_MAX);
    GatherParams g;
    for (int i = 0; i < GATHER_MAX; ++i) {
        const int j = i < n ? i : 0;
        g.src[i] = reinterpret_cast<const uint8_t*>(srcs[j]); g.dst[i] = reinterpret_cast<uint8_t*>(dsts[j]);
        g.row_bytes[i] = row_bytes[j]; g.shift[i] = shifts[j];
    }
    g.pos_dev = pos_dev; g.T = T;
    gather_at_pos_kernel<<<dim3(B, n), 128, 0, stream>>>(g);
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}

// ============================================================================================================================
// Tied output heads of the rendered fields + token sampling in one launch (modules/sampling.py:28-59 top-k filtering, softmax at
// a temperature, one draw; models/scoreperformer/wrappers.py:358-397: PAD and MASK are never emitted).  One CTA per score, one
// warp per field: logits = e_f . table_f^T stay in registers (V <= 256: up to 8 per lane), the k largest are peeled off by k
// warp-wide arg-max rounds (k = 1 is greedy decoding: the lowest index wins ties, like torch.argmax), the draw uses a counter
// based hash of (seed, position, score, field), and the token goes straight into tokens[b, pos + 1, field].
// A field may instead carry top-p (sampling.py:12-18) or top-a (sampling.py:29-32): its logits are bitonic-sorted across the warp
// (descending, the lowest index first among equal values), the filter keeps a prefix of that order by the temperature-1 softmax,
// and the draw runs over the kept prefix.  Per-field token bans (a 256-bit mask) are applied before any filter.
namespace {

constexpr int SF_MAX_FIELDS = 8;
constexpr int SF_TOPK = 0, SF_TOPP = 1, SF_TOPA = 2;        // filter of a field

struct SampleParams {
    const __nv_bfloat16* e;       // [B, ld_e] normalised head projection (all fields)
    int ld_e;
    const __nv_bfloat16* table;   // [sum V, 128]
    int n_fields;
    int field[SF_MAX_FIELDS], offset[SF_MAX_FIELDS], V[SF_MAX_FIELDS], k[SF_MAX_FIELDS];
    int filter[SF_MAX_FIELDS];    // SF_TOPK (k above), SF_TOPP (thres in fa) or SF_TOPA (min_p_pow in fa, min_p_ratio in fb)
    float fa[SF_MAX_FIELDS], fb[SF_MAX_FIELDS];
    uint32_t ban[SF_MAX_FIELDS][8];   // token v of field w is never emitted if bit v of ban[w] is set
    int n_banned;                 // tokens [0, n_banned) are never emitted
    float inv_temperature;
    uint64_t seed;
    const long long* pos_dev;
    long long* tokens;            // [B, T, F]
    int T, F;
    unsigned* advance;            // optional [2]: [0] = CTA counter (zero between launches), [1] = word to clear (the stack kernel's barrier)
};

// top-k (k = 1: greedy) over the logits of one field, lg_row = its 256 logits in shared memory (-inf: banned / beyond V)
__device__ __forceinline__ int sample_topk(const SampleParams& p, const float* lg_row, int k, int b, int w, int lane, long long pos) {
    float lg[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) lg[i] = lg_row[lane + 32 * i];
    // k rounds of warp arg-max: round t leaves its winner (value, token) in lane t
    float top_val = -INFINITY;
    int top_idx = 0;
    for (int t = 0; t < k; ++t) {
        float best = -INFINITY;
        int best_i = 0x7fffffff;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int v = lane + 32 * i;
            if (lg[i] > best) { best = lg[i]; best_i = v; }      // ascending v within a lane: the lowest index wins ties
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
            if (ob > best || (ob == best && oi < best_i)) { best = ob; best_i = oi; }
        }
        if (lane == t) { top_val = best; top_idx = best_i; }
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (lane + 32 * i == best_i) lg[i] = -INFINITY;
    }
    int token = __shfl_sync(0xffffffffu, top_idx, 0);
    if (k > 1) {
        // softmax over the k kept logits at the temperature, then one draw by inverse cdf
        const float m = __shfl_sync(0xffffffffu, top_val, 0);
        float pr = (lane < k && top_val > -INFINITY) ? __expf((top_val - m) * p.inv_temperature) : 0.f;
        float cdf = pr;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float up = __shfl_up_sync(0xffffffffu, cdf, o);
            if (lane >= o) cdf += up;
        }
        const float total = __shfl_sync(0xffffffffu, cdf, 31);
        const uint32_t r = spb_hash32(p.seed + (uint64_t)pos * 0x9E3779B97F4A7C15ull, (uint64_t)b * SF_MAX_FIELDS + (uint64_t)w);
        const float u01 = (float)(r >> 8) * (1.f / 16777216.f) * total;
        const unsigned ge = __ballot_sync(0xffffffffu, lane < k && cdf > u01);
        const int pick = ge != 0 ? __ffs(ge) - 1 : k - 1;
        token = __shfl_sync(0xffffffffu, top_idx, pick);
    }
    return token;
}

// top-p / top-a over the logits of one field.  The 256 (logit, token) pairs are sorted across the warp -- descending, the lowest
// token first among equal logits (the greedy rule) -- by a bitonic network, lane L ending with ranks 8L .. 8L+7 (strides < 8 are
// exchanges inside a lane, the others shuffles).  The temperature-1 softmax q_r / Z of the sorted logits decides which prefix of
// ranks is kept, rank 0 always:
//   top-p (sampling.py:12-18): rank r >= 1 is kept iff q_0 + ... + q_{r-1} <= thres Z  (the reference's `cum > thres` shifted by one);
//   top-a (sampling.py:29-32): rank r is kept iff q_r / Z >= (1 / Z)^min_p_pow min_p_ratio  (1 / Z = the largest probability).
// The kept ranks are drawn from as in top-k: softmax at the temperature, inverse cdf with the same counter hash.
__device__ __forceinline__ int sample_sorted(const SampleParams& p, const float* lg_row, int b, int w, int lane, long long pos) {
    float val[8];
    int idx[8];
    {
        const float4 a = *reinterpret_cast<const float4*>(lg_row + 8 * lane);
        const float4 c = *reinterpret_cast<const float4*>(lg_row + 8 * lane + 4);
        val[0] = a.x; val[1] = a.y; val[2] = a.z; val[3] = a.w; val[4] = c.x; val[5] = c.y; val[6] = c.z; val[7] = c.w;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) idx[i] = 8 * lane + i;
    // x comes before y in the sorted order (token indices are unique: a strict total order)
    auto before = [](float xv, int xi, float yv, int yi) { return xv > yv || (xv == yv && xi < yi); };
#pragma unroll
    for (int kk = 2; kk <= 256; kk <<= 1) {
#pragma unroll
        for (int j = kk >> 1; j > 0; j >>= 1) {
            if (j >= 8) {
                const int lj = j >> 3;
                const bool lower = (lane & lj) == 0;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    // the lower element of the pair takes the one that comes first when (rank & kk) == 0, else the one after
                    const bool take_first = lower == (((8 * lane + i) & kk) == 0);
                    const float ov = __shfl_xor_sync(0xffffffffu, val[i], lj);
                    const int oi = __shfl_xor_sync(0xffffffffu, idx[i], lj);
                    if (before(ov, oi, val[i], idx[i]) == take_first) { val[i] = ov; idx[i] = oi; }
                }
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    if (i & j) continue;
                    const bool first_low = ((8 * lane + i) & kk) == 0;
                    if (before(val[i | j], idx[i | j], val[i], idx[i]) == first_low) {
                        const float tv = val[i]; val[i] = val[i | j]; val[i | j] = tv;
                        const int ti = idx[i]; idx[i] = idx[i | j]; idx[i | j] = ti;
                    }
                }
            }
        }
    }
    // temperature-1 weights q = exp(logit - max) and the mass of the ranks before this lane's first (warp scan)
    const float m = __shfl_sync(0xffffffffu, val[0], 0);
    float q[8], s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { q[i] = __expf(val[i] - m); s += q[i]; }       // banned / beyond V: exp(-inf) = 0
    float incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float up = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += up;
    }
    const float Z = __shfl_sync(0xffffffffu, incl, 31);
    float cum = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) cum = 0.f;
    const bool top_p = p.filter[w] == SF_TOPP;
    const float lim = top_p ? p.fa[w] * Z : __powf(1.f / Z, p.fa[w]) * p.fb[w] * Z;
    float wt[8], ws = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const bool keep = (lane == 0 && i == 0) || (top_p ? cum <= lim : q[i] >= lim);
        cum += q[i];
        wt[i] = keep ? __expf((val[i] - m) * p.inv_temperature) : 0.f;
        ws += wt[i];
    }
    // softmax of the kept ranks at the temperature, one draw by inverse cdf: the lane whose running sum passes u, then its rank
    float wincl = ws;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float up = __shfl_up_sync(0xffffffffu, wincl, o);
        if (lane >= o) wincl += up;
    }
    const float total = __shfl_sync(0xffffffffu, wincl, 31);
    float acc = __shfl_up_sync(0xffffffffu, wincl, 1);
    if (lane == 0) acc = 0.f;
    const uint32_t r = spb_hash32(p.seed + (uint64_t)pos * 0x9E3779B97F4A7C15ull, (uint64_t)b * SF_MAX_FIELDS + (uint64_t)w);
    const float u = (float)(r >> 8) * (1.f / 16777216.f) * total;
    const unsigned hit = __ballot_sync(0xffffffffu, ws > 0.f && wincl > u);
    const unsigned nonzero = __ballot_sync(0xffffffffu, ws > 0.f);          // holds lane 0: rank 0 is always kept
    const int src = hit != 0u ? __ffs(hit) - 1 : 31 - __clz(nonzero);
    int token = idx[0];
    bool found = false;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        if (wt[i] > 0.f && !found) {               // the last kept rank of the lane if rounding leaves u above its running sum
            token = idx[i];
            acc += wt[i];
            found = acc > u;
        }
    }
    return __shfl_sync(0xffffffffu, token, src);
}

__global__ void __launch_bounds__(32 * SF_MAX_FIELDS)
sample_fields_kernel(SampleParams p) {
    const int b = blockIdx.x, w = threadIdx.x >> 5, lane = threadIdx.x & 31;      // the block has exactly n_fields warps
    const int f = p.field[w], V = p.V[w], k = p.k[w];
    const long long pos = *p.pos_dev;
    // logits of 32 vocabulary rows at a time: every lane multiplies ITS four dims of e with the same four dims of each row (one
    // coalesced 256-byte row per load instruction; a lane reading whole rows costs 32 L1 wavefronts per instruction), then a
    // transposing butterfly (31 shuffles) leaves the complete dot product of row 32 i + L in lane L
    float e4[4];
    {
        const uint2 u = *reinterpret_cast<const uint2*>(p.e + (size_t)b * p.ld_e + f * 128 + lane * 4);
        const float2 a = unpack_bf16x2(u.x), c = unpack_bf16x2(u.y);
        e4[0] = a.x; e4[1] = a.y; e4[2] = c.x; e4[3] = c.y;
    }
    const __nv_bfloat16* tbase = p.table + (size_t)p.offset[w] * 128 + lane * 4;
    __shared__ __align__(16) float s_lg[SF_MAX_FIELDS][256];
    uint2 un[32];                                            // the rows of the next group are in flight while this one is reduced
#pragma unroll
    for (int r = 0; r < 32; ++r) un[r] = r < V ? __ldg(reinterpret_cast<const uint2*>(tbase + (size_t)r * 128)) : make_uint2(0u, 0u);
#pragma unroll 1                                             // one copy of the 32-row body: the kernel is short, its code should be too
    for (int i = 0; i < 8; ++i) {
        s_lg[w][lane + 32 * i] = -INFINITY;
        if (32 * i >= V) continue;                           // warp-uniform
        float x[32];
#pragma unroll
        for (int r = 0; r < 32; ++r) {
            const float2 a = unpack_bf16x2(un[r].x), c = unpack_bf16x2(un[r].y);
            x[r] = e4[0] * a.x + e4[1] * a.y + e4[2] * c.x + e4[3] * c.y;
        }
        if (32 * (i + 1) < V) {
#pragma unroll
            for (int r = 0; r < 32; ++r) {
                const int v = 32 * (i + 1) + r;
                un[r] = v < V ? __ldg(reinterpret_cast<const uint2*>(tbase + (size_t)v * 128)) : make_uint2(0u, 0u);
            }
        }
#pragma unroll
        for (int s_ = 16; s_ >= 1; s_ >>= 1) {
            const bool upper = (lane & s_) != 0;
#pragma unroll
            for (int r = 0; r < s_; ++r) {
                const float send = upper ? x[r] : x[r + s_];
                const float keep = upper ? x[r + s_] : x[r];
                x[r] = keep + __shfl_xor_sync(0xffffffffu, send, s_);
            }
        }
        const int v = lane + 32 * i;
        if (v < V && v >= p.n_banned && ((p.ban[w][i] >> lane) & 1u) == 0u) s_lg[w][v] = x[0];
    }
    __syncwarp();
    const int token = p.filter[w] == SF_TOPK ? sample_topk(p, s_lg[w], k, b, w, lane, pos)
                                             : sample_sorted(p, s_lg[w], b, w, lane, pos);
    if (lane == 0 && pos + 1 < p.T) p.tokens[((size_t)b * p.T + (size_t)(pos + 1)) * p.F + f] = token;
    if (p.advance != nullptr) {
        // the last CTA to finish ends the note-step: position += 1 and the decode-stack kernel's grid-barrier word back to zero
        // (every other CTA read the position before it counted itself in), instead of two more launches per step
        __shared__ int s_last;
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            s_last = atomicAdd(p.advance, 1u) == gridDim.x - 1;
        }
        __syncthreads();
        if (s_last && threadIdx.x == 0) {
            *const_cast<long long*>(p.pos_dev) = pos + 1;
            p.advance[0] = 0u;
            p.advance[1] = 0u;
        }
    }
}

}  // namespace

namespace {

// Both entry points: the filter arrays may be NULL (every field top-k, no per-field bans).
int launch_sample_fields(const char* name, const void* e, int ld_e, const void* table, const int* fields, const int* offsets,
                         const int* vocab, const int* topk, int n_fields, int n_banned, float temperature, uint64_t seed,
                         const long long* pos_dev, long long* tokens, int B, int T, int F, unsigned* advance, const float* top_p,
                         const float* top_a_pow, const float* top_a_ratio, const uint32_t* ban_bits, cudaStream_t stream) {
    if (B <= 0 || n_fields <= 0) return SPB_OK;
    SPB_CHECK_ARG(e && table && fields && offsets && vocab && topk && pos_dev && tokens, "%s: null pointer", name);
    SPB_CHECK_ARG(n_fields <= SF_MAX_FIELDS && ld_e % 4 == 0 && temperature > 0.f, "%s: at most %d fields, ld_e %% 4 == 0, temperature > 0", name, SF_MAX_FIELDS);
    SPB_CHECK_ARG((top_a_pow == nullptr) == (top_a_ratio == nullptr), "%s: top_a_pow and top_a_ratio go together", name);
    SampleParams p;
    p.e = reinterpret_cast<const __nv_bfloat16*>(e); p.ld_e = ld_e;
    p.table = reinterpret_cast<const __nv_bfloat16*>(table);
    p.n_fields = n_fields;
    for (int i = 0; i < n_fields; ++i) {
        SPB_CHECK_ARG(vocab[i] >= 1 && vocab[i] <= 256 && topk[i] >= 1 && topk[i] <= 32 && fields[i] >= 0 && fields[i] < F,
                      "%s: field %d needs V <= 256 and 1 <= k <= 32 (V %d, k %d)", name, fields[i], vocab[i], topk[i]);
        p.field[i] = fields[i]; p.offset[i] = offsets[i]; p.V[i] = vocab[i]; p.k[i] = topk[i] < vocab[i] ? topk[i] : vocab[i];
        p.filter[i] = SF_TOPK; p.fa[i] = 0.f; p.fb[i] = 0.f;
        const bool want_p = top_p != nullptr && top_p[i] >= 0.f, want_a = top_a_ratio != nullptr && top_a_ratio[i] > 0.f;
        SPB_CHECK_ARG(top_p == nullptr || std::isfinite(top_p[i]), "%s: field %d: top_p must be finite (< 0 = off)", name, fields[i]);
        SPB_CHECK_ARG(top_a_pow == nullptr || (std::isfinite(top_a_pow[i]) && std::isfinite(top_a_ratio[i])),
                      "%s: field %d: top-a parameters must be finite (ratio <= 0 = off)", name, fields[i]);
        SPB_CHECK_ARG(!(want_p && want_a), "%s: field %d: at most one of top-p and top-a", name, fields[i]);
        if (want_p) { p.filter[i] = SF_TOPP; p.fa[i] = top_p[i]; }
        if (want_a) { p.filter[i] = SF_TOPA; p.fa[i] = top_a_pow[i]; p.fb[i] = top_a_ratio[i]; }
        int left = 0;                                        // tokens the field may still emit
        for (int wd = 0; wd < 8; ++wd) {
            p.ban[i][wd] = ban_bits != nullptr ? ban_bits[8 * i + wd] : 0u;
            for (int bit = 0; bit < 32; ++bit) {
                const int v = 32 * wd + bit;
                left += v >= n_banned && v < vocab[i] && ((p.ban[i][wd] >> bit) & 1u) == 0u;
            }
        }
        SPB_CHECK_ARG(ban_bits == nullptr || left > 0, "%s: field %d: every token is banned", name, fields[i]);
    }
    p.n_banned = n_banned; p.inv_temperature = 1.f / temperature; p.seed = seed; p.pos_dev = pos_dev;
    p.tokens = tokens; p.T = T; p.F = F; p.advance = advance;
    sample_fields_kernel<<<B, 32 * n_fields, 0, stream>>>(p);
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}

}  // namespace

// e bf16 [B, ld_e] (LayerNorm'ed head projection, 128 columns per field), table bf16 [sum V, 128]; for each of the n_fields listed
// fields (field index, first table row, vocabulary, k of the top-k filter; k = 1: greedy) one token is written to
// tokens[b, *pos_dev + 1, field] (int64 [B, T, F]).  V <= 256, k <= 32, at most 8 fields.
extern "C" int spb_sample_fields(const void* e, int ld_e, const void* table, const int* fields, const int* offsets, const int* vocab,
                                 const int* topk, int n_fields, int n_banned, float temperature, uint64_t seed, const long long* pos_dev,
                                 long long* tokens, int B, int T, int F, unsigned* advance, cudaStream_t stream) {
    return launch_sample_fields("spb_sample_fields", e, ld_e, table, fields, offsets, vocab, topk, n_fields, n_banned, temperature, seed,
                                pos_dev, tokens, B, T, F, advance, nullptr, nullptr, nullptr, nullptr, stream);
}

// spb_sample_fields with per-field filters (host arrays, each may be NULL = off for every field): top_p[i] >= 0 selects top-p with
// that threshold (0 keeps the arg-max only), top_a_ratio[i] > 0 selects top-a with (top_a_pow[i], top_a_ratio[i]); a field with
// neither samples top-k with topk[i].  ban_bits[8 i .. 8 i + 7] (uint32) is a 256-bit set of tokens field i never emits, applied
// with [0, n_banned) before the filter.
extern "C" int spb_sample_fields_filtered(const void* e, int ld_e, const void* table, const int* fields, const int* offsets, const int* vocab,
                                          const int* topk, int n_fields, int n_banned, float temperature, uint64_t seed,
                                          const long long* pos_dev, long long* tokens, int B, int T, int F, unsigned* advance,
                                          const float* top_p, const float* top_a_pow, const float* top_a_ratio, const uint32_t* ban_bits,
                                          cudaStream_t stream) {
    return launch_sample_fields("spb_sample_fields_filtered", e, ld_e, table, fields, offsets, vocab, topk, n_fields, n_banned, temperature,
                                seed, pos_dev, tokens, B, T, F, advance, top_p, top_a_pow, top_a_ratio, ban_bits, stream);
}

// ============================================================================================================================
// Start of a streaming call of a render session (decode.py `_RenderSession`): the session keeps bf16 copies of the decoder's
// weights and a stack plan between calls, so before it enqueues the note-steps it has to know whether the weights moved under it.
// torch's version counters do not tell (the flat AdamW kernel writes parameters through raw pointers), so this launch hashes the
// bit patterns of every parameter and buffer of the decoder into a 64-bit fingerprint:
//     fingerprint = sum over words i of splitmix64((i << 32) | word_i)   (mod 2^64)
// where i numbers the 32-bit words of all listed tensors in table order.  The index mixing makes a moved value count; the sum is
// order-independent, so CTAs hash any slice they like and meet in one integer atomic.  The last CTA compares the fingerprint with
// the stored one, writes the stale flag the host reads, and stores the new fingerprint.  The same launch also zeroes the stack
// plan's `advance` words (sample_fields' CTA counter and the stack kernel's grid-barrier word: a plan that outlives a call must not
// rely on the sampler of an earlier call having cleared them) and writes the call's start position.
namespace {

constexpr int SB_THREADS = 256;

struct SessionBeginParams {
    const long long* table;       // [n, 3]: device address, number of 32-bit words, index of the first word
    int n;
    unsigned long long* state;    // [4]: stored fingerprint, running sum, finished CTAs (both zero between launches), stale flag
    unsigned* advance;            // [2]
    long long* pos_dev;
    long long start;
};

__device__ __forceinline__ unsigned long long fingerprint_term(unsigned long long index, unsigned word) {
    unsigned long long z = ((index << 32) | word) + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

__global__ void __launch_bounds__(SB_THREADS) session_begin_kernel(SessionBeginParams p) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        p.advance[0] = 0u;
        p.advance[1] = 0u;
        *p.pos_dev = p.start;
    }
    const long long tid = (long long)blockIdx.x * SB_THREADS + threadIdx.x, nth = (long long)gridDim.x * SB_THREADS;
    unsigned long long acc = 0;
    for (int t = 0; t < p.n; ++t) {
        const unsigned* w = reinterpret_cast<const unsigned*>(p.table[3 * t]);
        const long long n = p.table[3 * t + 1];
        const unsigned long long first = (unsigned long long)p.table[3 * t + 2];
        long long done = 0;
        if ((reinterpret_cast<uintptr_t>(w) & 15) == 0) {         // 16-byte loads over the aligned body
            const uint4* w4 = reinterpret_cast<const uint4*>(w);
            const long long n4 = n >> 2;
            for (long long i = tid; i < n4; i += nth) {
                const uint4 v = __ldg(w4 + i);
                const unsigned long long g = first + 4ull * (unsigned long long)i;
                acc += fingerprint_term(g, v.x) + fingerprint_term(g + 1, v.y) + fingerprint_term(g + 2, v.z) + fingerprint_term(g + 3, v.w);
            }
            done = n4 << 2;
        }
        for (long long i = done + tid; i < n; i += nth) acc += fingerprint_term(first + (unsigned long long)i, __ldg(w + i));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    __shared__ unsigned long long s_part[SB_THREADS / 32];
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x != 0) return;
    unsigned long long sum = 0;
#pragma unroll
    for (int i = 0; i < SB_THREADS / 32; ++i) sum += s_part[i];
    atomicAdd(p.state + 1, sum);
    __threadfence();
    if (atomicAdd(p.state + 2, 1ull) != gridDim.x - 1) return;
    // the last CTA: every other CTA added its part before it counted itself in
    __threadfence();
    const unsigned long long fp = atomicExch(p.state + 1, 0ull);
    p.state[3] = fp != p.state[0] ? 1ull : 0ull;
    p.state[0] = fp;
    p.state[2] = 0ull;
}

}  // namespace

// table: DEVICE int64 [n_tensors, 3] (address, number of 32-bit words, index of the first word); state: device uint64 [4] (stored
// fingerprint, two words that must be zero between launches, stale flag written here); advance: the stack plan's uint32 [2];
// pos_dev: device int64 set to `start`.
extern "C" int spb_session_begin(const long long* table, int n_tensors, unsigned long long* state, unsigned* advance, long long* pos_dev,
                                 long long start, cudaStream_t stream) {
    SPB_CHECK_ARG(table && state && advance && pos_dev && n_tensors >= 0 && start >= 0, "spb_session_begin: bad arguments");
    SessionBeginParams p;
    p.table = table; p.n = n_tensors; p.state = state; p.advance = advance; p.pos_dev = pos_dev; p.start = start;
    session_begin_kernel<<<4 * spb_num_sms(), SB_THREADS, 0, stream>>>(p);
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}
